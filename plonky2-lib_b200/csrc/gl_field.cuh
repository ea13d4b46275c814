// Goldilocks field p = 2^64 - 2^32 + 1 on the B200 integer pipes.
//
// plonky2_field::goldilocks_field::GoldilocksField (SURVEY 8a P0; the type the reference imports at
// src/smt/goldilocks_poseidon/mod.rs:9 and src/zkdsa/circuits/mod.rs:81-100).
//
// Representation: a u64 in [0, 2^64) that may be non-canonical (>= p), exactly like upstream keeps
// it internally; every value that leaves the device goes through gl_canon().  Arithmetic is exact,
// so results are bit-identical with the CPU whatever the evaluation order.
//
// 64x64->128 products are four IMAD.WIDE.U32 (32x32+64) on the FMA pipe; the reduction uses
// 2^64 = 2^32 - 1 and 2^96 = -1 (mod p), one more IMAD plus carry-chain adds on the ALU pipe.
#pragma once
#include <cstdint>

#ifndef GL_HD
#ifdef __CUDACC__
#define GL_HD __host__ __device__ __forceinline__
#define GL_D __device__ __forceinline__
#else
#define GL_HD inline
#define GL_D inline
#endif
#endif

typedef uint64_t u64;
typedef uint32_t u32;

#define GL_P 0xFFFFFFFF00000001ULL
#define GL_EPS 0xFFFFFFFFULL

// ------------------------------------------------------------------------------------------------
// host-side exact arithmetic (twiddle / constant tables are generated on the host at ctx creation)
// ------------------------------------------------------------------------------------------------
namespace glh {
typedef unsigned __int128 u128;
inline u64 canon(u64 x) { return x >= GL_P ? x - GL_P : x; }
inline u64 reduce(u128 x) { return (u64)(x % GL_P); }
inline u64 add(u64 a, u64 b) { return reduce((u128)a + b); }
inline u64 sub(u64 a, u64 b) { return reduce((u128)canon(a) + GL_P - canon(b)); }
inline u64 mul(u64 a, u64 b) { return reduce((u128)a * b); }
inline u64 pow(u64 a, u64 e) {
    u64 r = 1;
    a = canon(a);
    while (e) {
        if (e & 1) r = mul(r, a);
        a = mul(a, a);
        e >>= 1;
    }
    return r;
}
inline u64 inv(u64 a) { return pow(a, GL_P - 2); }
// Field::primitive_root_of_unity(k) = POWER_OF_TWO_GENERATOR^(2^(32-k)), generator 7^((p-1)/2^32)
inline u64 root_of_unity(unsigned lg) {
    u64 g = pow(7, (GL_P - 1) >> 32);
    for (unsigned i = lg; i < 32; i++) g = mul(g, g);
    return g;
}
// QuadraticExtension: F[X]/(X^2 - 7)
struct ext {
    u64 a, b;
};
inline ext ext_mul(ext x, ext y) {
    return {add(mul(x.a, y.a), mul(7, mul(x.b, y.b))), add(mul(x.a, y.b), mul(x.b, y.a))};
}
inline ext ext_pow(ext x, u64 e) {
    ext r = {1, 0};
    while (e) {
        if (e & 1) r = ext_mul(r, x);
        x = ext_mul(x, x);
        e >>= 1;
    }
    return r;
}
}  // namespace glh

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// device arithmetic
// ------------------------------------------------------------------------------------------------
GL_D u64 gl_pack(u32 lo, u32 hi) { return ((u64)hi << 32) | lo; }

// x (128 bit) -> [0, 2^64), x = r0 + 2^32 r1 + 2^64 r2 + 2^96 r3.  2^64 = 2^32 - 1, 2^96 = -1 (mod p):
//   x = (r0 + 2^32 r1) + 2^32 r2 - (r2 + r3)
// One 64-bit add (carry K1), one 64-bit subtract of the 33-bit g = r2 + r3 (borrow K2), then the net
// wrap k = K1 - K2 in {-1, 0, 1} is folded back as k * (2^32 - 1).  All on the ALU pipe, no multiply
// (IMAD.HI runs at a third of the IMAD rate on B200: profiles/r1_pipe_peaks.json).
GL_D u64 gl_reduce128(u64 lo, u64 hi) {
    u32 r0 = (u32)lo, r1 = (u32)(lo >> 32), r2 = (u32)hi, r3 = (u32)(hi >> 32), w0, w1;
    asm("{\n\t"
        ".reg .u32 k, g0, g1, nk, sg;\n\t"
        "add.cc.u32 %1, %3, %4;\n\t"     // w1 = r1 + r2
        "addc.u32 k, 0, 0;\n\t"          // K1
        "add.cc.u32 g0, %4, %5;\n\t"     // g = r2 + r3
        "addc.u32 g1, 0, 0;\n\t"
        "sub.cc.u32 %0, %2, g0;\n\t"     // w -= g
        "subc.cc.u32 %1, %1, g1;\n\t"
        "subc.u32 k, k, 0;\n\t"          // k = K1 - K2
        "sub.u32 nk, 0, k;\n\t"          // low word of k * (2^32 - 1)
        "shr.s32 sg, k, 31;\n\t"         // high word: -1 when k = -1
        "add.cc.u32 %0, %0, nk;\n\t"
        "addc.u32 %1, %1, sg;\n\t"
        "}"
        : "=&r"(w0), "=&r"(w1)
        : "r"(r0), "r"(r1), "r"(r2), "r"(r3));
    return gl_pack(w0, w1);
}

GL_D u64 gl_mul(u64 a, u64 b) {
    unsigned __int128 p = (unsigned __int128)a * b;
    return gl_reduce128((u64)p, (u64)(p >> 64));
}
// a^2 = l + 2^32 (m + m) + 2^64 h with l = a0^2, m = a0 a1, h = a1^2 (a = a0 + 2^32 a1): three wide products instead of
// gl_mul's four; the cross product enters the carry chain twice instead of being shifted.  No partial sum exceeds a^2.
GL_D u64 gl_sqr(u64 a) {
    u32 r0, r1, r2, r3;
    asm("{\n\t"
        ".reg .u32 a0, a1, l1, m0, m1, h0, h1;\n\t"
        ".reg .u64 l, m, h;\n\t"
        "mov.b64 {a0, a1}, %4;\n\t"
        "mul.wide.u32 l, a0, a0;\n\t"
        "mul.wide.u32 m, a0, a1;\n\t"
        "mul.wide.u32 h, a1, a1;\n\t"
        "mov.b64 {%0, l1}, l;\n\t"
        "mov.b64 {m0, m1}, m;\n\t"
        "mov.b64 {h0, h1}, h;\n\t"
        "add.cc.u32 %1, l1, m0;\n\t"
        "addc.cc.u32 %2, h0, m1;\n\t"
        "addc.u32 %3, h1, 0;\n\t"
        "add.cc.u32 %1, %1, m0;\n\t"
        "addc.cc.u32 %2, %2, m1;\n\t"
        "addc.u32 %3, %3, 0;\n\t"
        "}"
        : "=&r"(r0), "=&r"(r1), "=&r"(r2), "=&r"(r3)
        : "l"(a));
    return gl_reduce128(gl_pack(r0, r1), gl_pack(r2, r3));
}

// a + b where b is canonical (< p): one wrap correction suffices
GL_D u64 gl_add_c(u64 a, u64 b_canonical) {
    u64 s = a + b_canonical;
    return s + ((s < a) ? GL_EPS : 0ULL);
}
// general a + b, both possibly non-canonical: a second wrap can happen (only if both >= p).  Carry-flag
// chains: 8 ALU instructions (the C form with 64-bit compares compiles to 12).
GL_D u64 gl_add(u64 a, u64 b) {
    u32 a0 = (u32)a, a1 = (u32)(a >> 32), b0 = (u32)b, b1 = (u32)(b >> 32), r0, r1;
    asm("{\n\t"
        ".reg .u32 m;\n\t"
        "add.cc.u32 %0, %2, %4;\n\t"
        "addc.cc.u32 %1, %3, %5;\n\t"
        "addc.u32 m, 0, 0;\n\t"          // the carry, through add-family instructions only (PTX defines CC.CF for
        "neg.s32 m, m;\n\t"              // addc after add.cc; nothing here reads it as a borrow): carry ? 0xffffffff : 0
        "add.cc.u32 %0, %0, m;\n\t"     //   = carry * (2^32 - 1)
        "addc.cc.u32 %1, %1, 0;\n\t"
        "addc.u32 m, 0, 0;\n\t"
        "neg.s32 m, m;\n\t"
        "add.cc.u32 %0, %0, m;\n\t"
        "addc.u32 %1, %1, 0;\n\t"
        "}"
        : "=&r"(r0), "=&r"(r1)
        : "r"(a0), "r"(a1), "r"(b0), "r"(b1));
    return gl_pack(r0, r1);
}
// general a - b
GL_D u64 gl_sub(u64 a, u64 b) {
    u32 a0 = (u32)a, a1 = (u32)(a >> 32), b0 = (u32)b, b1 = (u32)(b >> 32), r0, r1;
    asm("{\n\t"
        ".reg .u32 m;\n\t"
        "sub.cc.u32 %0, %2, %4;\n\t"
        "subc.cc.u32 %1, %3, %5;\n\t"
        "subc.u32 m, 0, 0;\n\t"          // 0 - 0 - borrow (sub family after sub.cc, as PTX defines it): borrow ? 0xffffffff : 0
        "sub.cc.u32 %0, %0, m;\n\t"
        "subc.cc.u32 %1, %1, 0;\n\t"
        "subc.u32 m, 0, 0;\n\t"
        "sub.cc.u32 %0, %0, m;\n\t"
        "subc.u32 %1, %1, 0;\n\t"
        "}"
        : "=&r"(r0), "=&r"(r1)
        : "r"(a0), "r"(a1), "r"(b0), "r"(b1));
    return gl_pack(r0, r1);
}
GL_D u64 gl_canon(u64 x) { return x >= GL_P ? x - GL_P : x; }
GL_D u64 gl_neg(u64 a) { return gl_sub(0, a); }

// a * b + c + d with ONE reduction: (2^64 - 1)^2 + 2 (2^64 - 1) = 2^128 - 1, so the sum fits 128 bits
GL_D u64 gl_mad2(u64 a, u64 b, u64 c, u64 d) {
    unsigned __int128 p = (unsigned __int128)a * b;
    p += c;
    p += d;
    return gl_reduce128((u64)p, (u64)(p >> 64));
}
// base^e from the host's 3 x 1024 power table of base (e < 2^30)
GL_D u64 gl_powtab(const u64* __restrict__ tab, u64 e) {
    u64 r = __ldg(tab + (e & 1023));
    if (e >> 10) {
        r = gl_mul(r, __ldg(tab + 1024 + ((e >> 10) & 1023)));
        if (e >> 20) r = gl_mul(r, __ldg(tab + 2048 + ((e >> 20) & 1023)));
    }
    return r;
}

GL_D u64 gl_pow(u64 a, u64 e) {
    u64 r = 1;
    while (e) {
        if (e & 1) r = gl_mul(r, a);
        a = gl_sqr(a);
        e >>= 1;
    }
    return r;
}

// QuadraticExtension<GoldilocksField>: F[X]/(X^2 - 7)
struct gl_ext {
    u64 a, b;
};
GL_D gl_ext gl_ext_add(gl_ext x, gl_ext y) { return {gl_add(x.a, y.a), gl_add(x.b, y.b)}; }
GL_D gl_ext gl_ext_mul(gl_ext x, gl_ext y) {
    u64 c0 = gl_add(gl_mul(x.a, y.a), gl_mul(7, gl_mul(x.b, y.b)));
    u64 c1 = gl_add(gl_mul(x.a, y.b), gl_mul(x.b, y.a));
    return {c0, c1};
}
#endif  // __CUDACC__
