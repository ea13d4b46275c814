"""Host-side mirror of the plonky2 plugin surface that Plonky2-lib reaches (SURVEY.md 8b), over the
C ABI of include/gl_b200.h.

Names, argument meaning and error behaviour follow the upstream Rust interface so the parity tests
read like the reference's own: `PolynomialBatch.from_values / from_coeffs`, `MerkleTree.new /
prove / get`, `PoseidonHash.hash_no_pad / two_to_one / hash_pad / hash_or_noop`, `FriConfig`,
`PoseidonNodeHash.calc_node_hash` (src/smt/goldilocks_poseidon/mod.rs:158-184) and
`SparseMerkleProcessProof.check` (src/smt/proof/process.rs:47-51).  Upstream functions are infallible
and panic on contract violations; here a violation raises `GlPanic` carrying the library's message.

Buffers: numpy uint64 arrays are host memory (GL_HOST); torch CUDA tensors with an 8-byte dtype are
device memory (GL_DEVICE) and are used in place.  Nothing in this module computes field arithmetic:
every result comes from libgl_b200.so.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import List, Optional, Sequence

import numpy as np

from . import _native as N
from . import wire

P = 0xFFFFFFFF00000001


class GlPanic(RuntimeError):
    """What `panic!` is upstream: a contract violation or a CUDA failure (code in .code)."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"[GL_E {code}] {msg}")
        self.code = code


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


class DeviceBuffer:
    """A block of device memory owned by the host mirror (gl_dev_alloc): `shape` uint64 elements."""

    def __init__(self, shape, ctx: "Context"):
        self.shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.nbytes = int(np.prod(self.shape)) * 8
        self._ctx = ctx
        p = C.c_void_p()
        ctx.check(ctx._lib.gl_dev_alloc(ctx._h, self.nbytes, C.byref(p)))
        self.ptr = p.value

    def to_host(self, count_elems: Optional[int] = None) -> np.ndarray:
        n = int(np.prod(self.shape)) if count_elems is None else count_elems
        out = np.empty(n, dtype=np.uint64)
        self._ctx.check(self._ctx._lib.gl_copy(self._ctx._h, out.ctypes.data, N.GL_HOST, self.ptr, N.GL_DEVICE, n * 8))
        return out.reshape(self.shape) if count_elems is None else out

    def from_host(self, arr: np.ndarray):
        a = np.ascontiguousarray(arr, dtype=np.uint64)
        assert a.nbytes <= self.nbytes
        self._ctx.check(self._ctx._lib.gl_copy(self._ctx._h, self.ptr, N.GL_DEVICE, a.ctypes.data, N.GL_HOST, a.nbytes))
        return self

    def free(self):
        if getattr(self, "ptr", None) and self._ctx._h:
            self._ctx._lib.gl_dev_free(self._ctx._h, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class _Buf:
    """pointer + space of a caller buffer (numpy host array, torch CUDA tensor or DeviceBuffer)."""

    __slots__ = ("ptr", "space", "keep", "nbytes")

    def __init__(self, x, writable: bool = False):
        if x is None:
            self.ptr, self.space, self.keep, self.nbytes = None, None, None, 0
            return
        if isinstance(x, DeviceBuffer):
            self.ptr, self.space, self.keep, self.nbytes = x.ptr, N.GL_DEVICE, x, x.nbytes
            return
        if _is_torch(x):
            if not x.is_cuda:
                x = x.numpy()
            else:
                if not x.is_contiguous() or x.element_size() != 8:
                    raise TypeError("device buffers must be contiguous tensors of an 8-byte dtype")
                self.ptr, self.space, self.keep = x.data_ptr(), N.GL_DEVICE, x
                self.nbytes = x.numel() * 8
                return
        if not isinstance(x, np.ndarray) or x.dtype != np.uint64 or not x.flags.c_contiguous:
            raise TypeError("host buffers must be C-contiguous numpy uint64 arrays")
        if writable and not x.flags.writeable:
            raise TypeError("output buffer is read-only")
        self.ptr, self.space, self.keep, self.nbytes = x.ctypes.data, N.GL_HOST, x, x.nbytes


def _h(x) -> np.ndarray:
    return np.ascontiguousarray(x, dtype=np.uint64)


def _same_space(*bufs: _Buf) -> int:
    spaces = {b.space for b in bufs if b.space is not None}
    if len(spaces) > 1:
        raise TypeError("all buffers of one call must live in the same space (all host or all device)")
    return spaces.pop() if spaces else N.GL_HOST


class Context:
    """gl_ctx: one device, one stream.  `Context.default()` is what the mirror classes use."""

    _default: Optional["Context"] = None

    def __init__(self, device: int = 0):
        self._lib = N.load()
        h = C.c_void_p()
        rc = self._lib.gl_ctx_create(device, C.byref(h))
        if rc:
            raise GlPanic(rc, (self._lib.gl_last_error(None) or b"").decode())
        self._h = h
        self.device = device

    @classmethod
    def default(cls) -> "Context":
        if cls._default is None:
            cls._default = Context(0)
        return cls._default

    def check(self, rc: int):
        if rc:
            raise GlPanic(rc, (self._lib.gl_last_error(self._h) or b"").decode())

    def set_shard(self, index: int, count: int):
        self.check(self._lib.gl_ctx_set_shard(self._h, index, count))

    def set_salt_seed(self, seed: int):
        """Reproducible blinding salt (tests); by default the seed comes from the OS entropy source."""
        self.check(self._lib.gl_ctx_set_salt_seed(self._h, seed & 0xFFFFFFFFFFFFFFFF))

    def sync(self):
        self.check(self._lib.gl_ctx_sync(self._h))

    @property
    def stream(self) -> int:
        return int(self._lib.gl_ctx_stream(self._h) or 0)

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.gl_ctx_kernel_launches(self._h))

    PHASES = ("copy_in", "ifft", "coeffs_out", "lde_ntt", "leaf_hash", "tree_levels")

    def commit_phase_ms(self) -> dict:
        """Device time (ms) of each phase of the last PolynomialBatch.from_* call."""
        out = (C.c_float * 6)()
        self.check(self._lib.gl_ctx_commit_phase_ms(self._h, out))
        return dict(zip(self.PHASES, [float(x) for x in out]))

    def trim(self):
        self.check(self._lib.gl_ctx_trim(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gl_ctx_destroy(self._h)
            self._h = None
            if Context._default is self:
                Context._default = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ctx(ctx: Optional[Context]) -> Context:
    return ctx if ctx is not None else Context.default()


def pinned_empty(shape, ctx: Optional[Context] = None) -> np.ndarray:
    """uint64 array in page-locked host memory (gl_host_alloc); freed when the array is collected."""
    lib = N.load()
    n = int(np.prod(shape))
    p = C.c_void_p()
    rc = lib.gl_host_alloc(n * 8, C.byref(p))
    if rc:
        raise GlPanic(rc, (lib.gl_last_error(None) or b"").decode())

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            lib.gl_host_free(self.ptr)

    owner = _Owner(p)
    buf = (C.c_uint64 * n).from_address(p.value)
    return _PinnedArray(np.frombuffer(buf, dtype=np.uint64).reshape(shape), owner)


class _PinnedArray(np.ndarray):
    """ndarray view that keeps its pinned allocation alive."""

    def __new__(cls, arr, owner):
        obj = np.asarray(arr).view(cls)
        obj._owner = owner
        return obj

    def __array_finalize__(self, obj):
        self._owner = getattr(obj, "_owner", None)


# ------------------------------------------------------------------------------------------------
# WrappedHashOut text form (src/smt/goldilocks_poseidon/hash/mod.rs:84-119; the JSON the zkdsa tests pin,
# src/zkdsa/circuits/mod.rs:136-153): "0x" + hex of HashOut::to_bytes() (4 x u64 little endian) byte-reversed
# ------------------------------------------------------------------------------------------------
def hash_out_to_hex(h) -> str:
    b = np.ascontiguousarray(h, dtype="<u8").reshape(4).tobytes()
    return "0x" + b[::-1].hex()


def hash_out_from_hex(s: str) -> np.ndarray:
    """Accepts what the reference's Deserialize accepts: a 0x prefix, an even number of hex digits, at most 32 bytes
    (shorter strings are the low-order bytes)."""
    if not s.startswith("0x"):
        raise ValueError(f"fail to strip 0x-prefix: given value {s} does not start with 0x")
    try:
        b = bytes.fromhex(s[2:])
    except ValueError as e:
        raise ValueError(f"fail to parse a hex string: {e}") from None
    if len(b) > 32:
        raise ValueError("too long hexadecimal sequence")
    le = b[::-1] + bytes(32 - len(b))
    return np.frombuffer(le, dtype="<u8").astype(np.uint64)


# ------------------------------------------------------------------------------------------------
# plonky2::hash::poseidon::PoseidonHash (Hasher<F>)
# ------------------------------------------------------------------------------------------------
class PoseidonHash:
    HASH_SIZE = 32
    SPONGE_WIDTH = 12
    SPONGE_RATE = 8

    @staticmethod
    def permute(states, ctx: Optional[Context] = None):
        """PoseidonPermutation::permute over a batch [m][12]; returns a new array (host) / in place (device)."""
        ctx = _ctx(ctx)
        if not _is_torch(states):
            states = _h(states).copy()
        single = states.ndim == 1
        s2 = states.reshape(-1, 12)
        b = _Buf(s2, writable=True)
        ctx.check(ctx._lib.gl_poseidon_permute_batch(ctx._h, b.ptr, s2.shape[0], b.space))
        return s2.reshape(12) if single else s2

    @staticmethod
    def two_to_one(left, right, out=None, ctx: Optional[Context] = None):
        """Hasher::two_to_one (src/smt/goldilocks_poseidon/mod.rs:165, src/zkdsa/account.rs:165); [m][4] or [4]."""
        ctx = _ctx(ctx)
        dev = _is_torch(left) and left.is_cuda
        if not dev:
            left, right = _h(left), _h(right)
        single = left.ndim == 1
        l2, r2 = left.reshape(-1, 4), right.reshape(-1, 4)
        if l2.shape != r2.shape:
            raise GlPanic(N.GL_E_ARG, "two_to_one: shape mismatch")
        if out is None:
            if dev:
                import torch

                out = torch.empty_like(l2)
            else:
                out = np.empty_like(l2)
        bl, br, bo = _Buf(l2), _Buf(r2), _Buf(out, writable=True)
        ctx.check(ctx._lib.gl_poseidon_two_to_one_batch(ctx._h, bl.ptr, br.ptr, bo.ptr, l2.shape[0], _same_space(bl, br, bo)))
        return out.reshape(4) if single else out

    @staticmethod
    def hash_no_pad(inputs, out=None, ctx: Optional[Context] = None):
        """Hasher::hash_no_pad; [m][len] -> [m][4], or [len] -> [4]."""
        ctx = _ctx(ctx)
        dev = _is_torch(inputs) and inputs.is_cuda
        if not dev:
            inputs = _h(inputs)
        single = inputs.ndim == 1
        x2 = inputs.reshape(1, -1) if single else inputs
        m, ln = x2.shape
        if out is None:
            if dev:
                import torch

                out = torch.empty((m, 4), dtype=x2.dtype, device=x2.device)
            else:
                out = np.empty((m, 4), dtype=np.uint64)
        bi, bo = _Buf(x2), _Buf(out, writable=True)
        ctx.check(ctx._lib.gl_poseidon_hash_no_pad_batch(ctx._h, bi.ptr, ln, m, bo.ptr, _same_space(bi, bo)))
        return out.reshape(4) if single else out

    @staticmethod
    def hash_pad(inputs, ctx: Optional[Context] = None):
        """Hasher::hash_pad: append 1, zeros, 1 up to a multiple of SPONGE_WIDTH, then hash_no_pad
        (this fork generation pads to the width: src/smt/goldilocks_poseidon/mod.rs:167-181 must equal
        src/smt/gadgets/common.rs:87-101).  Host inputs only (the padding is a host-side reshape)."""
        x = _h(inputs)
        single = x.ndim == 1
        x2 = x.reshape(1, -1) if single else x
        m, ln = x2.shape
        total = ln + 2
        while total % PoseidonHash.SPONGE_WIDTH:
            total += 1
        padded = np.zeros((m, total), dtype=np.uint64)
        padded[:, :ln] = x2
        padded[:, ln] = 1
        padded[:, total - 1] = 1
        out = PoseidonHash.hash_no_pad(padded, ctx=ctx)
        return out.reshape(4) if single else out

    @staticmethod
    def hash_or_noop(inputs, ctx: Optional[Context] = None):
        """Hasher::hash_or_noop: rows of at most 4 elements are zero-padded copies, else hash_no_pad."""
        x = _h(inputs)
        single = x.ndim == 1
        x2 = x.reshape(1, -1) if single else x
        if x2.shape[1] <= 4:
            out = np.zeros((x2.shape[0], 4), dtype=np.uint64)
            out[:, : x2.shape[1]] = x2 % np.uint64(P)
        else:
            out = PoseidonHash.hash_no_pad(x2, ctx=ctx)
        return out.reshape(4) if single else out


# ------------------------------------------------------------------------------------------------
# plonky2::hash::merkle_tree::MerkleTree
# ------------------------------------------------------------------------------------------------
def _prove_from_digests(digests: np.ndarray, num_leaves: int, cap_height: int, leaf_index: int) -> np.ndarray:
    """MerkleTree::prove's index walk over the in-order digest buffer."""
    L = num_leaves.bit_length() - 1 - cap_height
    if L <= 0:
        return np.zeros((0, 4), dtype=np.uint64)
    per = 2 * ((1 << L) - 1)
    sub = leaf_index >> L
    buf = digests[sub * per : (sub + 1) * per]
    pair = leaf_index & ((1 << L) - 1)
    sib = np.empty((L, 4), dtype=np.uint64)
    for i in range(L):
        parity = pair & 1
        pair >>= 1
        sib[i] = buf[2 * ((pair << (i + 1)) + (1 << i) - 1) + (1 - parity)]
    return sib


class MerkleTree:
    """MerkleTree<F, PoseidonHash>{leaves, digests, cap}."""

    def __init__(self, leaves: np.ndarray, digests: np.ndarray, cap: np.ndarray, cap_height: int):
        self.leaves, self.digests, self.cap, self.cap_height = leaves, digests, cap, cap_height

    @classmethod
    def new(cls, leaves, cap_height: int, ctx: Optional[Context] = None) -> "MerkleTree":
        ctx = _ctx(ctx)
        leaves = _h(leaves)
        if leaves.ndim != 2:
            raise GlPanic(N.GL_E_ARG, "MerkleTree::new: leaves must be [num_leaves][leaf_len]")
        n, ll = leaves.shape
        nd = max(2 * (n - (1 << cap_height)), 0)
        digests = np.empty((nd, 4), dtype=np.uint64)
        cap = np.empty((1 << cap_height, 4), dtype=np.uint64)
        bl, bd, bc = _Buf(leaves), _Buf(digests, True), _Buf(cap, True)
        ctx.check(ctx._lib.gl_merkle_build(ctx._h, bl.ptr, n, ll, cap_height, bd.ptr, bc.ptr, N.GL_HOST))
        return cls(leaves, digests, cap, cap_height)

    def get(self, i: int) -> np.ndarray:
        return self.leaves[i]

    def prove(self, leaf_index: int) -> np.ndarray:
        """MerkleProof.siblings, leaf level first: [log2(num_leaves) - cap_height][4]."""
        return _prove_from_digests(self.digests, self.leaves.shape[0], self.cap_height, leaf_index)


class ResidentMerkleTree:
    """The merkle_tree of a device-resident PolynomialBatch: cap on the host, leaves and digests behind
    the gl_commit handle.  `.leaves` / `.digests` download the mirror on first use ("mirror mode")."""

    def __init__(self, batch: "PolynomialBatch", cap: np.ndarray):
        self._b = batch
        self.cap = cap
        self.cap_height = batch.cap_height
        self._leaves = None
        self._digests = None

    def _mirror(self, want_leaves: bool, want_digests: bool):
        b = self._b
        lib, ctx = b._ctx._lib, b._ctx
        if want_leaves and self._leaves is None:
            self._leaves = np.empty((b.num_local_leaves, b.leaf_len), dtype=np.uint64)
            ctx.check(lib.gl_commit_download(b._h, self._leaves.ctypes.data, None, N.GL_HOST))
        if want_digests and self._digests is None:
            nd = 2 * (b.num_local_leaves - (1 << b.cap_local_bits))
            self._digests = np.empty((nd, 4), dtype=np.uint64)
            ctx.check(lib.gl_commit_download(b._h, None, self._digests.ctypes.data, N.GL_HOST))

    @property
    def leaves(self) -> np.ndarray:
        self._mirror(True, False)
        return self._leaves

    @property
    def digests(self) -> np.ndarray:
        self._mirror(False, True)
        return self._digests

    def get(self, i: int) -> np.ndarray:
        return self._b.open([i])[0][0]

    def prove(self, leaf_index: int) -> np.ndarray:
        return self._b.open([leaf_index])[1][0]


def merkle_verify_batch(leaves, leaf_indices, paths, cap, ctx: Optional[Context] = None) -> np.ndarray:
    """verify_merkle_proof_to_cap (plonky2::hash::merkle_proofs) for k proofs against one cap: leaves [k][leaf_len],
    leaf_indices [k], paths [k][L][4] (what PolynomialBatch.open / MerkleTree.prove return), cap [2^h][4].
    Returns a bool array: does proof i lead to its cap entry."""
    ctx = _ctx(ctx)
    lv, ix, pt, cp = _h(leaves), _h(leaf_indices).reshape(-1), _h(paths), _h(cap).reshape(-1, 4)
    k = ix.shape[0]
    if lv.ndim != 2 or lv.shape[0] != k or pt.ndim != 3 or pt.shape[0] != k or pt.shape[2] != 4:
        raise GlPanic(N.GL_E_ARG, "merkle_verify_batch: leaves [k][len], leaf_indices [k], paths [k][L][4] expected")
    h = cp.shape[0]
    if h == 0 or h & (h - 1):
        raise GlPanic(N.GL_E_ARG, "merkle_verify_batch: the cap must hold a power of two of digests")
    ok = np.zeros(k, dtype=np.int32)
    ctx.check(ctx._lib.gl_merkle_verify_batch(ctx._h, lv.ctypes.data, lv.shape[1], ix.ctypes.data, pt.ctypes.data, pt.shape[1],
                                              cp.ctypes.data, h.bit_length() - 1, k, ok.ctypes.data, N.GL_HOST))
    return ok.astype(bool)


# ------------------------------------------------------------------------------------------------
# plonky2::fri::oracle::PolynomialBatch
# ------------------------------------------------------------------------------------------------
class PolynomialBatch:
    """PolynomialBatch{polynomials, merkle_tree, degree_log, rate_bits, blinding}, LDE resident on the device."""

    def __init__(self):
        raise TypeError("use PolynomialBatch.from_values / from_coeffs")

    @classmethod
    def _make(cls, inputs, is_values: bool, rate_bits: int, blinding: bool, cap_height: int, ctx, want_coeffs):
        blinding = bool(blinding)
        ctx = _ctx(ctx)
        if isinstance(inputs, (list, tuple)) and inputs and all(isinstance(a, np.ndarray) and a.ndim == 1 for a in inputs):
            return cls._make_cols(list(inputs), is_values, rate_bits, blinding, cap_height, ctx, want_coeffs)
        dev = _is_torch(inputs) and inputs.is_cuda
        if not dev:
            inputs = _h(inputs)
        if inputs.ndim != 2:
            raise GlPanic(N.GL_E_ARG, "polynomials must be [columns][n]")
        c, n = int(inputs.shape[0]), int(inputs.shape[1])
        if n == 0 or n & (n - 1):
            raise GlPanic(N.GL_E_ARG, "log2_strict: polynomial length is not a power of two")
        lg = n.bit_length() - 1
        self = object.__new__(cls)
        self._ctx = ctx
        self.degree_log, self.rate_bits, self.blinding, self.cap_height = lg, rate_bits, blinding, cap_height
        self.num_columns = c
        cap = np.zeros((1 << cap_height, 4), dtype=np.uint64)
        h = C.c_void_p()
        bi = _Buf(inputs)
        self._polys = None
        if dev:
            import torch

            cap_dev = torch.zeros((1 << cap_height, 4), dtype=inputs.dtype, device=inputs.device)
            bc = _Buf(cap_dev, True)
        else:
            bc = _Buf(cap, True)
        if is_values:
            co = None
            if want_coeffs:
                if dev:
                    import torch

                    co = torch.empty_like(inputs)
                else:
                    co = np.empty_like(inputs)
            bo = _Buf(co, True)
            if blinding:
                rc = ctx._lib.gl_commit_from_values_ex(ctx._h, bi.ptr, None, lg, c, rate_bits, 1, cap_height, bo.ptr, None, bc.ptr,
                                                       C.byref(h), bi.space)
            else:
                rc = ctx._lib.gl_commit_from_values(ctx._h, bi.ptr, lg, c, rate_bits, cap_height, bo.ptr, bc.ptr, C.byref(h), bi.space)
            self._polys = co
        else:
            if blinding:
                rc = ctx._lib.gl_commit_from_coeffs_ex(ctx._h, bi.ptr, None, lg, c, rate_bits, 1, cap_height, bc.ptr, C.byref(h), bi.space)
            else:
                rc = ctx._lib.gl_commit_from_coeffs(ctx._h, bi.ptr, lg, c, rate_bits, cap_height, bc.ptr, C.byref(h), bi.space)
            self._polys = inputs
        ctx.check(rc)
        if dev:
            cap = cap_dev.cpu().numpy().view(np.uint64)
        self._finish_make(h, cap, n)
        return self

    @classmethod
    def _make_cols(cls, cols, is_values: bool, rate_bits: int, blinding: bool, cap_height: int, ctx, want_coeffs):
        """One host array per polynomial, as the reference holds them (Vec<PolynomialValues<F>>): no flattening,
        gl_commit_from_values_cols / gl_commit_from_coeffs_cols."""
        cols = [_h(a) for a in cols]
        c, n = len(cols), int(cols[0].shape[0])
        if any(a.shape[0] != n for a in cols):
            raise GlPanic(N.GL_E_ARG, "assert_eq!(p.len(), degree): polynomials of different lengths")
        if n == 0 or n & (n - 1):
            raise GlPanic(N.GL_E_ARG, "log2_strict: polynomial length is not a power of two")
        lg = n.bit_length() - 1
        self = object.__new__(cls)
        self._ctx = ctx
        self.degree_log, self.rate_bits, self.blinding, self.cap_height = lg, rate_bits, blinding, cap_height
        self.num_columns = c
        cap = np.zeros((1 << cap_height, 4), dtype=np.uint64)
        h = C.c_void_p()
        ptrs = (C.c_void_p * c)(*[a.ctypes.data for a in cols])
        if is_values:
            co, optrs = None, None
            if want_coeffs:
                co = [np.empty(n, dtype=np.uint64) for _ in range(c)]
                optrs = (C.c_void_p * c)(*[a.ctypes.data for a in co])
            if blinding:
                rc = ctx._lib.gl_commit_from_values_ex(ctx._h, None, ptrs, lg, c, rate_bits, 1, cap_height, None, optrs, cap.ctypes.data,
                                                       C.byref(h), N.GL_HOST)
            else:
                rc = ctx._lib.gl_commit_from_values_cols(ctx._h, ptrs, lg, c, rate_bits, cap_height, optrs, cap.ctypes.data, C.byref(h))
            self._polys = co
        else:
            if blinding:
                rc = ctx._lib.gl_commit_from_coeffs_ex(ctx._h, None, ptrs, lg, c, rate_bits, 1, cap_height, cap.ctypes.data, C.byref(h),
                                                       N.GL_HOST)
            else:
                rc = ctx._lib.gl_commit_from_coeffs_cols(ctx._h, ptrs, lg, c, rate_bits, cap_height, cap.ctypes.data, C.byref(h))
            self._polys = cols
        ctx.check(rc)
        self._finish_make(h, cap, n)
        return self

    def _finish_make(self, h, cap, n):
        ctx = self._ctx
        self._h = h
        lb, le = C.c_uint64(), C.c_uint64()
        ctx.check(ctx._lib.gl_commit_info(h, None, None, None, None, C.byref(lb), C.byref(le)))
        self.leaf_begin, self.leaf_end = lb.value, le.value
        self.num_local_leaves = le.value - lb.value
        ll = C.c_uint32()
        ctx.check(ctx._lib.gl_commit_leaf_len(h, C.byref(ll)))
        self.leaf_len = ll.value   # MerkleTree.leaves[i].len(): num_columns, + SALT_SIZE when blinding
        total = n << self.rate_bits
        self.cap_local_bits = self.cap_height - ((total // self.num_local_leaves).bit_length() - 1)
        self.merkle_tree = ResidentMerkleTree(self, cap)

    @classmethod
    def from_values(cls, values, rate_bits: int, blinding: bool, cap_height: int, timing=None, fft_root_table=None,
                    ctx: Optional[Context] = None, want_coeffs: bool = True) -> "PolynomialBatch":
        """values: [columns][n] evaluations on the subgroup (Vec<PolynomialValues<F>>), or a list of 1-D arrays
        (one per polynomial, never flattened: coefficients then come back the same way).  `timing` and
        `fft_root_table` are accepted for signature parity and ignored (the device keeps its own tables)."""
        return cls._make(values, True, rate_bits, blinding, cap_height, ctx, want_coeffs)

    @classmethod
    def from_coeffs(cls, polynomials, rate_bits: int, blinding: bool, cap_height: int, timing=None,
                    fft_root_table=None, ctx: Optional[Context] = None) -> "PolynomialBatch":
        return cls._make(polynomials, False, rate_bits, blinding, cap_height, ctx, False)

    @property
    def polynomials(self):
        """Vec<PolynomialCoeffs<F>> as [columns][n]."""
        if self._polys is None:
            self._polys = np.empty((self.num_columns, 1 << self.degree_log), dtype=np.uint64)
            self._ctx.check(self._ctx._lib.gl_commit_coeffs(self._h, self._polys.ctypes.data, N.GL_HOST))
        return self._polys

    def eval_at(self, point) -> np.ndarray:
        """OpeningSet::new for this batch: every polynomial at the extension point (a0, a1) -> [columns][2], computed from
        the resident coefficients."""
        pt = (C.c_uint64 * 2)(int(point[0]) % P, int(point[1]) % P)
        out = np.empty((self.num_columns, 2), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.gl_commit_eval(self._h, pt, out.ctypes.data, N.GL_HOST))
        return out

    def get_lde_values(self, index, step: int) -> np.ndarray:
        """PolynomialBatch::get_lde_values(index, step) for one index or a list: [k][columns]."""
        idx = _h(np.atleast_1d(index))
        out = np.empty((idx.shape[0], self.num_columns), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.gl_commit_get_lde_values(self._h, idx.ctypes.data, idx.shape[0], step, out.ctypes.data, N.GL_HOST))
        return out[0] if np.ndim(index) == 0 else out

    def open(self, leaf_indices: Sequence[int]):
        """(rows [k][leaf_len], paths [k][L][4]) = (tree.get(i), tree.prove(i).siblings) for every i; a blinded batch's rows
        carry their SALT_SIZE salt elements after the polynomial values."""
        idx = _h(np.asarray(leaf_indices))
        k = idx.shape[0]
        L = self.degree_log + self.rate_bits - self.cap_height
        rows = np.empty((k, self.leaf_len), dtype=np.uint64)
        paths = np.empty((k, L, 4), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.gl_commit_open(self._h, idx.ctypes.data, k, rows.ctypes.data, paths.ctypes.data, N.GL_HOST))
        return rows, paths

    def device_ptrs(self):
        """(lde pointer, leading dimension, digests pointer) of the resident data (column-major leaves)."""
        a, b, ld = C.c_void_p(), C.c_void_p(), C.c_uint64()
        self._ctx.check(self._ctx._lib.gl_commit_device_ptrs(self._h, C.byref(a), C.byref(ld), C.byref(b)))
        return a.value, ld.value, b.value

    def free(self):
        if getattr(self, "_h", None) and self._ctx._h:
            self._ctx._lib.gl_commit_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------
# N3: plonky2::plonk::prover::compute_quotient_polys on the resident oracles
# ------------------------------------------------------------------------------------------------
GATE_NOOP, GATE_CONSTANT, GATE_PUBLIC_INPUT, GATE_U32_INTERLEAVE, GATE_UNINTERLEAVE_TO_U32, GATE_UNINTERLEAVE_TO_B32 = range(6)


def compute_quotient_polys(circuit, gates, k_is, constants_sigmas: "PolynomialBatch", wires: "PolynomialBatch",
                           zs_partial_products: "PolynomialBatch", public_inputs_hash, betas, gammas, alphas, ctx=None) -> np.ndarray:
    """compute_quotient_polys (prover step 8): the num_challenges * quotient_degree_factor coefficient chunks of the quotient,
    [chunks][n], from the three oracles resident on the device -- no LDE row crosses PCIe.  circuit: (degree_bits,
    num_wires, num_routed_wires, num_constants incl. selectors, num_selectors, num_challenges, quotient_degree_factor,
    num_gates); gates: [(kind, num_ops, selector_index, group_start, group_end)], gate i = index i.  The chunks go straight
    into PolynomialBatch.from_coeffs."""
    ctx = _ctx(ctx)
    cd = N.Circuit(*[int(v) for v in circuit])
    arr = (N.Gate * len(gates))(*[N.Gate(*[int(v) for v in tuple(g)[:5]], 0) for g in gates])
    k, pih, b, g, a = _h(k_is), _h(public_inputs_hash), _h(betas), _h(gammas), _h(alphas)
    n = 1 << cd.degree_bits
    out = np.empty((cd.num_challenges * cd.quotient_degree_factor, n), dtype=np.uint64)
    ctx.check(ctx._lib.gl_quotient_polys(ctx._h, C.byref(cd), arr, k.ctypes.data, constants_sigmas._h, wires._h, zs_partial_products._h,
                                         pih.ctypes.data, b.ctypes.data, g.ctypes.data, a.ctypes.data, out.ctypes.data, N.GL_HOST))
    return out


def permutation_zs(circuit, k_is, constants_sigmas: "PolynomialBatch", wires: "PolynomialBatch", betas, gammas, out=None,
                   ctx=None):
    """all_wires_permutation_partial_products (prover step 3): the Z and partial-product columns, values on the subgroup,
    [num_challenges * ceil(num_routed_wires / quotient_degree_factor)][n] in the order the prover commits them, computed from
    the coefficients the two resident commits hold.  circuit: the same tuple as compute_quotient_polys takes.  out: None (a
    new numpy array), a numpy array, a torch CUDA tensor or a DeviceBuffer (the columns stay on the device and go straight
    into PolynomialBatch.from_values).  Returns (zs, grand_products): grand_products[c] is 1 exactly when the witness
    satisfies every copy constraint; a product other than 1 is returned, not raised."""
    ctx = _ctx(ctx)
    cd = N.Circuit(*[int(v) for v in circuit])
    k, b, g = _h(k_is), _h(betas), _h(gammas)
    nch = cd.num_challenges
    if len(b) < nch or len(g) < nch:
        raise GlPanic(N.GL_E_ARG, "permutation_zs: fewer betas / gammas than num_challenges")
    if len(k) < cd.num_routed_wires:
        raise GlPanic(N.GL_E_ARG, "permutation_zs: fewer k_is than num_routed_wires")
    deg = max(cd.quotient_degree_factor, 1)
    shape = (nch * -(-cd.num_routed_wires // deg), 1 << cd.degree_bits)
    if out is None:
        out = np.empty(shape, dtype=np.uint64)
    o = _Buf(out, writable=True)
    if o.nbytes < shape[0] * shape[1] * 8:
        raise GlPanic(N.GL_E_ARG, "permutation_zs: output buffer too small")
    grand = np.zeros(max(nch, 1), dtype=np.uint64)
    ctx.check(ctx._lib.gl_permutation_zs(ctx._h, C.byref(cd), k.ctypes.data, constants_sigmas._h, wires._h, b.ctypes.data,
                                         g.ctypes.data, o.ptr, o.space, grand.ctypes.data))
    return out, grand[:nch]


def opening_set_lengths(circuit) -> dict:
    """OpeningSet field -> number of extension values, for a circuit tuple as compute_quotient_polys takes it."""
    cd = N.Circuit(*[int(v) for v in circuit])
    nch, qdf = cd.num_challenges, cd.quotient_degree_factor
    num_prods = -(-cd.num_routed_wires // qdf) - 1
    return dict(zip(wire.OPENING_SET_FIELDS, (cd.num_constants, cd.num_routed_wires, cd.num_wires, nch, nch, nch * num_prods, nch * qdf)))


def prove(circuit, gates, k_is, constants_sigmas: "PolynomialBatch", circuit_digest, fri_params, wires, public_inputs=(),
          ctx=None) -> dict:
    """plonky2::plonk::prover::prove from the witness on, in one call (gl_prove): the wires, Z and quotient commits, the
    transcript, the OpeningSet and the opening proof all on the device; one copy brings the proof back.  circuit / gates /
    k_is as compute_quotient_polys takes them; constants_sigmas: the resident prover-data commit; circuit_digest: the four
    elements of prover_data.circuit_digest; fri_params: fri.FriParams.  wires: the witness [num_wires][n] as a numpy array, a
    list of 1-D numpy arrays (one per wire), a torch CUDA tensor or a DeviceBuffer.  Returns dict(caps=(wires_cap,
    plonk_zs_partial_products_cap, quotient_polys_cap), openings={OpeningSet field: [k][2]}, opening_proof=FriProof as
    fri.parse_flat_proof gives it, public_inputs, words=the stream gl_prove wrote); wire.proof_with_public_inputs_to_bytes
    turns it into ProofWithPublicInputs bytes."""
    from .fri import c_params, parse_flat_proof

    ctx = _ctx(ctx)
    cd = N.Circuit(*[int(v) for v in circuit])
    arr = (N.Gate * len(gates))(*[N.Gate(*[int(v) for v in tuple(g)[:5]], 0) for g in gates])
    k, digest, pis = _h(k_is), _h(circuit_digest), _h(public_inputs).reshape(-1)
    if len(k) < cd.num_routed_wires or digest.shape != (4,) or len(gates) < cd.num_gates:
        raise GlPanic(N.GL_E_ARG, "prove: fewer k_is than num_routed_wires or gates than num_gates, or a circuit digest that is "
                                  "not four elements")
    prm = c_params(fri_params)
    # the library reads num_wires x 2^degree_bits words of witness and cannot check the caller's sizes: they are checked here
    n = 1 << cd.degree_bits
    flat, cols, space, keep = None, None, N.GL_HOST, None
    if isinstance(wires, (list, tuple)):
        keep = [_h(w) for w in wires]
        if len(keep) != cd.num_wires or any(w.shape != (n,) for w in keep):
            raise GlPanic(N.GL_E_ARG, f"prove: the witness must be num_wires = {cd.num_wires} columns of 2^degree_bits = {n} values")
        cols = (C.c_void_p * len(keep))(*[w.ctypes.data for w in keep])
    else:
        dev = isinstance(wires, DeviceBuffer) or _is_torch(wires)
        b = _Buf(wires if dev else _h(wires))
        if (b.nbytes < cd.num_wires * n * 8) if dev else (b.keep.shape != (cd.num_wires, n)):
            raise GlPanic(N.GL_E_ARG, f"prove: the witness must be [num_wires = {cd.num_wires}][2^degree_bits = {n}]")
        flat, space, keep = b.ptr, b.space, b
    words = C.c_uint64(0)
    args = (ctx._h, C.byref(cd), arr, k.ctypes.data, constants_sigmas._h, digest.ctypes.data, C.byref(prm), flat, cols, space,
            pis.ctypes.data, pis.size)
    rc = ctx._lib.gl_prove(*args, None, 0, C.byref(words))     # the size: a NULL buffer is rejected after it is set
    if words.value == 0:
        ctx.check(rc)
    out = np.empty(words.value, dtype=np.uint64)
    ctx.check(ctx._lib.gl_prove(*args, out.ctypes.data, out.size, C.byref(words)))
    del keep
    h = fri_params.config.cap_height
    at = 0
    caps = []
    for _ in range(3):
        caps.append(out[at:at + (4 << h)].reshape(-1, 4))
        at += 4 << h
    lens = opening_set_lengths(circuit)
    openings = {}
    for f, cnt in lens.items():
        openings[f] = out[at:at + 2 * cnt].reshape(-1, 2)
        at += 2 * cnt
    widths = [constants_sigmas.leaf_len, cd.num_wires, lens["plonk_zs"] + lens["partial_products"], lens["quotient_polys"]]
    return {"caps": tuple(caps), "openings": openings, "opening_proof": parse_flat_proof(out[at:], widths, fri_params),
            "public_inputs": pis.copy(), "words": out}


# ------------------------------------------------------------------------------------------------
# gl_group: one commit sharded over several GPUs, NCCL behind the C ABI (SURVEY 8e)
# ------------------------------------------------------------------------------------------------
class Group:
    """gl_group.  `Group.local(devices)` holds every rank in this process (what a Rust prover driving a whole box does);
    `Group.from_token(ctx, rank, nranks, token)` holds one rank of a group that spans processes (rank 0 makes the token
    with `Group.unique_id()` and hands the 128 bytes to the others, e.g. over torch.distributed or a file)."""

    @staticmethod
    def _share_torch_nccl():
        """libgl_b200.so binds NCCL with dlopen at its first gl_group_* call and prefers a copy the process already holds.
        A Python process that will ALSO use torch must let torch load its bundled NCCL first: loading the system
        libnccl.so.2 before `import torch` makes the loader hand that older copy to libtorch_cuda (same SONAME) and the
        import fails with missing symbols.  (A host without torch -- the Rust prover -- just gets the system NCCL.)"""
        try:
            import torch  # noqa: F401
        except Exception:
            pass

    def __init__(self, ctxs: Sequence[Context], rank0: int, nranks: int, token: Optional[bytes]):
        self._share_torch_nccl()
        self._lib = N.load()
        self.ctxs = list(ctxs)
        self.nlocal, self.rank0, self.nranks = len(self.ctxs), rank0, nranks
        arr = (C.c_void_p * self.nlocal)(*[c._h for c in self.ctxs])
        tok = (C.c_uint8 * N.GL_GROUP_ID_BYTES).from_buffer_copy(token) if token is not None else None
        h = C.c_void_p()
        rc = self._lib.gl_group_create(arr, self.nlocal, rank0, nranks, tok, C.byref(h))
        if rc:
            raise GlPanic(rc, (self._lib.gl_group_last_error(None) or b"").decode())
        self._h = h

    @staticmethod
    def unique_id() -> bytes:
        Group._share_torch_nccl()
        lib = N.load()
        buf = (C.c_uint8 * N.GL_GROUP_ID_BYTES)()
        rc = lib.gl_group_unique_id(buf)
        if rc:
            raise GlPanic(rc, (lib.gl_group_last_error(None) or b"").decode())
        return bytes(buf)

    @classmethod
    def local(cls, devices: Sequence[int]) -> "Group":
        return cls([Context(d) for d in devices], 0, len(devices), None)

    @classmethod
    def from_token(cls, ctx: Context, rank: int, nranks: int, token: bytes) -> "Group":
        return cls([ctx], rank, nranks, token)

    def check(self, rc: int):
        if rc:
            raise GlPanic(rc, (self._lib.gl_group_last_error(self._h) or b"").decode())

    @property
    def nccl_version(self) -> int:
        v = C.c_int(0)
        self.check(self._lib.gl_group_info(self._h, None, None, None, C.byref(v)))
        return v.value

    def commit_phase_ms(self) -> dict:
        out = (C.c_float * 6)()
        self.check(self._lib.gl_group_commit_phase_ms(self._h, out))
        return dict(zip(Context.PHASES, [float(x) for x in out]))

    def commit(self, inputs, rate_bits: int, cap_height: int, is_values: bool = True, want_coeffs: bool = True,
               stream_hash: bool = False, blinding: bool = False) -> "ShardedPolynomialBatch":
        """PolynomialBatch::from_values / from_coeffs over the group.  `inputs`: one host array [c][n] (shared by the local
        ranks), or a list with one CUDA tensor per local rank (the whole batch on each GPU)."""
        dev = isinstance(inputs, (list, tuple)) and len(inputs) == self.nlocal and all(_is_torch(x) and x.is_cuda for x in inputs)
        if dev:
            c, n = int(inputs[0].shape[0]), int(inputs[0].shape[1])
            bufs = [_Buf(x) for x in inputs]
            ptrs = (C.c_void_p * self.nlocal)(*[b.ptr for b in bufs])
            space = N.GL_DEVICE
        else:
            inputs = _h(inputs)
            if inputs.ndim != 2:
                raise GlPanic(N.GL_E_ARG, "polynomials must be [columns][n]")
            c, n = int(inputs.shape[0]), int(inputs.shape[1])
            ptrs = (C.c_void_p * self.nlocal)(*[inputs.ctypes.data] * self.nlocal)
            space = N.GL_HOST
        if n == 0 or n & (n - 1):
            raise GlPanic(N.GL_E_ARG, "log2_strict: polynomial length is not a power of two")
        lg = n.bit_length() - 1
        caps = [np.zeros((1 << cap_height, 4), dtype=np.uint64) for _ in range(self.nlocal)]
        coeffs = None
        hs = (C.c_void_p * self.nlocal)()
        flags = (N.GL_COMMIT_STREAM_HASH if stream_hash else 0) | (N.GL_COMMIT_BLINDING if blinding else 0)
        if dev:
            import torch

            cap_dev = [torch.zeros((1 << cap_height, 4), dtype=torch.int64, device=x.device) for x in inputs]
            cap_ptrs = (C.c_void_p * self.nlocal)(*[t.data_ptr() for t in cap_dev])
        else:
            cap_ptrs = (C.c_void_p * self.nlocal)(*[a.ctypes.data for a in caps])
        if is_values:
            co_ptrs = None
            if want_coeffs:
                if dev:
                    import torch

                    coeffs = [torch.empty_like(x) for x in inputs]
                    co_ptrs = (C.c_void_p * self.nlocal)(*[t.data_ptr() for t in coeffs])
                else:
                    coeffs = np.zeros_like(inputs)      # every local rank writes ITS polynomials into the one array
                    co_ptrs = (C.c_void_p * self.nlocal)(*[coeffs.ctypes.data] * self.nlocal)
            rc = self._lib.gl_group_commit_from_values(self._h, ptrs, lg, c, rate_bits, cap_height, co_ptrs, cap_ptrs, hs, space, flags)
        else:
            rc = self._lib.gl_group_commit_from_coeffs(self._h, ptrs, lg, c, rate_bits, cap_height, cap_ptrs, hs, space, flags)
        self.check(rc)
        if dev:
            caps = [t.cpu().numpy().view(np.uint64) for t in cap_dev]
        return ShardedPolynomialBatch(self, [C.c_void_p(h) for h in hs], caps, coeffs, lg, c, rate_bits, cap_height,
                                      c + (N.GL_SALT_SIZE if blinding else 0))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gl_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ShardedPolynomialBatch:
    """The local shards of one PolynomialBatch committed over a Group: the whole cap on every rank, `open` for any leaf."""

    def __init__(self, group: Group, handles, caps, coeffs, degree_log, c, rate_bits, cap_height, leaf_len=None):
        self.group, self._hs, self.caps, self.coeffs = group, handles, caps, coeffs
        self._degree_log, self.num_columns, self.rate_bits, self.cap_height = degree_log, c, rate_bits, cap_height
        self.leaf_len = leaf_len or c          # c + SALT_SIZE for a blinded commit
        self.cap = caps[0]

    @property
    def _h(self):
        """The first local rank's shard: every rank holds ALL coefficients after the all-gather, so OpeningSet::new and
        the FRI polynomial (gl_commit_eval, gl_fri_final_poly) run on any one rank; only leaves / digests are sharded."""
        return self._hs[0]

    @property
    def degree_log(self) -> int:
        return self._degree_log

    def eval_at(self, point) -> np.ndarray:
        ctx = self.group.ctxs[0]
        pt = (C.c_uint64 * 2)(int(point[0]) % P, int(point[1]) % P)
        out = np.empty((self.num_columns, 2), dtype=np.uint64)
        ctx.check(ctx._lib.gl_commit_eval(self._h, pt, out.ctypes.data, N.GL_HOST))
        return out

    def open(self, leaf_indices: Sequence[int]):
        """(rows [k][c], paths [k][L][4]) for GLOBAL leaf indices, whoever owns them (gl_group_commit_open); the same
        arrays on every local rank, the first rank's are returned."""
        g = self.group
        idx = _h(np.asarray(leaf_indices))
        k = idx.shape[0]
        L = self._degree_log + self.rate_bits - self.cap_height
        rows = [np.empty((k, self.leaf_len), dtype=np.uint64) for _ in range(g.nlocal)]
        paths = [np.empty((k, L, 4), dtype=np.uint64) for _ in range(g.nlocal)]
        hs = (C.c_void_p * g.nlocal)(*[h.value for h in self._hs])
        rp = (C.c_void_p * g.nlocal)(*[a.ctypes.data for a in rows])
        pp = (C.c_void_p * g.nlocal)(*[a.ctypes.data for a in paths])
        g.check(g._lib.gl_group_commit_open(g._h, hs, idx.ctypes.data, k, rp, pp, N.GL_HOST))
        self.all_rows, self.all_paths = rows, paths
        return rows[0], paths[0]

    def free(self):
        for h in self._hs:
            if h and h.value:
                self.group._lib.gl_commit_free(h)
        self._hs = []

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------
# plonky2_field::fft / polynomial
# ------------------------------------------------------------------------------------------------
def _fft_call(name, data, shift, ctx):
    ctx = _ctx(ctx)
    dev = _is_torch(data) and data.is_cuda
    if not dev:
        data = _h(data).copy()
    single = data.ndim == 1
    d2 = data.reshape(1, -1) if single else data
    c, n = d2.shape
    if n == 0 or n & (n - 1):
        raise GlPanic(N.GL_E_ARG, "log2_strict: length is not a power of two")
    b = _Buf(d2, True)
    fn = getattr(ctx._lib, name)
    if shift is None:
        ctx.check(fn(ctx._h, b.ptr, n.bit_length() - 1, c, b.space))
    else:
        ctx.check(fn(ctx._h, b.ptr, n.bit_length() - 1, c, shift, b.space))
    return d2.reshape(-1) if single else d2


def fft(coeffs, ctx=None):
    """PolynomialCoeffs::fft over [c][n] (or [n])."""
    return _fft_call("gl_fft_batch", coeffs, None, ctx)


def ifft(values, ctx=None):
    """PolynomialValues::ifft."""
    return _fft_call("gl_ifft_batch", values, None, ctx)


def coset_fft(coeffs, shift: int = 7, ctx=None):
    return _fft_call("gl_coset_fft_batch", coeffs, shift, ctx)


def coset_ifft(values, shift: int = 7, ctx=None):
    return _fft_call("gl_coset_ifft_batch", values, shift, ctx)


# ------------------------------------------------------------------------------------------------
# plonky2::fri  (configuration + the data-parallel pieces of fri_committed_trees / fri_proof_of_work)
# ------------------------------------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class FriReductionStrategy:
    """ConstantArityBits(arity_bits, final_poly_bits)."""

    arity_bits: int = 4
    final_poly_bits: int = 5

    def reduction_arity_bits(self, degree_bits: int, rate_bits: int, cap_height: int) -> list:
        out = []
        d = degree_bits
        while d > self.final_poly_bits and d + rate_bits - self.arity_bits >= cap_height:
            out.append(self.arity_bits)
            d -= self.arity_bits
        return out


@dataclasses.dataclass(frozen=True)
class FriConfig:
    rate_bits: int = 3
    cap_height: int = 4
    proof_of_work_bits: int = 16
    reduction_strategy: FriReductionStrategy = FriReductionStrategy()
    num_query_rounds: int = 28


@dataclasses.dataclass(frozen=True)
class CircuitConfig:
    num_wires: int = 135
    num_routed_wires: int = 80
    num_constants: int = 2
    num_challenges: int = 2
    zero_knowledge: bool = False
    max_quotient_degree_factor: int = 8
    fri_config: FriConfig = FriConfig()

    @staticmethod
    def standard_recursion_config() -> "CircuitConfig":
        return CircuitConfig()

    @staticmethod
    def standard_ecc_config() -> "CircuitConfig":
        return CircuitConfig(num_wires=136)

    @staticmethod
    def wide_ecc_config() -> "CircuitConfig":
        return CircuitConfig(num_wires=234)


def fri_layer_tree(values_ext, arity_bits: int, cap_height: int, want_digests: bool = True, ctx=None):
    """One layer of fri_committed_trees: (digests, cap) of MerkleTree::new over the bit-reversed,
    arity-chunked extension values [len][2]."""
    ctx = _ctx(ctx)
    v = _h(values_ext)
    ln = v.shape[0]
    nl = ln >> arity_bits
    nd = max(2 * (nl - (1 << cap_height)), 0)
    digests = np.empty((nd, 4), dtype=np.uint64) if want_digests else None
    cap = np.empty((1 << cap_height, 4), dtype=np.uint64)
    ctx.check(ctx._lib.gl_fri_layer_tree(ctx._h, v.ctypes.data, ln, arity_bits, cap_height,
                                          digests.ctypes.data if want_digests else None, cap.ctypes.data, N.GL_HOST))
    return digests, cap


def fri_fold(coeffs_ext, arity_bits: int, beta, shift: int, ctx=None):
    """(folded coefficients, their values on shift * <w>) for one FRI reduction."""
    ctx = _ctx(ctx)
    cf = _h(coeffs_ext)
    ln = cf.shape[0]
    out_len = ln >> arity_bits
    folded = np.empty((out_len, 2), dtype=np.uint64)
    nxt = np.empty((out_len, 2), dtype=np.uint64)
    b = (C.c_uint64 * 2)(int(beta[0]), int(beta[1]))
    ctx.check(ctx._lib.gl_fri_fold(ctx._h, cf.ctypes.data, ln, arity_bits, b, shift, folded.ctypes.data, nxt.ctypes.data, N.GL_HOST))
    return folded, nxt


def fri_proof_of_work(state12, input_pos: int, min_leading_zeros: int, ctx=None) -> int:
    """Deterministic fri_proof_of_work: the smallest witness."""
    ctx = _ctx(ctx)
    s = (C.c_uint64 * 12)(*[int(x) for x in state12])
    w = C.c_uint64()
    ctx.check(ctx._lib.gl_pow_grind(ctx._h, s, input_pos, min_leading_zeros, C.byref(w)))
    return w.value


# ------------------------------------------------------------------------------------------------
# src/smt: PoseidonNodeHash + SparseMerkleProcessProof::check over batches
# ------------------------------------------------------------------------------------------------
class PoseidonNodeHash:
    """NodeHash for the Poseidon SMT (src/smt/goldilocks_poseidon/mod.rs:158-184), batched."""

    @staticmethod
    def calc_leaf_hash(keys, values, ctx=None):
        ctx = _ctx(ctx)
        k, v = _h(keys), _h(values)
        single = k.ndim == 1
        k2, v2 = k.reshape(-1, 4), v.reshape(-1, 4)
        out = np.empty_like(k2)
        ctx.check(ctx._lib.gl_smt_leaf_hash_batch(ctx._h, k2.ctypes.data, v2.ctypes.data, out.ctypes.data, k2.shape[0], N.GL_HOST))
        return out.reshape(4) if single else out

    @staticmethod
    def calc_internal_hash(left, right, ctx=None):
        return PoseidonHash.two_to_one(left, right, ctx=ctx)


PROCESS_NOOP, PROCESS_UPDATE, PROCESS_INSERT, PROCESS_DELETE = 0, 1, 2, 3

SMT_HDR_DTYPE = np.dtype(
    [("old_root", "<u8", 4), ("old_key", "<u8", 4), ("old_value", "<u8", 4),
     ("new_root", "<u8", 4), ("new_key", "<u8", 4), ("new_value", "<u8", 4),
     ("is_old0", "<u4"), ("fnc", "<u4")]
)
assert SMT_HDR_DTYPE.itemsize == C.sizeof(N.SmtProofHdr)


def smt_check_process_proofs(headers: np.ndarray, sib_pool: np.ndarray, sib_off: np.ndarray, ctx=None) -> np.ndarray:
    """SparseMerkleProcessProof::check for a batch.  status 0 = verify_smt_process_proof would return
    normally; k > 0 = its k-th assert would panic (DESIGN.md lists them)."""
    ctx = _ctx(ctx)
    hd = np.ascontiguousarray(headers, dtype=SMT_HDR_DTYPE)
    pool = _h(sib_pool).reshape(-1, 4)
    off = _h(sib_off)
    m = hd.shape[0]
    if off.shape[0] != m + 1:
        raise GlPanic(N.GL_E_ARG, "sib_off must have m + 1 entries")
    status = np.empty(m, dtype=np.int32)
    ctx.check(ctx._lib.gl_smt_verify_process_batch(ctx._h, hd.ctypes.data, pool.ctypes.data, off.ctypes.data, m, status.ctypes.data, N.GL_HOST))
    return status


def _smt_final_map(k: np.ndarray, v: np.ndarray):
    """What a sequence of `tree.set(k[t], v[t])` calls leaves: per key the LAST value, keys whose last value is zero are
    gone (set with the default value removes, src/smt/tree.rs:143-155).  The compact tree depends only on this map."""
    kc = np.where(k >= np.uint64(P), k - np.uint64(P), k)
    vc = np.where(v >= np.uint64(P), v - np.uint64(P), v)
    rows = np.ascontiguousarray(kc).view([("k", "<u8", 4)]).reshape(-1)
    _, first_rev = np.unique(rows[::-1], return_index=True)          # first occurrence in the reversed order = last call
    last = np.sort(kc.shape[0] - 1 - first_rev)
    keep = last[(vc[last] != 0).any(axis=1)]
    return np.ascontiguousarray(k[keep]), np.ascontiguousarray(v[keep])


def smt_build_tree(keys, values, want_nodes: bool = False, ctx=None):
    """N2: the sparse Merkle tree of src/smt/tree.rs holding `keys -> values`, built in one pass on the device.
    Returns root [4] (and, with want_nodes, the internal nodes [(hash, left, right)] as an [k][12] array plus the
    leaf hashes [m'][4] of the entries that remain): what m successive `tree.set(key, value)` calls leave in the root
    and node stores.  As with `set`, keys may repeat (the last value wins) and a zero value removes its key: such
    batches are first reduced to the map they leave (the tree is history independent); gl_smt_build itself takes
    distinct keys with non-zero values and returns GL_E_ARG otherwise, like SparseMerkleTree::insert."""
    ctx = _ctx(ctx)
    k, v = _h(keys).reshape(-1, 4), _h(values).reshape(-1, 4)
    if k.shape != v.shape:
        raise GlPanic(N.GL_E_ARG, "smt_build_tree: keys and values differ in shape")
    if ((v % np.uint64(P)) == 0).all(axis=1).any():     # removals in the batch: order matters, resolve it first
        k, v = _smt_final_map(k, v)
    try:
        return _smt_build_distinct(ctx, k, v, want_nodes)
    except GlPanic as e:
        if "already exists" not in str(e):
            raise
    k, v = _smt_final_map(k, v)                          # repeated keys: updates, the last value wins
    return _smt_build_distinct(ctx, k, v, want_nodes)


def _smt_build_distinct(ctx, k, v, want_nodes: bool):
    m = k.shape[0]
    root = np.zeros(4, dtype=np.uint64)
    count = C.c_uint64(0)
    if want_nodes:
        cap = max(4 * m + 1024, 1024)
        nodes = np.empty((cap, 12), dtype=np.uint64)
        leaf_hashes = np.empty((m, 4), dtype=np.uint64)
        while True:
            ctx.check(ctx._lib.gl_smt_build(ctx._h, k.ctypes.data, v.ctypes.data, m, root.ctypes.data, nodes.ctypes.data, cap,
                                            C.byref(count), leaf_hashes.ctypes.data, N.GL_HOST))
            if count.value <= cap:
                break
            cap = int(count.value)
            nodes = np.empty((cap, 12), dtype=np.uint64)
        return root, nodes[: count.value].copy(), leaf_hashes
    ctx.check(ctx._lib.gl_smt_build(ctx._h, k.ctypes.data, v.ctypes.data, m, root.ctypes.data, None, 0, C.byref(count), None,
                                    N.GL_HOST))
    return root


def smt_set_proofs(keys, values, ctx=None):
    """N2: the SparseMerkleProcessProofs of m successive `tree.set(keys[t], values[t])` calls on an EMPTY tree
    (src/smt/tree.rs:143-155), all computed in one pass on the device.  Keys may repeat and values may be zero, as with
    `set`: insert / update / delete / no-op.  Returns (headers [m] of SMT_HDR_DTYPE, sib_pool [total][4], sib_off [m + 1])
    -- the layout smt_check_process_proofs takes; the siblings of proof t are sib_pool[sib_off[t]:sib_off[t + 1]]."""
    ctx = _ctx(ctx)
    k, v = _h(keys).reshape(-1, 4), _h(values).reshape(-1, 4)
    if k.shape != v.shape:
        raise GlPanic(N.GL_E_ARG, "smt_set_proofs: keys and values differ in shape")
    m = k.shape[0]
    hdr = np.zeros(m, dtype=SMT_HDR_DTYPE)
    off = np.zeros(m + 1, dtype=np.uint64)
    total = C.c_uint64(0)
    cap = max(32 * m, 1024)       # a random batch needs ~ log2(m) siblings per proof
    while True:
        pool = np.empty((cap, 4), dtype=np.uint64)
        ctx.check(ctx._lib.gl_smt_set_proofs(ctx._h, k.ctypes.data, v.ctypes.data, m, hdr.ctypes.data, pool.ctypes.data, cap,
                                                off.ctypes.data, C.byref(total), N.GL_HOST))
        if total.value <= cap:
            return hdr, pool[: total.value].copy() if total.value < cap // 2 else pool[: total.value], off
        cap = int(total.value)


# ------------------------------------------------------------------------------------------------
# src/zkdsa: the native (non-circuit) side of the Poseidon signature scheme, over batches
# ------------------------------------------------------------------------------------------------
def zkdsa_public_keys(private_keys, ctx=None) -> np.ndarray:
    """private_key_to_public_key for every key: PoseidonHash::two_to_one(sk, sk) (src/zkdsa/account.rs:164-166)."""
    sk = _h(private_keys).reshape(-1, 4)
    return PoseidonHash.two_to_one(sk, sk, ctx=ctx)


def zkdsa_addresses(public_keys) -> np.ndarray:
    """public_key_to_address: the first element of the public key (src/zkdsa/account.rs:168-170)."""
    return _h(public_keys).reshape(-1, 4)[:, 0].copy()


def zkdsa_sign(private_keys, messages, ctx=None) -> np.ndarray:
    """SimpleSignature: PoseidonHash::two_to_one(private_key, message) (src/zkdsa/circuits/mod.rs:62-75)."""
    return PoseidonHash.two_to_one(_h(private_keys).reshape(-1, 4), _h(messages).reshape(-1, 4), ctx=ctx)


def zkdsa_public_inputs_json(message, public_key, signature) -> str:
    """SerializableSimpleSignaturePublicInputs as serde_json writes it (src/zkdsa/circuits/mod.rs:108-153)."""
    return ('{"message":"%s","public_key":"%s","signature":"%s"}'
            % (hash_out_to_hex(message), hash_out_to_hex(public_key), hash_out_to_hex(signature)))


SMT_INCLUSION_DTYPE = np.dtype(
    [("root", "<u8", 4), ("key", "<u8", 4), ("value", "<u8", 4), ("not_found_key", "<u8", 4), ("not_found_value", "<u8", 4),
     ("found", "<u4"), ("is_old0", "<u4")]
)


assert SMT_INCLUSION_DTYPE.itemsize == C.sizeof(N.SmtInclusionHdr)


def smt_find_batch(keys, values, queries, ctx=None):
    """`tree.find(q)` (src/smt/tree.rs:588-676) for every query against the tree that `tree.set(keys[t], values[t])`,
    t = 0 .. m-1, leave when they start from an empty tree.  Returns (SparseMerkleInclusionProof headers [nq] of
    SMT_INCLUSION_DTYPE, sib_pool [total][4], sib_off [nq + 1]); siblings of proof i = sib_pool[sib_off[i]:sib_off[i + 1]]."""
    ctx = _ctx(ctx)
    k, v, q = _h(keys).reshape(-1, 4), _h(values).reshape(-1, 4), _h(queries).reshape(-1, 4)
    if k.shape != v.shape:
        raise GlPanic(N.GL_E_ARG, "smt_find_batch: keys and values differ in shape")
    m, nq = k.shape[0], q.shape[0]
    hdr = np.zeros(nq, dtype=SMT_INCLUSION_DTYPE)
    off = np.zeros(nq + 1, dtype=np.uint64)
    total = C.c_uint64(0)
    cap = max(48 * nq, 1024)
    while True:
        pool = np.empty((cap, 4), dtype=np.uint64)
        ctx.check(ctx._lib.gl_smt_find_batch(ctx._h, k.ctypes.data, v.ctypes.data, m, q.ctypes.data, nq, hdr.ctypes.data,
                                             pool.ctypes.data, cap, off.ctypes.data, C.byref(total), N.GL_HOST))
        if total.value <= cap:
            return hdr, pool[: total.value].copy(), off
        cap = int(total.value)


# ------------------------------------------------------------------------------------------------
# serde_json forms of the SMT proofs (src/smt/proof/process.rs:12-23,53-59; src/smt/proof/inclusion.rs:5-33):
# fields in declaration order, hashes as WrappedHashOut hex strings, the role as its variant name
# ------------------------------------------------------------------------------------------------
PROCESS_ROLES = ("ProcessNoOp", "ProcessUpdate", "ProcessInsert", "ProcessDelete")


def smt_process_proofs_to_json(headers: np.ndarray, sib_pool: np.ndarray, sib_off: np.ndarray) -> List[str]:
    """One serde_json string per SparseMerkleProcessProof<GoldilocksHashOut, ..> of the batch layout."""
    import json

    hd = np.ascontiguousarray(headers, dtype=SMT_HDR_DTYPE)
    pool, off = _h(sib_pool).reshape(-1, 4), _h(sib_off)
    out = []
    for t in range(hd.shape[0]):
        h = hd[t]
        obj = {f: hash_out_to_hex(h[f]) for f in ("old_root", "old_key", "old_value", "new_root", "new_key", "new_value")}
        obj["siblings"] = [hash_out_to_hex(x) for x in pool[int(off[t]):int(off[t + 1])]]
        obj["is_old0"] = bool(h["is_old0"])
        obj["fnc"] = PROCESS_ROLES[int(h["fnc"])]
        out.append(json.dumps(obj, separators=(",", ":")))
    return out


def smt_process_proofs_from_json(texts: Sequence[str]):
    """The inverse: (headers, sib_pool, sib_off) in the layout gl_smt_verify_process_batch takes."""
    import json

    hd = np.zeros(len(texts), dtype=SMT_HDR_DTYPE)
    off = np.zeros(len(texts) + 1, dtype=np.uint64)
    sibs = []
    for t, text in enumerate(texts):
        obj = json.loads(text)
        for f in ("old_root", "old_key", "old_value", "new_root", "new_key", "new_value"):
            hd[f][t] = hash_out_from_hex(obj[f])
        hd["is_old0"][t] = 1 if obj["is_old0"] else 0
        if obj["fnc"] not in PROCESS_ROLES:
            raise ValueError(f"unknown variant `{obj['fnc']}`, expected one of {', '.join('`%s`' % r for r in PROCESS_ROLES)}")
        hd["fnc"][t] = PROCESS_ROLES.index(obj["fnc"])
        sibs += [hash_out_from_hex(x) for x in obj["siblings"]]
        off[t + 1] = len(sibs)
    pool = np.array(sibs, dtype=np.uint64).reshape(-1, 4) if sibs else np.zeros((0, 4), dtype=np.uint64)
    return hd, pool, off


def smt_inclusion_proofs_to_json(headers: np.ndarray, sib_pool: np.ndarray, sib_off: np.ndarray) -> List[str]:
    """One serde_json string per SparseMerkleInclusionProof<GoldilocksHashOut, ..> (what smt_find_batch returns)."""
    import json

    hd = np.ascontiguousarray(headers, dtype=SMT_INCLUSION_DTYPE)
    pool, off = _h(sib_pool).reshape(-1, 4), _h(sib_off)
    out = []
    for i in range(hd.shape[0]):
        h = hd[i]
        obj = {"root": hash_out_to_hex(h["root"]), "found": bool(h["found"]), "key": hash_out_to_hex(h["key"]),
               "value": hash_out_to_hex(h["value"]), "not_found_key": hash_out_to_hex(h["not_found_key"]),
               "not_found_value": hash_out_to_hex(h["not_found_value"]),
               "siblings": [hash_out_to_hex(x) for x in pool[int(off[i]):int(off[i + 1])]], "is_old0": bool(h["is_old0"])}
        out.append(json.dumps(obj, separators=(",", ":")))
    return out


def smt_inclusion_proofs_from_json(texts: Sequence[str]):
    import json

    hd = np.zeros(len(texts), dtype=SMT_INCLUSION_DTYPE)
    off = np.zeros(len(texts) + 1, dtype=np.uint64)
    sibs = []
    for i, text in enumerate(texts):
        obj = json.loads(text)
        for f in ("root", "key", "value", "not_found_key", "not_found_value"):
            hd[f][i] = hash_out_from_hex(obj[f])
        hd["found"][i] = 1 if obj["found"] else 0
        hd["is_old0"][i] = 1 if obj["is_old0"] else 0
        sibs += [hash_out_from_hex(x) for x in obj["siblings"]]
        off[i + 1] = len(sibs)
    pool = np.array(sibs, dtype=np.uint64).reshape(-1, 4) if sibs else np.zeros((0, 4), dtype=np.uint64)
    return hd, pool, off
