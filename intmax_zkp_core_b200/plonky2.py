"""Host-side mirror of the plonky2 API surface the commitment path sits behind.

Same names, argument meaning and error behaviour as plonky2 @ f99ed9c (the crate intmax-zkp-core pins at
/root/reference/Cargo.toml:12 and re-exports at /root/reference/src/lib.rs:12):

    PolynomialBatch::from_values / from_coeffs / get_lde_values        plonky2/src/fri/oracle.rs
    MerkleTree::new / prove / get, MerkleCap, MerkleProof              plonky2/src/hash/merkle_tree.rs
    verify_merkle_proof_to_cap                                         plonky2/src/hash/merkle_proofs.rs
    PoseidonHash::{hash_no_pad, hash_or_noop, hash_pad, two_to_one}    plonky2/src/hash/poseidon.rs, hashing.rs
    PoseidonPermutation::permute
    PolynomialValues::ifft, PolynomialCoeffs::{fft, lde, coset_fft}    field/src/polynomial/mod.rs

Everything computes on the GPU through the C ABI (include/b200zkp.h); numpy arrays of uint64 stand in for
Vec<F>.  The Rust toolchain is absent in this environment, so this Python layer (and host/plonky2_api.hpp
for C++) plays the role of the patched plonky2 crate; INTEGRATION.md shows the Rust binding itself.
Field elements are uint64; inputs may be non-canonical, outputs are canonical.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import B200ZkpError

P = 0xFFFFFFFF00000001
SALT_SIZE = 4
NUM_HASH_OUT_ELTS = 4
SPONGE_WIDTH = 12
SPONGE_RATE = 8


def _u64(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(np.asarray(a, dtype=np.uint64))
    if shape is not None:
        a = a.reshape(shape)
    return a


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def log2_strict(n: int) -> int:
    """plonky2_util::log2_strict: panics (ValueError here) unless n is a power of two."""
    if n <= 0 or n & (n - 1):
        raise ValueError(f"Not a power of two: {n}")
    return n.bit_length() - 1


def reverse_bits(x: int, bits: int) -> int:
    r = 0
    for _ in range(bits):
        r = (r << 1) | (x & 1)
        x >>= 1
    return r


class Context:
    """One device + stream + twiddle cache (b200zkp_ctx).  `stream` may be a raw cudaStream_t to share."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self._lib = _lib.lib()
        h = C.c_void_p()
        rc = self._lib.b200zkp_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != 0:
            raise B200ZkpError(rc, "b200zkp_ctx_create failed (is a CUDA device present? there is no CPU fallback)")
        self._h = h
        self.device = device

    def check(self, rc: int):
        if rc != 0:
            raise B200ZkpError(rc, self._lib.b200zkp_last_error(self._h).decode())

    def synchronize(self):
        self.check(self._lib.b200zkp_ctx_synchronize(self._h))

    STAGES = ("intt", "lde", "leaf_hash", "tree")

    def trim(self):
        """Synchronise and hand every cached device buffer back to the driver (b200zkp_ctx_trim)."""
        self.check(self._lib.b200zkp_ctx_trim(self._h))

    def set_pool_limit(self, nbytes: int):
        """Upper bound of the per-context cache of freed device buffers (default: 1/8 of the device memory)."""
        self.check(self._lib.b200zkp_ctx_set_pool_limit(self._h, int(nbytes)))

    def set_timing(self, enabled: bool):
        self.check(self._lib.b200zkp_ctx_set_timing(self._h, int(enabled)))

    def stage_ms(self) -> dict:
        """Synchronise and return {stage: (total ms, spans)} recorded since the last call."""
        ms = (C.c_double * 4)()
        cnt = (C.c_uint32 * 4)()
        self.check(self._lib.b200zkp_ctx_stage_ms(self._h, ms, cnt))
        return {s: (float(ms[i]), int(cnt[i])) for i, s in enumerate(self.STAGES)}

    @property
    def launch_count(self) -> int:
        return int(self._lib.b200zkp_ctx_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.b200zkp_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


# ------------------------------------------------------------------------------------------------ hashing
class HashOut:
    """plonky2 HashOut<F>: 4 field elements."""

    __slots__ = ("elements",)

    def __init__(self, elements):
        self.elements = _u64(elements, (4,))

    def to_bytes(self) -> bytes:
        """GenericHashOut::to_bytes: 4 canonical u64, little endian (HASH_SIZE = 32)."""
        return self.elements.astype("<u8").tobytes()

    def to_hex(self) -> str:
        """The reference's WrappedHashOut hex form: the 32 bytes reversed
        (/root/reference/src/sparse_merkle_tree/goldilocks_poseidon/hash/mod.rs:84-119)."""
        return "0x" + self.to_bytes()[::-1].hex()

    @staticmethod
    def from_hex(s: str) -> "HashOut":
        raw = bytes.fromhex(s[2:] if s.startswith("0x") else s)
        raw = raw.rjust(32, b"\0")[::-1]
        return HashOut(np.frombuffer(raw, dtype="<u8"))

    def __eq__(self, other):
        return isinstance(other, HashOut) and bool((self.elements == other.elements).all())

    def __repr__(self):
        return f"HashOut({[int(x) for x in self.elements]})"


class PoseidonPermutation:
    @staticmethod
    def permute(state, ctx: Optional[Context] = None) -> np.ndarray:
        """state: (12,) or (m, 12) -> same shape."""
        ctx = ctx or default_context()
        s = _u64(state)
        flat = s.reshape(-1, SPONGE_WIDTH)
        out = np.empty_like(flat)
        ctx.check(ctx._lib.b200zkp_poseidon_permute(ctx._h, _p(flat), flat.shape[0], _p(out)))
        return out.reshape(s.shape)


class PoseidonHash:
    """plonky2 `impl Hasher<F> for PoseidonHash` (HASH_SIZE = 32)."""

    HASH_SIZE = 32

    @staticmethod
    def hash_no_pad_batch(rows, ctx: Optional[Context] = None) -> np.ndarray:
        ctx = ctx or default_context()
        r = _u64(rows)
        assert r.ndim == 2
        out = np.empty((r.shape[0], 4), dtype=np.uint64)
        ctx.check(ctx._lib.b200zkp_hash_no_pad(ctx._h, _p(r), r.shape[0], r.shape[1], _p(out)))
        return out

    @staticmethod
    def hash_or_noop_batch(rows, ctx: Optional[Context] = None) -> np.ndarray:
        ctx = ctx or default_context()
        r = _u64(rows)
        assert r.ndim == 2
        out = np.empty((r.shape[0], 4), dtype=np.uint64)
        ctx.check(ctx._lib.b200zkp_hash_or_noop(ctx._h, _p(r), r.shape[0], r.shape[1], _p(out)))
        return out

    @staticmethod
    def hash_no_pad(inputs, ctx: Optional[Context] = None) -> HashOut:
        x = _u64(inputs).reshape(1, -1)
        return HashOut(PoseidonHash.hash_no_pad_batch(x, ctx)[0])

    @staticmethod
    def hash_or_noop(inputs, ctx: Optional[Context] = None) -> HashOut:
        x = _u64(inputs).reshape(1, -1)
        return HashOut(PoseidonHash.hash_or_noop_batch(x, ctx)[0])

    @staticmethod
    def hash_pad(inputs, ctx: Optional[Context] = None) -> HashOut:
        """hashing.rs hash_n_to_hash_with_pad: append 1, zero-fill to a multiple of SPONGE_WIDTH, last = 1
        (the rule /root/reference/src/sparse_merkle_tree/gadgets/common.rs:87-101 relies on)."""
        x = [int(v) for v in np.asarray(inputs, dtype=np.uint64).reshape(-1)]
        x.append(1)
        while (len(x) + 1) % SPONGE_WIDTH:
            x.append(0)
        x.append(1)
        return PoseidonHash.hash_no_pad(x, ctx)

    @staticmethod
    def two_to_one(left, right, ctx: Optional[Context] = None) -> HashOut:
        l = left.elements if isinstance(left, HashOut) else left
        r = right.elements if isinstance(right, HashOut) else right
        return HashOut(PoseidonHash.two_to_one_batch(_u64(l, (1, 4)), _u64(r, (1, 4)), ctx)[0])

    @staticmethod
    def two_to_one_batch(left, right, ctx: Optional[Context] = None) -> np.ndarray:
        ctx = ctx or default_context()
        l, r = _u64(left).reshape(-1, 4), _u64(right).reshape(-1, 4)
        assert l.shape == r.shape
        out = np.empty_like(l)
        ctx.check(ctx._lib.b200zkp_two_to_one(ctx._h, _p(l), _p(r), l.shape[0], _p(out)))
        return out


# ------------------------------------------------------------------------------------------------ Merkle tree
class MerkleCap:
    """plonky2 MerkleCap<F, H>(Vec<H::Hash>)."""

    def __init__(self, elements):
        self.elements = _u64(elements).reshape(-1, 4)

    def height(self) -> int:
        return log2_strict(self.elements.shape[0])

    def __len__(self):
        return self.elements.shape[0]

    def __getitem__(self, i) -> HashOut:
        return HashOut(self.elements[i])

    def flatten(self) -> np.ndarray:
        return self.elements.reshape(-1)

    def __eq__(self, other):
        return isinstance(other, MerkleCap) and self.elements.shape == other.elements.shape and bool(
            (self.elements == other.elements).all())


class MerkleProof:
    """plonky2 MerkleProof { siblings }: bottom-up, log2(N) - cap_height entries."""

    def __init__(self, siblings):
        self.siblings = _u64(siblings).reshape(-1, 4)

    def __len__(self):
        return self.siblings.shape[0]


class MerkleTree:
    """plonky2 MerkleTree<F, H> { leaves, digests, cap }; digests/leaves stay on the device until read."""

    def __init__(self):
        raise TypeError("use MerkleTree.new(leaves, cap_height)")

    @classmethod
    def new(cls, leaves, cap_height: int, ctx: Optional[Context] = None) -> "MerkleTree":
        ctx = ctx or default_context()
        lv = _u64(leaves)
        if lv.ndim != 2:
            raise ValueError("leaves must be a (N, leaf_len) array")
        n = lv.shape[0]
        lg = log2_strict(n)  # plonky2: log2_strict(leaves.len())
        if cap_height > lg:
            # plonky2 assert!: "cap_height={} should be at most log2(leaves.len())={}"
            raise ValueError(f"cap_height={cap_height} should be at most log2(leaves.len())={lg}")
        self = object.__new__(cls)
        self._ctx = ctx
        self.leaves = lv
        self.cap_height = cap_height
        h = C.c_void_p()
        ctx.check(ctx._lib.b200zkp_merkle_new(ctx._h, _p(lv), n, lv.shape[1], cap_height, C.byref(h)))
        self._h = h
        cap = np.empty((1 << cap_height, 4), dtype=np.uint64)
        ctx.check(ctx._lib.b200zkp_tree_cap(h, _p(cap)))
        self.cap = MerkleCap(cap)
        self._digests = None
        return self

    @property
    def digests(self) -> np.ndarray:
        if self._digests is None:
            n = self.leaves.shape[0]
            d = np.empty((2 * (n - (1 << self.cap_height)), 4), dtype=np.uint64)
            self._ctx.check(self._ctx._lib.b200zkp_tree_digests(self._h, _p(d) if d.size else None))
            self._digests = d
        return self._digests

    def get(self, i: int) -> np.ndarray:
        return self.leaves[i]

    def prove(self, leaf_index: int) -> MerkleProof:
        return self.prove_many([leaf_index])[0]

    def prove_many(self, indices: Sequence[int]):
        idx = _u64(indices)
        n_layers = log2_strict(self.leaves.shape[0]) - self.cap_height
        sib = np.empty((idx.size, n_layers, 4), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_tree_prove(self._h, _p(idx), idx.size, _p(sib) if sib.size else None))
        return [MerkleProof(sib[i]) for i in range(idx.size)]

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and getattr(self._ctx, "_h", None):
            self._ctx._lib.b200zkp_tree_free(h)
            self._h = None


def verify_merkle_proof_to_cap(leaf_data, leaf_index: int, merkle_cap: MerkleCap, proof: MerkleProof,
                               ctx: Optional[Context] = None) -> None:
    """merkle_proofs.rs: raises ValueError("Invalid Merkle proof.") on mismatch."""
    cur = PoseidonHash.hash_or_noop(leaf_data, ctx)
    index = leaf_index
    for sib in proof.siblings:
        if index & 1:
            cur = PoseidonHash.two_to_one(sib, cur, ctx)
        else:
            cur = PoseidonHash.two_to_one(cur, sib, ctx)
        index >>= 1
    if cur != merkle_cap[index]:
        raise ValueError("Invalid Merkle proof.")


# ------------------------------------------------------------------------------------------------ polynomials
class PolynomialValues:
    def __init__(self, values):
        self.values = _u64(values).reshape(-1)
        log2_strict(self.values.size)

    def ifft(self, ctx: Optional[Context] = None) -> "PolynomialCoeffs":
        return PolynomialCoeffs(ifft_batch(self.values.reshape(1, -1), ctx)[0])

    def coset_ifft(self, shift: int, ctx: Optional[Context] = None) -> "PolynomialCoeffs":
        """values on shift * <w_n> (natural order) -> coefficients (plonky2_field polynomial/mod.rs)"""
        return PolynomialCoeffs(coset_ifft_batch(self.values.reshape(1, -1), shift, ctx)[0])

    def __len__(self):
        return self.values.size


class PolynomialCoeffs:
    def __init__(self, coeffs):
        self.coeffs = _u64(coeffs).reshape(-1)
        log2_strict(self.coeffs.size)

    def fft(self, ctx: Optional[Context] = None) -> PolynomialValues:
        return PolynomialValues(fft_batch(self.coeffs.reshape(1, -1), ctx)[0])

    def lde(self, rate_bits: int) -> "PolynomialCoeffs":
        return PolynomialCoeffs(np.concatenate([self.coeffs, np.zeros(self.coeffs.size * ((1 << rate_bits) - 1), np.uint64)]))

    def coset_lde_values(self, rate_bits: int, ctx: Optional[Context] = None) -> PolynomialValues:
        """lde(rate_bits).coset_fft(F::coset_shift()): values at 7 * w_N^i, natural order (A4)."""
        return PolynomialValues(coset_lde_batch(self.coeffs.reshape(1, -1), rate_bits, ctx)[0])

    def __len__(self):
        return self.coeffs.size


def fft_batch(coeffs, ctx: Optional[Context] = None) -> np.ndarray:
    ctx = ctx or default_context()
    x = _u64(coeffs).copy()
    k, n = x.shape
    ctx.check(ctx._lib.b200zkp_ntt(ctx._h, _p(x), log2_strict(n), k))
    return x


def ifft_batch(values, ctx: Optional[Context] = None) -> np.ndarray:
    ctx = ctx or default_context()
    x = _u64(values).copy()
    k, n = x.shape
    ctx.check(ctx._lib.b200zkp_intt(ctx._h, _p(x), log2_strict(n), k))
    return x


def coset_ifft_batch(values, shift: int, ctx: Optional[Context] = None) -> np.ndarray:
    """PolynomialValues::coset_ifft(shift) over the rows of a (k, n) array"""
    ctx = ctx or default_context()
    x = _u64(values).copy()
    if x.ndim != 2:
        raise ValueError("expected a (k, n) array")
    ctx.check(ctx._lib.b200zkp_coset_intt(ctx._h, _p(x), log2_strict(x.shape[1]), x.shape[0], int(shift) % 2**64))
    return x


def coset_lde_batch(coeffs, rate_bits: int, ctx: Optional[Context] = None) -> np.ndarray:
    ctx = ctx or default_context()
    x = _u64(coeffs)
    k, n = x.shape
    out = np.empty((k, n << rate_bits), dtype=np.uint64)
    ctx.check(ctx._lib.b200zkp_coset_lde(ctx._h, _p(x), log2_strict(n), k, rate_bits, _p(out)))
    return out


class _BatchMerkleTree:
    """The `merkle_tree` field of a PolynomialBatch: cap on the host, leaves/digests fetched on demand."""

    def __init__(self, batch: "PolynomialBatch"):
        self._b = batch
        self._digests = None
        self._leaves = None

    @property
    def cap(self) -> MerkleCap:
        return self._b._cap

    @property
    def leaves(self) -> np.ndarray:
        if self._leaves is None:
            b = self._b
            N = 1 << (b.degree_log + b.rate_bits)
            out = np.empty((N, b.num_polys + b.salt_size), dtype=np.uint64)
            b._ctx.check(b._ctx._lib.b200zkp_batch_leaves(b._h, _p(out)))
            self._leaves = out
        return self._leaves

    @property
    def digests(self) -> np.ndarray:
        if self._digests is None:
            b = self._b
            N = 1 << (b.degree_log + b.rate_bits)
            d = np.empty((2 * (N - (1 << b.cap_height)), 4), dtype=np.uint64)
            b._ctx.check(b._ctx._lib.b200zkp_batch_digests(b._h, _p(d) if d.size else None))
            self._digests = d
        return self._digests

    def get(self, i: int) -> np.ndarray:
        return self._b.rows([i])[0][0]

    def prove(self, leaf_index: int) -> MerkleProof:
        return MerkleProof(self._b.rows([leaf_index], want_rows=False)[1][0])


class PolynomialBatch:
    """plonky2 PolynomialBatch<F, C, D> { polynomials, merkle_tree, degree_log, rate_bits, blinding }."""

    def __init__(self):
        raise TypeError("use PolynomialBatch.from_values / from_coeffs")

    @classmethod
    def _commit(cls, data, is_coeffs: bool, rate_bits: int, blinding: bool, cap_height: int,
                salt, ctx: Optional[Context], copy_back: bool = False):
        ctx = ctx or default_context()
        x = _u64(data)
        if x.ndim != 2 or x.shape[0] == 0:
            raise ValueError("expected a non-empty (k, n) array: one row per polynomial")
        k, n = x.shape
        n_log = log2_strict(n)
        N = n << rate_bits
        if cap_height > n_log + rate_bits:
            raise ValueError(f"cap_height={cap_height} should be at most log2(leaves.len())={n_log + rate_bits}")
        s = None
        if blinding:
            if salt is None:
                # plonky2 draws F::rand_vec(N) per salt column from the thread RNG; any uniform draw is a
                # valid commitment, parity tests pass `salt` explicitly.
                rng = np.random.default_rng()
                salt = rng.integers(0, P, size=(SALT_SIZE, N), dtype=np.uint64)
            s = _u64(salt)
            if s.shape != (SALT_SIZE, N):
                raise ValueError(f"salt must have shape ({SALT_SIZE}, {N})")
        self = object.__new__(cls)
        self._ctx = ctx
        self.degree_log = n_log
        self.rate_bits = rate_bits
        self.blinding = bool(blinding)
        self.cap_height = cap_height
        self.num_polys = k
        self.salt_size = SALT_SIZE if blinding else 0
        h = C.c_void_p()
        cap = np.empty((1 << cap_height, 4), dtype=np.uint64)
        if copy_back:
            # strict drop-in: every plonky2 struct field is materialised on the host in the same call, the D2H of
            # coefficients and leaves overlapping the leaf hash (b200zkp_commit_copy_back)
            polys = np.empty((k, n), dtype=np.uint64)
            leaves = np.empty((N, k + self.salt_size), dtype=np.uint64)
            digests = np.empty((2 * (N - (1 << cap_height)), 4), dtype=np.uint64)
            ctx.check(ctx._lib.b200zkp_commit_copy_back(ctx._h, _p(x), int(is_coeffs), n_log, k, rate_bits, cap_height, _p(s),
                                                        _p(polys), _p(leaves), _p(digests) if digests.size else None, _p(cap),
                                                        C.byref(h)))
        else:
            fn = ctx._lib.b200zkp_commit_from_coeffs if is_coeffs else ctx._lib.b200zkp_commit_from_values
            ctx.check(fn(ctx._h, _p(x), n_log, k, rate_bits, cap_height, _p(s), C.byref(h)))
            ctx.check(ctx._lib.b200zkp_batch_cap(h, _p(cap)))
        self._h = h
        self._cap = MerkleCap(cap)
        self.merkle_tree = _BatchMerkleTree(self)
        self._polys = None
        if copy_back:
            self._polys = polys
            self.merkle_tree._leaves = leaves
            self.merkle_tree._digests = digests
        return self

    @classmethod
    def from_values(cls, values, rate_bits: int, blinding: bool, cap_height: int, timing=None,
                    fft_root_table=None, salt=None, ctx: Optional[Context] = None, copy_back: bool = False) -> "PolynomialBatch":
        """values: (k, n) — k PolynomialValues of n points each.  `timing` / `fft_root_table` are accepted
        for signature parity (the ctx owns the root tables).  copy_back=True fills polynomials / leaves / digests on
        the host in the same call (strict drop-in); otherwise they stay in HBM until an accessor asks."""
        return cls._commit(values, False, rate_bits, blinding, cap_height, salt, ctx, copy_back)

    @classmethod
    def from_coeffs(cls, polynomials, rate_bits: int, blinding: bool, cap_height: int, timing=None,
                    fft_root_table=None, salt=None, ctx: Optional[Context] = None, copy_back: bool = False) -> "PolynomialBatch":
        return cls._commit(polynomials, True, rate_bits, blinding, cap_height, salt, ctx, copy_back)

    @classmethod
    def from_device(cls, tensor, rate_bits: int, blinding: bool, cap_height: int, is_coeffs: bool = False,
                    ctx: Optional[Context] = None, salt=None) -> "PolynomialBatch":
        """from_values (from_coeffs with is_coeffs) of a (k, n) CUDA tensor of 64-bit words already in HBM
        (b200zkp_batch_from_device): asynchronous on the ctx stream, nothing crosses PCIe.  The batch keeps `tensor` (and
        `salt`, (4, N) on the device when blinding) alive for its own lifetime, so the commit never reads freed memory.
        `coeffs` and `lde` are torch views of the handle's coefficients and leaf-order LDE."""
        from .device import _dev_view
        ctx = ctx or default_context()
        if tensor.dim() != 2 or not tensor.is_cuda or not tensor.is_contiguous() or tensor.element_size() != 8 or tensor.shape[0] == 0:
            raise ValueError("expected a non-empty contiguous (k, n) CUDA tensor of 64-bit words")
        k, n = tensor.shape
        n_log = log2_strict(n)
        if cap_height > n_log + rate_bits:
            raise ValueError(f"cap_height={cap_height} should be at most log2(leaves.len())={n_log + rate_bits}")
        if blinding:
            if salt is None or tuple(salt.shape) != (SALT_SIZE, n << rate_bits) or not salt.is_cuda or not salt.is_contiguous():
                raise ValueError(f"blinding needs a contiguous ({SALT_SIZE}, {n << rate_bits}) CUDA salt tensor")
        else:
            salt = None
        h = C.c_void_p()
        ctx.check(ctx._lib.b200zkp_batch_from_device(ctx._h, C.c_void_p(tensor.data_ptr()), int(is_coeffs), n_log, k, rate_bits,
                                                     cap_height, C.c_void_p(salt.data_ptr()) if salt is not None else None,
                                                     C.byref(h)))
        self = object.__new__(cls)
        self._ctx, self._h, self._keep = ctx, h, (tensor, salt)
        self.degree_log, self.rate_bits, self.blinding, self.cap_height = n_log, rate_bits, bool(blinding), cap_height
        self.num_polys, self.salt_size = k, SALT_SIZE if blinding else 0
        self._polys = None
        coeffs, lde, _, cap = self.device_ptrs()
        self.coeffs = _dev_view(coeffs, (k, n), ctx.device)
        self.lde = _dev_view(lde, (k + self.salt_size, n << rate_bits), ctx.device)
        self._cap_dev = _dev_view(cap, (1 << cap_height, 4), ctx.device)
        self._cap_host = None
        self.merkle_tree = _BatchMerkleTree(self)
        return self

    @property
    def _cap(self) -> MerkleCap:
        """the Merkle cap, read back on first use (for a device commit that synchronises the ctx stream)"""
        if self._cap_host is None:
            cap = np.empty((1 << self.cap_height, 4), dtype=np.uint64)
            self._ctx.check(self._ctx._lib.b200zkp_batch_cap(self._h, _p(cap)))
            self._cap_host = MerkleCap(cap)
        return self._cap_host

    @_cap.setter
    def _cap(self, cap: MerkleCap):
        self._cap_host = cap

    @property
    def polynomials(self) -> np.ndarray:
        """(k, n) coefficient vectors."""
        if self._polys is None:
            out = np.empty((self.num_polys, 1 << self.degree_log), dtype=np.uint64)
            self._ctx.check(self._ctx._lib.b200zkp_batch_coeffs(self._h, _p(out)))
            self._polys = out
        return self._polys

    def get_lde_values(self, index: int, step: int = 1) -> np.ndarray:
        """&leaves[reverse_bits(index * step, degree_log + rate_bits)][..len - salt]"""
        out = np.empty(self.num_polys, dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_batch_lde_values(self._h, index, step, _p(out)))
        return out

    def rows(self, indices: Sequence[int], want_rows: bool = True, want_proofs: bool = True):
        """Leaf rows and Merkle proofs for a list of leaf indices (what FRI query rounds open)."""
        idx = _u64(indices)
        n_layers = self.degree_log + self.rate_bits - self.cap_height
        rows = np.empty((idx.size, self.num_polys + self.salt_size), dtype=np.uint64) if want_rows else None
        sib = np.empty((idx.size, n_layers, 4), dtype=np.uint64) if want_proofs else None
        self._ctx.check(self._ctx._lib.b200zkp_batch_rows(self._h, _p(idx), idx.size, _p(rows),
                                                          _p(sib) if (sib is not None and sib.size) else None))
        return rows, sib

    def eval_ext2(self, zeta) -> np.ndarray:
        """OpeningSet::new's `p.to_extension().eval(zeta)` for every polynomial of the batch: zeta = (re, im) in
        F_p[X]/(X^2 - 7); returns (k, 2).  Evaluated on the device from the resident coefficients."""
        z = _u64(zeta, (2,))
        out = np.empty((self.num_polys, 2), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_batch_eval_ext2(self._h, _p(z), _p(out)))
        return out

    def device_ptrs(self):
        ptrs = [C.c_void_p() for _ in range(4)]
        self._ctx.check(self._ctx._lib.b200zkp_batch_device_ptrs(self._h, *[C.byref(p) for p in ptrs]))
        return tuple(p.value for p in ptrs)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and getattr(self._ctx, "_h", None):
            self._ctx._lib.b200zkp_batch_free(h)
            self._h = None
