"""Host mirror of the prover steps around the commitments (SURVEY.md section 8f, row N1a): the permutation argument.

plonky2 @ f99ed9c, plonky2/src/plonk/prover.rs:
    all_wires_permutation_partial_products(witness, betas, gammas, prover_data, common_data)
    wires_permutation_partial_products_and_zs(witness, beta, gamma, prover_data, common_data)
reached from the reference through every prove() (/root/reference/src/transaction/circuits/mod.rs:453,
src/zkdsa/circuits/mod.rs:326, src/rollup/circuits/mod.rs:1247).  prove() then moves every Z to the front of the batch
(`zs_partial_products = [plonk_z_vecs, partial_products.concat()].concat()`) and commits it with
PolynomialBatch::from_values; `zs_partial_products` below returns that batch directly, and on the device path it feeds
the commitment without leaving HBM.  Same names and argument meaning as plonky2; no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import secrets
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .fri import batch_openings
from .plonky2 import SALT_SIZE, Context, MerkleCap, P, PolynomialBatch, _p, _u64, coset_ifft_batch, default_context, log2_strict

MULTIPLICATIVE_GROUP_GENERATOR = 7


def get_unique_coset_shifts(num_shifts: int) -> np.ndarray:
    """CommonCircuitData::k_is: k_j = g^j (plonky2/src/plonk/permutation_argument.rs / plonk_common.rs)"""
    out, x = [], 1
    for _ in range(num_shifts):
        out.append(x)
        x = x * MULTIPLICATIVE_GROUP_GENERATOR % P
    return np.array(out, dtype=np.uint64)


def num_partial_products(num_routed_wires: int, quotient_degree_factor: int) -> int:
    """CommonCircuitData::num_partial_products = ceil(num_routed_wires / quotient_degree_factor) - 1"""
    return -(-num_routed_wires // quotient_degree_factor) - 1


def zs_partial_products(wires, sigmas, k_is, betas: Sequence[int], gammas: Sequence[int], quotient_degree_factor: int,
                        ctx: Optional[Context] = None) -> np.ndarray:
    """The `Z + partial products` batch of prove(), ready for PolynomialBatch.from_values.

    wires, sigmas: (num_routed_wires, n) — the routed wire columns of the witness and the sigma polynomials' values
    on the subgroup; k_is: (num_routed_wires,); betas, gammas: one per challenge.
    Returns (num_challenges * (1 + num_partial_products), n): row c = Z of challenge c, then the partial products of
    challenge 0, of challenge 1, ..."""
    ctx = ctx or default_context()
    w, s = _u64(wires), _u64(sigmas)
    if w.ndim != 2 or w.shape != s.shape or w.shape[0] == 0:
        raise ValueError("wires and sigmas must be equal-shaped (num_routed_wires, n) arrays")
    R, n = w.shape
    n_log = log2_strict(n)
    k = _u64(k_is)
    b, g = _u64(np.asarray(betas, dtype=np.uint64)), _u64(np.asarray(gammas, dtype=np.uint64))
    if k.shape != (R,) or b.shape != g.shape or b.ndim != 1 or b.size == 0:
        raise ValueError("k_is must have one entry per routed wire, betas / gammas one per challenge")
    chunks = -(-R // quotient_degree_factor)
    out = np.empty((b.size * chunks, n), dtype=np.uint64)
    ctx.check(ctx._lib.b200zkp_partial_products_and_zs(ctx._h, _p(w), _p(s), n_log, R, quotient_degree_factor, _p(k), _p(b), _p(g),
                                                       b.size, _p(out)))
    return out


def wires_permutation_partial_products_and_zs(wires, sigmas, k_is, beta: int, gamma: int, quotient_degree_factor: int,
                                              ctx: Optional[Context] = None) -> np.ndarray:
    """plonky2's per-challenge form: rows [pp_0 .. pp_{num_prods-1}, Z] (Z last, as prover.rs returns it)."""
    cols = zs_partial_products(wires, sigmas, k_is, [beta], [gamma], quotient_degree_factor, ctx)
    return np.concatenate([cols[1:], cols[:1]], axis=0)


def all_wires_permutation_partial_products(wires, sigmas, k_is, betas, gammas, quotient_degree_factor: int,
                                           ctx: Optional[Context] = None):
    """one wires_permutation_partial_products_and_zs result per challenge (one launch sequence for all of them)"""
    cols = zs_partial_products(wires, sigmas, k_is, betas, gammas, quotient_degree_factor, ctx)
    Cn = len(betas)
    num_prods = cols.shape[0] // Cn - 1
    return [np.concatenate([cols[Cn + c * num_prods:Cn + (c + 1) * num_prods], cols[c:c + 1]], axis=0) for c in range(Cn)]


def zs_partial_products_device(ctx: Context, wires, sigmas, k_is, betas, gammas, quotient_degree_factor: int, out=None):
    """Device-resident form on torch int64 tensors (uint64 bit patterns): wires / sigmas (num_routed, n) CUDA tensors
    (rows may be a view of a wider witness matrix as long as each row is contiguous); returns the (C * chunks, n) batch
    in HBM, ready for device.commit_device."""
    import torch
    R, n = wires.shape
    n_log = log2_strict(n)
    assert wires.is_cuda and sigmas.is_cuda and wires.stride(1) == 1 and sigmas.stride(1) == 1 and sigmas.shape == wires.shape
    k = _u64(k_is)
    b, g = _u64(np.asarray(betas, dtype=np.uint64)), _u64(np.asarray(gammas, dtype=np.uint64))
    chunks = -(-R // quotient_degree_factor)
    if out is None:
        out = torch.empty((b.size * chunks, n), dtype=torch.int64, device=wires.device)
    ctx.check(ctx._lib.b200zkp_dev_partial_products_and_zs(ctx._h, C.c_void_p(wires.data_ptr()), wires.stride(0),
                                                           C.c_void_p(sigmas.data_ptr()), sigmas.stride(0), n_log, R,
                                                           quotient_degree_factor, _p(k), _p(b), _p(g), b.size,
                                                           C.c_void_p(out.data_ptr()), out.stride(0)))
    return out


class QuotientError(ValueError):
    """plonky2's `trim_to_len` panic: the vanishing polynomial is not divisible by Z_H (unsatisfied witness)."""


def quotient_poly_chunks(quotient_values, degree_bits: int, quotient_degree_factor: Optional[int] = None,
                         ctx: Optional[Context] = None) -> np.ndarray:
    """Tail of plonky2's compute_quotient_polys + the chunking in prove() (row N1c):

        quotient_values.map(|v| v.coset_ifft(F::coset_shift()))            // one polynomial per challenge
        quotient_poly.trim_to_len(quotient_degree); quotient_poly.chunks(degree)

    quotient_values: (num_challenges, n * 2^quotient_degree_bits) values on the coset 7 <w>, natural order.
    quotient_degree_factor (CommonCircuitData; chosen in min..=max, not necessarily a power of two; default: every chunk):
    coefficients from quotient_degree_factor * n on must vanish — plonky2 panics there, this raises QuotientError — and only
    quotient_degree_factor chunks per challenge are committed.
    Returns (num_challenges * quotient_degree_factor, n) coefficient chunks, the input of PolynomialBatch.from_coeffs."""
    q = _u64(quotient_values)
    if q.ndim != 2:
        raise ValueError("expected (num_challenges, n << quotient_degree_bits)")
    n = 1 << degree_bits
    if q.shape[1] % n or q.shape[1] < n:
        raise ValueError("quotient length must be a multiple of the degree")
    coeffs = coset_ifft_batch(q, MULTIPLICATIVE_GROUP_GENERATOR, ctx)
    total = q.shape[1] // n
    qdf = total if quotient_degree_factor is None else int(quotient_degree_factor)
    if not 0 < qdf <= total:
        raise ValueError("quotient_degree_factor out of range")
    if coeffs[:, qdf * n:].any():
        raise QuotientError("Quotient has failed: coefficients beyond quotient_degree_factor * n are not zero")
    return np.ascontiguousarray(coeffs[:, :qdf * n]).reshape(q.shape[0] * qdf, n)


def commit_quotient(quotient_values, degree_bits: int, rate_bits: int, blinding: bool, cap_height: int, salt=None,
                    ctx: Optional[Context] = None, quotient_degree_factor: Optional[int] = None) -> PolynomialBatch:
    """quotient_polys_commitment of prove(): PolynomialBatch::from_coeffs(all_quotient_poly_chunks, ...)"""
    return PolynomialBatch.from_coeffs(quotient_poly_chunks(quotient_values, degree_bits, quotient_degree_factor, ctx), rate_bits,
                                       blinding, cap_height, salt=salt, ctx=ctx)


def quotient_chunks_device(ctx: Context, quotient_values, degree_bits: int, quotient_degree_factor: Optional[int] = None):
    """device-resident form of quotient_poly_chunks: (C, n << q) CUDA tensor of quotient values -> the (C * quotient_degree_factor,
    n) coefficient chunks (default 2^q per challenge) in HBM; only the divisibility check (quotient_degree_factor < 2^q) reads
    one flag back"""
    import torch
    Cn, total = quotient_values.shape
    n = 1 << degree_bits
    assert quotient_values.is_cuda and quotient_values.is_contiguous() and total % n == 0
    coeffs = torch.empty_like(quotient_values)
    scratch = torch.empty_like(quotient_values)
    ctx.check(ctx._lib.b200zkp_dev_coset_intt(ctx._h, C.c_void_p(quotient_values.data_ptr()), total, C.c_void_p(coeffs.data_ptr()), total,
                                              C.c_void_p(scratch.data_ptr()), log2_strict(total), Cn, MULTIPLICATIVE_GROUP_GENERATOR))
    qdf = total // n if quotient_degree_factor is None else int(quotient_degree_factor)
    if not 0 < qdf <= total // n:
        raise ValueError("quotient_degree_factor out of range")
    if qdf < total // n:
        ctx.synchronize()       # (the ctx stream may not be torch's current stream)
        if bool(coeffs[:, qdf * n:].any()):
            raise QuotientError("Quotient has failed: coefficients beyond quotient_degree_factor * n are not zero")
        coeffs = coeffs[:, :qdf * n].contiguous()
        torch.cuda.current_stream(coeffs.device).synchronize()
    return coeffs.view(Cn * qdf, n)


def commit_quotient_device(ctx: Context, quotient_values, degree_bits: int, rate_bits: int, cap_height: int,
                           quotient_degree_factor: Optional[int] = None):
    """device-resident form: (C, n << q) CUDA tensor of quotient values -> DeviceCommitment of the C * quotient_degree_factor
    chunks (default 2^q); the coefficients never leave HBM (the divisibility check reads one flag back)"""
    from .device import commit_device
    chunks = quotient_chunks_device(ctx, quotient_values, degree_bits, quotient_degree_factor)
    return commit_device(ctx, chunks, rate_bits, cap_height, is_coeffs=True)


# ------------------------------------------------------------------------------------------------ row N1b: compute_quotient_polys
GATE_NOOP, GATE_CONSTANT, GATE_PUBLIC_INPUT, GATE_ARITHMETIC, GATE_POSEIDON = range(5)
(GATE_ARITHMETIC_EXTENSION, GATE_MUL_EXTENSION, GATE_BASE_SUM, GATE_REDUCING, GATE_REDUCING_EXTENSION, GATE_RANDOM_ACCESS,
 GATE_EXPONENTIATION, GATE_POSEIDON_MDS) = range(5, 13)
GATE_INTERPOLATION_HIGH_DEGREE, GATE_INTERPOLATION_LOW_DEGREE = 14, 15         # (13 is not assigned)
MAX_GATES = 16


class _VanishingDesc(C.Structure):
    _fields_ = [("degree_bits", C.c_uint32), ("quotient_degree_bits", C.c_uint32), ("quotient_degree_factor", C.c_uint32),
                ("num_routed_wires", C.c_uint32), ("num_challenges", C.c_uint32), ("num_selectors", C.c_uint32),
                ("n_gates", C.c_uint32),
                ("gate_kind", C.c_uint32 * MAX_GATES), ("gate_selector_index", C.c_uint32 * MAX_GATES),
                ("gate_group_begin", C.c_uint32 * MAX_GATES), ("gate_group_end", C.c_uint32 * MAX_GATES),
                ("gate_params", (C.c_uint32 * 3) * MAX_GATES),
                ("k_is", C.c_void_p), ("betas", C.c_void_p), ("gammas", C.c_void_p), ("alphas", C.c_void_p),
                ("public_inputs_hash", C.c_uint64 * 4)]


class CommonCircuitData:
    """What compute_quotient_polys needs of plonky2's CommonCircuitData: degree_bits, the gate list in CircuitBuilder's order with
    the selector polynomial and selector group of every gate (SelectorsInfo), quotient_degree_factor, k_is.
    gates: [(kind, selector_index, (group_begin, group_end)[, params]), ...]; params: the gate's own parameters
    (BaseSum (B, num_limbs), Reducing / ReducingExtension (num_coeffs,), RandomAccess (bits, num_copies, num_extra_constants),
    Exponentiation (num_power_bits,), HighDegreeInterpolation (subgroup_bits,) with subgroup_bits 1..5,
    LowDegreeInterpolation (subgroup_bits,) with subgroup_bits 1..4).  The u32 and comparison gates are refused
    (B200ZkpError with code -4); the interpolation layouts are restated from memory as for the other gates (include/b200zkp.h)"""

    def __init__(self, degree_bits: int, gates, num_selectors: int, quotient_degree_factor: int = 8, num_routed_wires: int = 80,
                 k_is=None):
        self.degree_bits, self.gates, self.num_selectors = degree_bits, list(gates), num_selectors
        self.quotient_degree_factor, self.num_routed_wires = quotient_degree_factor, num_routed_wires
        self.k_is = _u64(k_is) if k_is is not None else get_unique_coset_shifts(num_routed_wires)
        if len(self.gates) > MAX_GATES:
            raise ValueError("too many gate types")

    @property
    def quotient_degree_bits(self) -> int:
        return max(self.quotient_degree_factor - 1, 0).bit_length()        # log2_ceil


def compute_quotient_values_device(ctx: Context, common: CommonCircuitData, constants_sigmas_lde, wires_lde, zs_partial_products_lde,
                                   betas, gammas, alphas, public_inputs_hash, out=None):
    """compute_quotient_polys up to its coset_ifft, on the three LDEs where the commitments left them: (columns, N) CUDA tensors
    in leaf order (DeviceCommitment.lde).  Returns the (num_challenges, n << quotient_degree_bits) quotient values in natural order
    on the coset 7 <w> — the input of commit_quotient_device."""
    import torch
    q_bits = common.quotient_degree_bits
    Q = 1 << (common.degree_bits + q_bits)
    b, g, a = (_u64(np.asarray(v, dtype=np.uint64)) for v in (betas, gammas, alphas))
    if not (b.shape == g.shape == a.shape) or b.ndim != 1:
        raise ValueError("one beta, gamma and alpha per challenge")
    for t in (constants_sigmas_lde, wires_lde, zs_partial_products_lde):
        if not t.is_cuda or t.stride(1) != 1 or t.shape[1] < Q:
            raise ValueError("LDEs must be CUDA tensors of at least n << quotient_degree_bits leaves per column")
    chunks = -(-common.num_routed_wires // common.quotient_degree_factor)
    if constants_sigmas_lde.shape[0] != common.num_selectors + 2 + common.num_routed_wires or wires_lde.shape[0] < 135 \
            or zs_partial_products_lde.shape[0] != b.size * chunks:
        raise ValueError("batch widths do not match the circuit description")
    d = _VanishingDesc()
    d.degree_bits, d.quotient_degree_bits, d.quotient_degree_factor = common.degree_bits, q_bits, common.quotient_degree_factor
    d.num_routed_wires, d.num_challenges, d.num_selectors, d.n_gates = common.num_routed_wires, b.size, common.num_selectors, len(common.gates)
    for i, gate in enumerate(common.gates):
        kind, sel, grp = gate[:3]
        d.gate_kind[i], d.gate_selector_index[i], d.gate_group_begin[i], d.gate_group_end[i] = kind, sel, grp[0], grp[1]
        for j, v in enumerate(gate[3] if len(gate) > 3 else ()):
            d.gate_params[i][j] = int(v)
    k = _u64(common.k_is)
    d.k_is, d.betas, d.gammas, d.alphas = k.ctypes.data, b.ctypes.data, g.ctypes.data, a.ctypes.data
    for i, v in enumerate(public_inputs_hash):
        d.public_inputs_hash[i] = int(v)
    if out is None:
        out = torch.empty((b.size, Q), dtype=torch.int64, device=wires_lde.device)
    ctx.check(ctx._lib.b200zkp_dev_quotient_values(ctx._h, C.byref(d), C.c_void_p(constants_sigmas_lde.data_ptr()), constants_sigmas_lde.stride(0),
                                                   C.c_void_p(wires_lde.data_ptr()), wires_lde.stride(0),
                                                   C.c_void_p(zs_partial_products_lde.data_ptr()), zs_partial_products_lde.stride(0),
                                                   C.c_void_p(out.data_ptr()), out.stride(0)))
    return out


# ------------------------------------------------------------------------------------------------ salts
def random_field_device(ctx: Context, key: bytes, nonce: bytes, count: int, first: int = 0, out=None):
    """F::rand_vec on the device (b200zkp_dev_random_field): elements [first, first + count) of the ChaCha20 stream (key, nonce)
    as a (count,) int64 CUDA tensor of canonical field elements, written asynchronously on the ctx stream.  key: 32 bytes, secret;
    nonce: 12 bytes.  out: a contiguous int64 CUDA tensor of `count` elements to fill instead of a new one."""
    import torch
    key, nonce = bytes(key), bytes(nonce)
    if len(key) != 32 or len(nonce) != 12:
        raise ValueError("the key must be 32 bytes and the nonce 12 bytes")
    if out is None:
        out = torch.empty(int(count), dtype=torch.int64, device=f"cuda:{ctx.device}")
    elif not out.is_cuda or out.dtype != torch.int64 or not out.is_contiguous() or out.numel() != count:
        raise ValueError("out must be a contiguous int64 CUDA tensor of `count` elements")
    ctx.check(ctx._lib.b200zkp_dev_random_field(ctx._h, key, nonce, int(first), int(count),
                                                C.c_void_p(out.data_ptr()) if count else None))
    return out


# PlonkOracle indices: the salt of oracle i is drawn with the nonce le32(i) || 0^8
PLONK_ORACLE_WIRES, PLONK_ORACLE_ZS_PARTIAL_PRODUCTS, PLONK_ORACLE_QUOTIENT = 1, 2, 3


def oracle_nonce(oracle_index: int) -> bytes:
    return int(oracle_index).to_bytes(4, "little") + bytes(8)


def salt_device(ctx: Context, key: bytes, oracle_index: int, lde_size: int):
    """the (SALT_SIZE, N) salt of one blinded commitment: elements [0, SALT_SIZE * N) of the stream (key, oracle_nonce(oracle_index)),
    element c*N + i = salt column c at natural LDE row i (the layout PolynomialBatch.from_device takes)"""
    return random_field_device(ctx, key, oracle_nonce(oracle_index), SALT_SIZE * lde_size).view(SALT_SIZE, lde_size)


# ------------------------------------------------------------------------------------------------ the whole proof
class CircuitData:
    """What prove() needs of plonky2's CircuitData (prover_only + common): the CommonCircuitData above, the constants + sigmas
    PolynomialBatch (committed from HBM), the sigma values on H as a CUDA tensor, circuit_digest, FriParams, num_challenges,
    and CircuitConfig::zero_knowledge (fri_params.hiding follows it)."""

    def __init__(self, common: CommonCircuitData, constants_sigmas_commitment: PolynomialBatch, sigmas, circuit_digest,
                 fri_params, num_challenges: int, zero_knowledge: bool = False):
        self.common, self.constants_sigmas_commitment, self.sigmas = common, constants_sigmas_commitment, sigmas
        self.circuit_digest, self.fri_params, self.num_challenges = circuit_digest, fri_params, num_challenges
        self.zero_knowledge = bool(zero_knowledge)

    @property
    def num_constants(self) -> int:
        return self.common.num_selectors + 2


def circuit_data(ctx: Context, common: CommonCircuitData, constants_sigmas_values, fri_config, num_challenges: int = 2,
                 zero_knowledge: bool = False) -> CircuitData:
    """The commitment CircuitBuilder::build makes: constants_sigmas_values is the (num_constants + num_routed_wires, n) CUDA tensor
    of selector + gate-constant columns followed by the sigma columns, values on H.  circuit_digest =
    hash_no_pad(constants_sigmas_cap.flatten()) (restated from memory of plonky2 @ f99ed9c, unpinned like the rest).
    zero_knowledge: prove() salts the wires, Z + partial products and quotient commitments and FriParams.hiding is set; the
    blinding rows are part of the circuit the caller describes (CircuitBuilder::blind_and_pad).  Constants + sigmas are never
    salted."""
    from .plonky2 import PoseidonHash
    if constants_sigmas_values.shape != (common.num_selectors + 2 + common.num_routed_wires, 1 << common.degree_bits):
        raise ValueError("constants_sigmas_values must hold num_selectors + 2 + num_routed_wires columns of 2^degree_bits values")
    cfg = fri_config
    batch = PolynomialBatch.from_device(constants_sigmas_values, cfg.rate_bits, False, cfg.cap_height, ctx=ctx)
    digest = PoseidonHash.hash_no_pad(batch._cap.flatten(), ctx)
    return CircuitData(common, batch, constants_sigmas_values[common.num_selectors + 2:], digest,
                       cfg.fri_params(common.degree_bits, hiding=bool(zero_knowledge)), num_challenges, zero_knowledge)


@dataclass
class OpeningSet:
    """plonk/proof.rs OpeningSet: extension values (re, im) at zeta, plonk_zs_next at g zeta"""
    constants: List[Tuple[int, int]]
    plonk_sigmas: List[Tuple[int, int]]
    wires: List[Tuple[int, int]]
    plonk_zs: List[Tuple[int, int]]
    plonk_zs_next: List[Tuple[int, int]]
    partial_products: List[Tuple[int, int]]
    quotient_polys: List[Tuple[int, int]]

    def to_fri_openings(self) -> List[List[Tuple[int, int]]]:
        """the values batch by batch, in the order the challenger observes them"""
        return [self.constants + self.plonk_sigmas + self.wires + self.plonk_zs + self.partial_products + self.quotient_polys,
                self.plonk_zs_next]


@dataclass
class Proof:
    wires_cap: MerkleCap
    plonk_zs_partial_products_cap: MerkleCap
    quotient_polys_cap: MerkleCap
    openings: OpeningSet
    opening_proof: "FriProof"


@dataclass
class ProofWithPublicInputs:
    proof: Proof
    public_inputs: List[int]


def fri_instance(data: CircuitData, zeta, oracles) -> "FriInstanceInfo":
    """CommonCircuitData::get_fri_instance: every polynomial of the four oracles at zeta, the Zs at g zeta"""
    from .fri import FriBatchInfo, FriInstanceInfo, FriPolynomialInfo
    g = _root(data.common.degree_bits)
    zeta_next = (zeta[0] * g % P, zeta[1] * g % P)
    all_polys = [FriPolynomialInfo(o, i) for o, b in enumerate(oracles) for i in range(b.num_polys)]
    zs = FriPolynomialInfo.from_range(2, range(data.num_challenges))
    zk = data.zero_knowledge
    return FriInstanceInfo([FriBatchInfo(tuple(zeta), all_polys), FriBatchInfo(zeta_next, zs)], oracles_blinding=[False, zk, zk, zk])


def _root(n_log: int) -> int:
    return pow(1753635133440165772, 1 << (32 - n_log), P)


def _ext_pow(x, e: int):
    r, x = (1, 0), tuple(x)
    while e:
        if e & 1:
            r = ((r[0] * x[0] + 7 * r[1] * x[1]) % P, (r[0] * x[1] + r[1] * x[0]) % P)
        x = ((x[0] * x[0] + 7 * x[1] * x[1]) % P, 2 * x[0] * x[1] % P)
        e >>= 1
    return r


PROVE_STAGES = ("wires_commit", "z", "z_commit", "quotient_values", "quotient_commit", "openings", "fri")


def prove(ctx: Context, data: CircuitData, wires, public_inputs, mul_by_x: bool, on_stage=None, salt_key=None) -> ProofWithPublicInputs:
    """plonk/prover.rs prove() on the device, in plonky2's transcript order.  wires: the (135, n) CUDA tensor of witness values
    (num_wires columns); it is only read.  Every polynomial stays in HBM: only challenges, caps, openings and query answers
    cross PCIe.  Raises QuotientError for a witness whose vanishing polynomial is not divisible by Z_H (only checked when
    quotient_degree_factor < 2^quotient_degree_bits).  mul_by_x has no default, for the reason fri.prove_openings gives.
    on_stage(name), when given, is called as each stage is about to be enqueued (PROVE_STAGES) and with "end" after the last
    one, e.g. to record CUDA events on the ctx stream.
    With data.zero_knowledge, the wires, Z + partial products and quotient commitments are salted (plonky2's blinding = true):
    each salt is generated on the device inside its commit stage from the ChaCha20 stream of salt_key (random_field_device,
    nonce = the PlonkOracle index).  salt_key defaults to 32 fresh bytes from the OS for every proof; pass one only to
    reproduce a proof.  A salt_key for a circuit without zero_knowledge, or one that is not 32 bytes, is a ValueError."""
    import torch
    from .fri import Challenger, prove_openings
    from .plonky2 import PoseidonHash
    common, cfg = data.common, data.fri_params.config
    n = 1 << common.degree_bits
    if wires.dim() != 2 or wires.shape[1] != n or wires.shape[0] < 135 or not wires.is_cuda:
        raise ValueError("wires must be a (num_wires, 2^degree_bits) CUDA tensor")
    zk = data.zero_knowledge
    if salt_key is not None and not zk:
        raise ValueError("salt_key is only used when the circuit has zero_knowledge")
    if zk:
        salt_key = secrets.token_bytes(32) if salt_key is None else bytes(salt_key)
        if len(salt_key) != 32:
            raise ValueError("salt_key must be 32 bytes")
    N = n << cfg.rate_bits
    salt = (lambda oracle: salt_device(ctx, salt_key, oracle, N)) if zk else (lambda oracle: None)
    wires = wires.contiguous()
    torch.cuda.current_stream(wires.device).synchronize()        # inputs written on torch's stream are complete
    Cn = data.num_challenges
    challenger = Challenger(ctx)
    public_inputs_hash = PoseidonHash.hash_no_pad(_u64(list(public_inputs)), ctx)
    challenger.observe_hash(data.circuit_digest)
    challenger.observe_hash(public_inputs_hash)
    stage = on_stage or (lambda name: None)

    stage("wires_commit")
    wires_commitment = PolynomialBatch.from_device(wires, cfg.rate_bits, zk, cfg.cap_height, ctx=ctx, salt=salt(PLONK_ORACLE_WIRES))
    challenger.observe_cap(wires_commitment._cap)
    betas = challenger.get_n_challenges(Cn)
    gammas = challenger.get_n_challenges(Cn)

    stage("z")
    zpp = zs_partial_products_device(ctx, wires[:common.num_routed_wires], data.sigmas, common.k_is, betas, gammas,
                                     common.quotient_degree_factor)
    stage("z_commit")
    zpp_commitment = PolynomialBatch.from_device(zpp, cfg.rate_bits, zk, cfg.cap_height, ctx=ctx,
                                                 salt=salt(PLONK_ORACLE_ZS_PARTIAL_PRODUCTS))
    challenger.observe_cap(zpp_commitment._cap)
    alphas = challenger.get_n_challenges(Cn)

    cs = data.constants_sigmas_commitment
    stage("quotient_values")
    # (the salt columns come last in a blinded LDE: the quotient reads the polynomial columns only, as get_lde_values does)
    q = compute_quotient_values_device(ctx, common, cs.lde, wires_commitment.lde[:wires_commitment.num_polys],
                                       zpp_commitment.lde[:zpp_commitment.num_polys], betas, gammas, alphas,
                                       public_inputs_hash.elements)
    stage("quotient_commit")
    chunks = quotient_chunks_device(ctx, q, common.degree_bits, common.quotient_degree_factor)
    quotient_commitment = PolynomialBatch.from_device(chunks, cfg.rate_bits, zk, cfg.cap_height, is_coeffs=True, ctx=ctx,
                                                      salt=salt(PLONK_ORACLE_QUOTIENT))
    challenger.observe_cap(quotient_commitment._cap)

    zeta = challenger.get_extension_challenge()
    if _ext_pow(zeta, n) == (1, 0):
        raise ValueError("Opening point is in the subgroup.")
    oracles = [cs, wires_commitment, zpp_commitment, quotient_commitment]
    instance = fri_instance(data, zeta, oracles)
    stage("openings")
    at_zeta, at_next = batch_openings(instance, oracles)
    for values in (at_zeta, at_next):
        challenger.observe_extension_elements(values)
    nc = data.num_constants
    k_cs, k_w = cs.num_polys, wires_commitment.num_polys
    ow, oz = k_cs + k_w, k_cs + k_w + zpp_commitment.num_polys
    openings = OpeningSet(constants=at_zeta[:nc], plonk_sigmas=at_zeta[nc:k_cs], wires=at_zeta[k_cs:ow],
                          plonk_zs=at_zeta[ow:ow + Cn], plonk_zs_next=at_next, partial_products=at_zeta[ow + Cn:oz],
                          quotient_polys=at_zeta[oz:])
    stage("fri")
    opening_proof = prove_openings(instance, oracles, challenger, data.fri_params, mul_by_x)
    stage("end")
    proof = Proof(wires_commitment._cap, zpp_commitment._cap, quotient_commitment._cap, openings, opening_proof)
    return ProofWithPublicInputs(proof, [int(v) % P for v in public_inputs])
