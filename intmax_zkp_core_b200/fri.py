"""Rows N2 + N3 of SURVEY.md section 8(f): plonky2's opening proof on the device-resident commitments.

Mirrors, with the same names and argument meaning (plonky2 @ f99ed9c, un-vendored dependency of the reference; reached
from every `prove()`, e.g. /root/reference/src/rollup/circuits/mod.rs:1247):
    FriConfig / FriParams / FriReductionStrategy              plonky2/src/fri/mod.rs, fri/reduction_strategies.rs
    FriInstanceInfo / FriBatchInfo / FriPolynomialInfo        plonky2/src/fri/structure.rs
    Challenger (overwrite-mode duplex sponge)                 plonky2/src/iop/challenger.rs
    PolynomialBatch::prove_openings                           plonky2/src/fri/oracle.rs
    fri_proof / fri_committed_trees / fri_proof_of_work / fri_prover_query_rounds     plonky2/src/fri/prover.rs
    FriProof / FriQueryRound / FriQueryStep / FriInitialTreeProof                      plonky2/src/fri/proof.rs

The polynomial work (alpha-reduction of all oracle polynomials, division by X - z, the final LDE, every commit-phase
Merkle tree, the coefficient folds, the proof-of-work search, the query gathers) runs in the CUDA library on data that
never leaves HBM; this file only sequences the Fiat-Shamir transcript exactly where plonky2 draws each challenge.
Two things plonky2 leaves open are pinned here and named in DESIGN.md: the 2022 code multiplies final_poly by X
(`mul_by_x=True`), and the proof-of-work witness is the smallest one (rayon's find_any returns any).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .plonky2 import Context, HashOut, MerkleCap, MerkleProof, PolynomialBatch, PoseidonPermutation, _p, _u64, default_context

P = 0xFFFFFFFF00000001
SPONGE_RATE = 8
SPONGE_WIDTH = 12
Ext = Tuple[int, int]      # a + b X in F_p[X] / (X^2 - 7)
FRI_MUL_BY_X = 1


# ------------------------------------------------------------------------------------------------ parameters
@dataclass
class ConstantArityBits:
    """FriReductionStrategy::ConstantArityBits(arity_bits, final_poly_bits) — reduction_strategies.rs."""
    arity_bits: int
    final_poly_bits: int

    def reduction_arity_bits(self, degree_bits: int, rate_bits: int, cap_height: int, num_queries: int) -> List[int]:
        out = []
        while degree_bits > self.final_poly_bits and degree_bits + rate_bits - self.arity_bits >= cap_height:
            out.append(self.arity_bits)
            assert degree_bits >= self.arity_bits
            degree_bits -= self.arity_bits
        return out


@dataclass
class FriConfig:
    rate_bits: int = 3
    cap_height: int = 4
    proof_of_work_bits: int = 16
    reduction_strategy: object = field(default_factory=lambda: ConstantArityBits(4, 5))
    num_query_rounds: int = 28

    def fri_params(self, degree_bits: int, hiding: bool = False) -> "FriParams":
        arities = self.reduction_strategy.reduction_arity_bits(degree_bits, self.rate_bits, self.cap_height, self.num_query_rounds)
        return FriParams(config=self, hiding=hiding, degree_bits=degree_bits, reduction_arity_bits=arities)


def standard_recursion_fri_config() -> FriConfig:
    """The `fri_config` of CircuitConfig::standard_recursion_config(), the only configuration the reference proves with."""
    return FriConfig()


@dataclass
class FriParams:
    config: FriConfig
    hiding: bool
    degree_bits: int
    reduction_arity_bits: List[int]

    def lde_bits(self) -> int:
        return self.degree_bits + self.config.rate_bits

    def lde_size(self) -> int:
        return 1 << self.lde_bits()

    def final_poly_bits(self) -> int:
        return self.degree_bits - sum(self.reduction_arity_bits)


@dataclass
class FriPolynomialInfo:
    oracle_index: int
    polynomial_index: int

    @staticmethod
    def from_range(oracle_index: int, polynomial_indices: Sequence[int]) -> List["FriPolynomialInfo"]:
        return [FriPolynomialInfo(oracle_index, i) for i in polynomial_indices]


@dataclass
class FriBatchInfo:
    point: Ext
    polynomials: List[FriPolynomialInfo]


@dataclass
class FriInstanceInfo:
    batches: List[FriBatchInfo]
    oracles_blinding: Optional[List[bool]] = None


# ------------------------------------------------------------------------------------------------ transcript
class Challenger:
    """iop/challenger.rs: sponge_state / input_buffer / output_buffer, inputs overwrite the rate part.

    Same transcript as plonky2's, evaluated lazily: observations are only queued, and the permutations they imply (one per
    full chunk of 8, as `observe_element` triggers them, plus the one `get_challenge` runs on a partial chunk or an empty
    output buffer) run on the device in ONE call when the next challenge is drawn (b200zkp_duplex_chain).  A draw of
    several challenges asks for all the permutations it will need in the same call."""

    def __init__(self, ctx: Optional[Context] = None):
        self._ctx = ctx or default_context()
        self.sponge_state = np.zeros(SPONGE_WIDTH, dtype=np.uint64)
        self.input_buffer: List[int] = []        # every observation since the last draw (may exceed the rate: lazy)
        self.output_buffer: List[int] = []

    def observe_element(self, e: int):
        self.output_buffer = []
        self.input_buffer.append(int(e) % P)

    def observe_elements(self, es):
        es = [int(e) % P for e in np.asarray(es, dtype=np.uint64).reshape(-1).tolist()]
        if es:
            self.output_buffer = []
            self.input_buffer.extend(es)

    def observe_extension_element(self, e: Ext):
        self.observe_elements(list(e))

    def observe_extension_elements(self, es):
        self.observe_elements([x for e in es for x in e])

    def observe_hash(self, h):
        self.observe_elements(h.elements if isinstance(h, HashOut) else h)

    def observe_cap(self, cap):
        self.observe_elements(cap.flatten() if isinstance(cap, MerkleCap) else cap)

    def _chain(self, n_squeeze: int) -> np.ndarray:
        """every queued observation (with all the permutations it implies), then n_squeeze further permutations: one call"""
        m = len(self.input_buffer)
        state = np.ascontiguousarray(self.sponge_state, dtype=np.uint64)
        inputs = _u64(self.input_buffer) if m else None
        squeezed = np.zeros((max(n_squeeze, 1), SPONGE_RATE), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_duplex_chain(self._ctx._h, _p(state), _p(inputs) if m else None, m, n_squeeze,
                                                            _p(squeezed) if n_squeeze else None))
        self.sponge_state = state
        self.input_buffer = []
        return squeezed[:n_squeeze]

    def get_challenge(self) -> int:
        return self.get_n_challenges(1)[0]

    def get_n_challenges(self, n: int) -> List[int]:
        out: List[int] = []
        while len(out) < n:
            if self.input_buffer:
                # plonky2 duplexes on every 8th observation and once more for a partial chunk when a challenge is drawn
                self._chain(0)
                self.output_buffer = [int(v) for v in self.sponge_state[:SPONGE_RATE]]
            elif not self.output_buffer:
                # one permutation per 8 challenges still missing; challenges pop from the END of each block of rate words
                blocks = self._chain(-(-(n - len(out)) // SPONGE_RATE))
                for blk in blocks[:-1]:
                    out.extend(int(v) for v in blk[::-1])
                self.output_buffer = [int(v) for v in blocks[-1]]
            else:
                out.append(self.output_buffer.pop())
        return out

    def duplexing(self):
        """plonky2's name for one forced step: the queued observations, or one permutation when nothing is queued"""
        if self.input_buffer:
            self._chain(0)
            self.output_buffer = [int(v) for v in self.sponge_state[:SPONGE_RATE]]
        else:
            self.output_buffer = [int(v) for v in self._chain(1)[0]]

    def get_hash(self) -> HashOut:
        return HashOut(self.get_n_challenges(4))

    def get_extension_challenge(self) -> Ext:
        c = self.get_n_challenges(2)
        return (c[0], c[1])

    def duplexing(self):
        """plonky2's name for one flush (kept for callers that force it)"""
        self._duplex_once_or_absorb()


# ------------------------------------------------------------------------------------------------ proof
@dataclass
class FriInitialTreeProof:
    evals_proofs: List[Tuple[np.ndarray, MerkleProof]]      # per oracle: (leaf row, Merkle proof)


@dataclass
class FriQueryStep:
    evals: np.ndarray                                        # (arity, 2)
    merkle_proof: MerkleProof


@dataclass
class FriQueryRound:
    initial_trees_proof: FriInitialTreeProof
    steps: List[FriQueryStep]


@dataclass
class FriProof:
    commit_phase_merkle_caps: List[MerkleCap]
    query_round_proofs: List[FriQueryRound]
    final_poly: np.ndarray                                   # (len, 2) extension coefficients
    pow_witness: int


def _instance_args(instance: FriInstanceInfo, oracles: Sequence[PolynomialBatch]):
    """oracles, n_oracles, n_points, points, point_n_polys, poly_oracle, poly_index as b200zkp_fri_begin and
    b200zkp_batch_openings take them (each pointer keeps its array alive)"""
    handles = (C.c_void_p * len(oracles))(*[o._h for o in oracles])
    points = _u64([list(b.point) for b in instance.batches]).reshape(-1)
    counts = np.array([len(b.polynomials) for b in instance.batches], dtype=np.uint32)
    po = np.array([p.oracle_index for b in instance.batches for p in b.polynomials], dtype=np.uint32)
    pi = np.array([p.polynomial_index for b in instance.batches for p in b.polynomials], dtype=np.uint32)
    return (handles, len(oracles), len(instance.batches), _p(points), counts.ctypes.data_as(C.c_void_p),
            po.ctypes.data_as(C.c_void_p), pi.ctypes.data_as(C.c_void_p))


def batch_openings(instance: FriInstanceInfo, oracles: Sequence[PolynomialBatch], ctx: Optional[Context] = None) -> List[List[Ext]]:
    """OpeningSet::new in its FRI form (to_fri_openings): the value of every polynomial of `instance` at its batch's point,
    batch after batch, in the order the challenger observes them.  One device call for the whole instance
    (b200zkp_batch_openings) on the resident coefficients."""
    ctx = ctx or oracles[0]._ctx
    m = sum(len(b.polynomials) for b in instance.batches)
    out = np.empty((max(m, 1), 2), dtype=np.uint64)
    args = _instance_args(instance, oracles)
    ctx.check(ctx._lib.b200zkp_batch_openings(ctx._h, *args, _p(out)))
    vals = [(int(a), int(b)) for a, b in out[:m]]
    res, off = [], 0
    for b in instance.batches:
        res.append(vals[off:off + len(b.polynomials)])
        off += len(b.polynomials)
    return res


class FriCommitPhase:
    """Device state of one opening proof: current coefficients / values and the committed layer trees."""

    def __init__(self, ctx: Context, handle):
        self._ctx, self._h = ctx, handle

    @classmethod
    def from_oracles(cls, instance: FriInstanceInfo, oracles: Sequence[PolynomialBatch], alpha: Ext, mul_by_x: bool,
                     ctx: Optional[Context] = None) -> "FriCommitPhase":
        """prove_openings up to (and including) `lde_final_values`."""
        ctx = ctx or oracles[0]._ctx
        a = _u64(list(alpha))
        h = C.c_void_p()
        ctx.check(ctx._lib.b200zkp_fri_begin(ctx._h, *_instance_args(instance, oracles), _p(a), FRI_MUL_BY_X if mul_by_x else 0,
                                             C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_coeffs(cls, coeffs, rate_bits: int, ctx: Optional[Context] = None) -> "FriCommitPhase":
        """fri_proof's own entry: `lde_polynomial_coeffs` given as (n, 2) extension coefficients."""
        ctx = ctx or default_context()
        c = _u64(coeffs)
        assert c.ndim == 2 and c.shape[1] == 2
        n_log = int(c.shape[0]).bit_length() - 1
        assert 1 << n_log == c.shape[0]
        h = C.c_void_p()
        ctx.check(ctx._lib.b200zkp_fri_begin_from_coeffs(ctx._h, _p(c), n_log, rate_bits, C.byref(h)))
        return cls(ctx, h)

    def shape(self):
        s = (C.c_uint32 * 4)()
        self._ctx.check(self._ctx._lib.b200zkp_fri_shape(self._h, s))
        return dict(n_log=s[0], rate_bits=s[1], cur_log=s[2], layers=s[3])

    def coeffs(self) -> np.ndarray:
        out = np.empty((1 << self.shape()["cur_log"], 2), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_fri_coeffs(self._h, _p(out)))
        return out

    def commit_layer(self, arity_bits: int, cap_height: int) -> MerkleCap:
        cap = np.empty((1 << cap_height, 4), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_fri_commit_layer(self._h, arity_bits, cap_height, _p(cap)))
        return MerkleCap(cap)

    def fold(self, beta: Ext):
        self._ctx.check(self._ctx._lib.b200zkp_fri_fold(self._h, _p(_u64(list(beta)))))

    def final_poly(self) -> np.ndarray:
        s = self.shape()
        out = np.empty(((1 << s["cur_log"]) >> s["rate_bits"], 2), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_fri_final_poly(self._h, _p(out)))
        return out

    def query(self, layer: int, indices: Sequence[int], arity_bits: int, depth: int):
        idx = _u64(indices)
        evals = np.empty((idx.size, 1 << arity_bits, 2), dtype=np.uint64)
        sib = np.empty((idx.size, depth, 4), dtype=np.uint64)
        self._ctx.check(self._ctx._lib.b200zkp_fri_query(self._h, layer, _p(idx), idx.size, _p(evals),
                                                         _p(sib) if sib.size else None))
        return evals, sib

    def close(self):
        if self._h and getattr(self._ctx, "_h", None):
            self._ctx._lib.b200zkp_fri_free(self._h)
        self._h = None

    def __del__(self):
        self.close()


def fri_proof_of_work(current_hash: HashOut, config: FriConfig, ctx: Optional[Context] = None) -> int:
    """prover.rs fri_proof_of_work: hash_no_pad(current_hash || w).elements[0] with proof_of_work_bits leading zeros
    (64 - F::order().bits() = 0 for Goldilocks).  Returns the smallest such w."""
    ctx = ctx or default_context()
    state = np.zeros(SPONGE_WIDTH, dtype=np.uint64)
    state[:4] = current_hash.elements
    w = C.c_uint64()
    ctx.check(ctx._lib.b200zkp_pow_grind(ctx._h, _p(state), 4, 0, config.proof_of_work_bits, 0, C.byref(w)))
    return int(w.value)


def fri_proof(initial_merkle_trees: Sequence[PolynomialBatch], commit: FriCommitPhase, challenger: Challenger,
              fri_params: FriParams) -> FriProof:
    """prover.rs fri_proof: commit phase, proof of work, query rounds."""
    cfg = fri_params.config
    n = fri_params.lde_size()
    ctx = commit._ctx
    # commit phase (fri_committed_trees)
    caps = []
    for arity_bits in fri_params.reduction_arity_bits:
        cap = commit.commit_layer(arity_bits, cfg.cap_height)
        challenger.observe_cap(cap)
        caps.append(cap)
        commit.fold(challenger.get_extension_challenge())
    final_poly = commit.final_poly()
    challenger.observe_extension_elements([(int(a), int(b)) for a, b in final_poly])
    # proof of work
    pow_witness = fri_proof_of_work(challenger.get_hash(), cfg, ctx)
    # query phase: the indices are drawn first (they do not depend on the answers), the gathers are batched per tree
    x_indices = [challenger.get_challenge() % n for _ in range(cfg.num_query_rounds)]
    initial = [t.rows(x_indices) for t in initial_merkle_trees]
    steps_per_layer = []
    idx = list(x_indices)
    lde_bits = fri_params.lde_bits()
    for i, arity_bits in enumerate(fri_params.reduction_arity_bits):
        idx = [x >> arity_bits for x in idx]
        lde_bits -= arity_bits
        steps_per_layer.append(commit.query(i, idx, arity_bits, lde_bits - cfg.cap_height))
    rounds = []
    for r in range(cfg.num_query_rounds):
        ip = FriInitialTreeProof([(rows[r], MerkleProof(sib[r])) for rows, sib in initial])
        steps = [FriQueryStep(evals[r], MerkleProof(sib[r])) for evals, sib in steps_per_layer]
        rounds.append(FriQueryRound(ip, steps))
    return FriProof(caps, rounds, final_poly, pow_witness)


def prove_openings(instance: FriInstanceInfo, oracles: Sequence[PolynomialBatch], challenger: Challenger,
                   fri_params: FriParams, mul_by_x: bool) -> FriProof:
    """fri/oracle.rs PolynomialBatch::prove_openings.

    mul_by_x has no default on purpose: whether final_poly carries the factor X depends on the plonky2 revision (the 2022
    code inserts it, later code pads the quotient) and no proof fixture in the reference pins it (DESIGN.md section 4b) — the
    caller states which verifier the proof is for."""
    assert all(o.degree_log == fri_params.degree_bits and o.rate_bits == fri_params.config.rate_bits for o in oracles)
    alpha = challenger.get_extension_challenge()
    commit = FriCommitPhase.from_oracles(instance, oracles, alpha, mul_by_x)
    try:
        return fri_proof(oracles, commit, challenger, fri_params)
    finally:
        commit.close()
