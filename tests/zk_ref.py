"""TEST INFRASTRUCTURE: plonky2's zero_knowledge = true, restated from memory of plonky2 @ f99ed9c (parity unpinned).

    plonky2/src/plonk/circuit_builder.rs   blind_and_pad, blinding_counts
    plonky2/src/plonk/prover.rs            prove: wires, Z + partial products and quotient committed with blinding = true
    plonky2/src/fri/oracle.rs              a blinded PolynomialBatch appends SALT_SIZE = 4 columns of F::rand_vec(N)
    plonky2/src/fri/verifier.rs            FriParams.hiding: a blinded oracle's leaves hold num_polys + 4 words

- `blinding_counts` and `blind` turn no-op rows of a vanishing_ref / interpolation_ref circuit into the rows blind_and_pad adds:
  regular rows with random wires, and pairs of rows whose routed wires are random and copy-constrained to each other.
- `salts` draws the three salts from the ChaCha20 stream of tests/chacha_ref.py the way prover.prove does.
- `prove` runs plonk_ref.prove's own code with the three salts passed to its commitments (`_SaltedCommits`); `verify` checks
  the leaf shapes, then runs plonk_ref.verify, which hashes whole leaves and reads only the polynomial columns."""
from __future__ import annotations

import copy
import random
import types
from typing import Sequence, Tuple

import numpy as np

import chacha_ref as CR
import plonk_ref as R
from oracle import oracle as O
from oracle import vanishing_ref as V

P = 0xFFFFFFFF00000001
D = 2
SALT_SIZE = 4
# PlonkOracle indices of the blinded oracles (constants + sigmas, index 0, are never blinded)
WIRES, ZS_PARTIAL_PRODUCTS, QUOTIENT = 1, 2, 3


def blinding_counts(degree_bits: int, fri: dict) -> Tuple[int, int]:
    """CircuitBuilder::blinding_counts for a circuit of 2^degree_bits rows: (regular_poly_openings, z_openings).
    fri: plonk_ref.fri_args form (arities are arity_bits)."""
    arity_bits = fri["arities"]
    fri_openings = fri["num_queries"] * (1 + D * sum((1 << a) - 1 for a in arity_bits)
                                         + D * ((1 << degree_bits) >> sum(arity_bits)))
    return D + fri_openings, 2 * D + fri_openings


def blind(c: V.Circuit, regular: int, pairs: int, seed: int = 0) -> V.Circuit:
    """a copy of `c` in which the last `regular + 2 * pairs` no-op rows are blinding rows: `regular` rows of random wires, then
    `pairs` pairs (a, b) whose routed wires hold the same random values, each cell (j, a) copy-constrained to (j, b).  The
    no-op rows' routed cells are fixed points of sigma before, so each pair's cells become 2-cycles:
    sigma_j[a] = k_j w^b, sigma_j[b] = k_j w^a.  Only wires and sigmas change; no-op rows have no constraints."""
    c = copy.deepcopy(c)
    rnd = random.Random(seed)
    noop = c.gates.index(V.NOOP)
    rows = [r for r in range(c.n) if c.row_gate[r] == noop]
    need = regular + 2 * pairs
    if need > len(rows):
        raise ValueError(f"{need} blinding rows do not fit in the circuit's {len(rows)} no-op rows")
    rows = rows[len(rows) - need:]
    w = V.root(c.n_log)
    cell = lambda j, r: c.k_is[j] * pow(w, r, P) % P
    for r in rows:
        for j in range(V.NUM_ROUTED):
            assert c.sigmas[j][r] == cell(j, r), "a blinding row's routed cell must be its own copy cycle"
        for j in range(V.NUM_WIRES):
            c.wires[j][r] = rnd.randrange(P)
    for i in range(pairs):
        a, b = rows[regular + 2 * i], rows[regular + 2 * i + 1]
        for j in range(V.NUM_ROUTED):
            c.wires[j][b] = c.wires[j][a]
            c.sigmas[j][a], c.sigmas[j][b] = cell(j, b), cell(j, a)
    c.blinding_rows = (rows[:regular], [(rows[regular + 2 * i], rows[regular + 2 * i + 1]) for i in range(pairs)])
    return c


def salts(key: bytes, n_log: int, rate_bits: int):
    """the (4, N) salts of the wires, Z + partial products and quotient commitments: elements [0, 4N) of the stream
    (key, le32(oracle index) || 0^8), element c*N + i = salt column c at natural LDE row i"""
    N = 1 << (n_log + rate_bits)
    return tuple(CR.elements(key, CR.nonce_for_oracle(o), 0, SALT_SIZE * N).reshape(SALT_SIZE, N)
                 for o in (WIRES, ZS_PARTIAL_PRODUCTS, QUOTIENT))


class _SaltedCommits:
    """oracle/oracle.py as plonk_ref.prove sees it, except that its commitments are salted in PlonkOracle order: plonk_ref.prove
    commits constants + sigmas (index 0, never blinded), then the wires, Z + partial products and quotient (1, 2, 3)"""

    def __init__(self, salt_columns):
        self._salts = [None] + list(salt_columns)
        self.calls = 0

    def __getattr__(self, name):
        return getattr(O, name)

    def commit(self, inp, rate_bits, cap_height, is_coeffs=False, salt=None):
        assert salt is None and self.calls < len(self._salts), "plonk_ref.prove commits four oracles, unsalted"
        salt = self._salts[self.calls]
        self.calls += 1
        return O.commit(inp, rate_bits, cap_height, is_coeffs=is_coeffs, salt=salt)


def prove(c: V.Circuit, public_inputs: Sequence[int], fri: dict, mul_by_x: bool, key: bytes, ref=V, wires=None) -> dict:
    """prove() with zero_knowledge = true: plonk_ref.prove's code, unchanged, with the three salts of `key` given to the wires,
    Z + partial products and quotient commitments"""
    oracle = _SaltedCommits(salts(key, c.n_log, fri["rate_bits"]))
    fn = R.prove
    salted = types.FunctionType(fn.__code__, dict(fn.__globals__, O=oracle), fn.__name__, fn.__defaults__, fn.__closure__)
    salted.__kwdefaults__ = fn.__kwdefaults__
    proof = salted(c, public_inputs, fri, mul_by_x, ref=ref, wires=wires)
    assert oracle.calls == 4
    return proof


def leaf_shapes_ok(proof: dict, num_polys: Sequence[int]) -> bool:
    """the verifier's shape check with hiding: every opened initial leaf of oracle o holds num_polys[o] words, plus SALT_SIZE for
    the blinded oracles 1..3"""
    want = [num_polys[0]] + [k + SALT_SIZE for k in num_polys[1:]]
    return all(len(row) == k for rnd in proof["opening_proof"]["rounds"] for (row, _), k in zip(rnd["initial"], want))


def verify(proof: dict, public_inputs: Sequence[int], c: V.Circuit, circuit_digest, constants_sigmas_cap, fri: dict,
           mul_by_x: bool, ref=V) -> bool:
    """plonk/verifier.rs verify with FriParams.hiding = true"""
    o = proof["openings"]
    ks = [len(o["constants"]) + len(o["plonk_sigmas"]), len(o["wires"]), len(o["plonk_zs"]) + len(o["partial_products"]),
          len(o["quotient_polys"])]
    if not leaf_shapes_ok(proof, ks):
        return False
    return R.verify(proof, public_inputs, c, circuit_digest, constants_sigmas_cap, fri, mul_by_x, ref=ref)


def strip_salts(proof: dict) -> dict:
    """the proof with the salt words taken off every opened leaf of the blinded oracles"""
    p = copy.deepcopy(proof)
    for rnd in p["opening_proof"]["rounds"]:
        rnd["initial"] = [rnd["initial"][0]] + [(np.asarray(row)[:-SALT_SIZE].copy(), sib) for row, sib in rnd["initial"][1:]]
    return p
