"""TEST INFRASTRUCTURE: a restated plonky2 prove() and verify() composed from the restatements under oracle/.

    plonky2 @ f99ed9c  plonky2/src/plonk/prover.rs     prove
                       plonky2/src/plonk/verifier.rs   verify, plonk/get_challenges.rs
                       plonky2/src/plonk/proof.rs      OpeningSet, to_fri_openings
                       plonky2/src/plonk/circuit_data.rs  get_fri_instance, circuit_digest

The prover strings together oracle.commit, perm_ref.partial_products_and_zs, `ref.quotient_values` (oracle/vanishing_ref, or
tests/interpolation_ref for circuits with the interpolation gates) and the coset iNTT, oracle.eval_ext2, fri_ref.prove_openings
and fri_ref's challenger, in plonky2's transcript order.  The verifier recomputes every challenge from the proof, evaluates the
vanishing polynomial at zeta from the openings over the quadratic extension and checks
    vanishing_i(zeta) == Z_H(zeta) * sum_j zeta^(n j) q_(i,j)(zeta)
for every challenge, then runs fri_ref.verify.  zero_knowledge = false throughout; parity unpinned, as for the pieces.

The vanishing polynomial at zeta runs vanishing_ref's own code unchanged on `Ext2`, a duck-typed element of F_p[X]/(X^2 - 7)
(`+ - *`, `% P` the identity, `pow(x, e, P)` the extension power).  Its one inversion, L_1's pow(v, P - 2, P), is
Fermat's inverse over F_p; `_vanishing_terms_at` runs that code with a `pow` that gives the extension inverse for it.
Pure Python: small sizes only."""
from __future__ import annotations

import builtins
import copy
import types
from typing import List, Sequence

import numpy as np

from oracle import fri_ref as F
from oracle import oracle as O
from oracle import perm_ref
from oracle import vanishing_ref as V

P = 0xFFFFFFFF00000001
W = 7
NUM_CHALLENGES = 2
QUOTIENT_DEGREE_FACTOR = 8
QUOTIENT_DEGREE_BITS = 3


# ---------------------------------------------------------------------------------------------------- the extension field
class Ext2:
    """a + b X in F_p[X] / (X^2 - 7), with the operators vanishing_ref's gate code applies to field elements"""
    __slots__ = ("a", "b")

    def __init__(self, a, b=0):
        self.a, self.b = int(a) % P, int(b) % P

    @staticmethod
    def _of(y) -> "Ext2":
        return y if isinstance(y, Ext2) else Ext2(y)

    def __add__(self, y):
        y = Ext2._of(y)
        return Ext2(self.a + y.a, self.b + y.b)

    __radd__ = __add__

    def __sub__(self, y):
        y = Ext2._of(y)
        return Ext2(self.a - y.a, self.b - y.b)

    def __rsub__(self, y):
        return Ext2._of(y) - self

    def __neg__(self):
        return Ext2(-self.a, -self.b)

    def __mul__(self, y):
        if not isinstance(y, Ext2):
            return Ext2(self.a * int(y), self.b * int(y))
        return Ext2(self.a * y.a + W * self.b * y.b, self.a * y.b + self.b * y.a)

    __rmul__ = __mul__

    def __mod__(self, m):
        assert m == P
        return self

    def __pow__(self, e, m=None):
        assert m is None or m == P
        r, x = Ext2(1), self
        e = int(e)
        while e:
            if e & 1:
                r = r * x
            x = x * x
            e >>= 1
        return r

    def inverse(self) -> "Ext2":
        d = builtins.pow((self.a * self.a - W * self.b * self.b) % P, P - 2, P)
        return Ext2(self.a * d, -self.b * d)

    def __eq__(self, y):
        y = Ext2._of(y)
        return self.a == y.a and self.b == y.b

    def __hash__(self):
        return hash((self.a, self.b))

    def __repr__(self):
        return f"Ext2({self.a}, {self.b})"

    def pair(self):
        return (self.a, self.b)


def _pow(x, e, m=None):
    if isinstance(x, Ext2) and e == P - 2 and m == P:
        return x.inverse()
    return builtins.pow(x, e, m) if m is not None else builtins.pow(x, e)


def _vanishing_terms_at(ref):
    fn = ref.vanishing_terms_at
    return types.FunctionType(fn.__code__, dict(fn.__globals__, pow=_pow), fn.__name__, fn.__defaults__, fn.__closure__)


# ---------------------------------------------------------------------------------------------------- helpers
def with_public_inputs(c: V.Circuit, public_inputs: Sequence[int]) -> V.Circuit:
    """a copy of `c` whose public-input row holds hash_no_pad(public_inputs): the row's four wires are fixed points of sigma, so
    the circuit stays satisfied"""
    c = copy.deepcopy(c)
    h = [int(v) for v in O.hash_no_pad([int(x) % P for x in public_inputs])]
    row = c.row_gate.index(c.gates.index(V.PUBLIC_INPUT))
    for i in range(4):
        assert c.sigmas[i][row] == c.k_is[i] * pow(V.root(c.n_log), row, P) % P
        c.wires[i][row] = h[i]
    c.pi_hash = h
    return c


def fri_args(n_log: int, rate_bits: int = 3, cap_height: int = 4, pow_bits: int = 16, num_queries: int = 28):
    """(rate_bits, cap_height, reduction arities, pow_bits, num_queries): standard_recursion_config's FRI by default"""
    arities, d = [], n_log
    while d > 5 and d + rate_bits - 4 >= cap_height:
        arities.append(4)
        d -= 4
    return dict(rate_bits=rate_bits, cap_height=cap_height, arities=arities, pow_bits=pow_bits, num_queries=num_queries)


def _coset_ifft(values: Sequence[int]) -> List[int]:
    """PolynomialValues::coset_ifft(7): values on 7 <w> in natural order -> coefficients"""
    coeffs = O.ifft(np.array(values, dtype=np.uint64))
    inv, pw, out = pow(V.GENERATOR, P - 2, P), 1, []
    for c in coeffs:
        out.append(int(c) * pw % P)
        pw = pw * inv % P
    return out


def instance(c: V.Circuit, zeta, ks: Sequence[int]):
    """get_fri_instance: every polynomial of the four oracles at zeta, the Zs at g zeta"""
    zeta_next = F.escale(zeta, V.root(c.n_log))
    return [(zeta, [(o, i) for o, k in enumerate(ks) for i in range(k)]), (zeta_next, [(2, i) for i in range(NUM_CHALLENGES)])]


def split_openings(c: V.Circuit, at_zeta, at_next, ks):
    nc = c.num_selectors + V.NUM_GATE_CONSTANTS
    ow, oz = ks[0] + ks[1], ks[0] + ks[1] + ks[2]
    return dict(constants=at_zeta[:nc], plonk_sigmas=at_zeta[nc:ks[0]], wires=at_zeta[ks[0]:ow],
                plonk_zs=at_zeta[ow:ow + NUM_CHALLENGES], partial_products=at_zeta[ow + NUM_CHALLENGES:oz],
                quotient_polys=at_zeta[oz:], plonk_zs_next=at_next)


def fri_openings(o: dict):
    return [o["constants"] + o["plonk_sigmas"] + o["wires"] + o["plonk_zs"] + o["partial_products"] + o["quotient_polys"],
            o["plonk_zs_next"]]


def circuit_digest(constants_sigmas_cap) -> List[int]:
    return [int(v) for v in O.hash_no_pad(np.asarray(constants_sigmas_cap, dtype=np.uint64).reshape(-1))]


# ---------------------------------------------------------------------------------------------------- prover
def prove(c: V.Circuit, public_inputs: Sequence[int], fri: dict, mul_by_x: bool, ref=V, wires=None) -> dict:
    """prove() for circuit `c` (wires: its witness unless given); returns dict(wires_cap, plonk_zs_partial_products_cap,
    quotient_polys_cap, openings (OpeningSet fields), opening_proof (fri_ref's form), circuit_digest, constants_sigmas_cap)"""
    r, h = fri["rate_bits"], fri["cap_height"]
    n = c.n
    wires = [list(map(int, col)) for col in (c.wires if wires is None else wires)]
    cs = O.commit(c.constants + c.sigmas, r, h)
    digest = circuit_digest(cs["cap"])
    ch = F.Challenger()
    ch.observe_elements(digest)
    ch.observe_elements(O.hash_no_pad([int(x) % P for x in public_inputs]))
    w = O.commit(wires, r, h)
    ch.observe_cap(w["cap"])
    betas = [ch.get_challenge() for _ in range(NUM_CHALLENGES)]
    gammas = [ch.get_challenge() for _ in range(NUM_CHALLENGES)]
    zpp_cols = perm_ref.partial_products_and_zs(wires[:V.NUM_ROUTED], c.sigmas, c.k_is, betas, gammas, QUOTIENT_DEGREE_FACTOR)
    zpp = O.commit(zpp_cols, r, h)
    ch.observe_cap(zpp["cap"])
    alphas = [ch.get_challenge() for _ in range(NUM_CHALLENGES)]
    nat = lambda com: [O.coset_lde(row, r) for row in com["coeffs"]]
    cw = copy.copy(c)
    cw.pi_hash = [int(v) for v in O.hash_no_pad([int(x) % P for x in public_inputs])]
    qv = ref.quotient_values(cw, nat(cs), nat(w), nat(zpp), betas, gammas, alphas, QUOTIENT_DEGREE_FACTOR, r, QUOTIENT_DEGREE_BITS)
    chunks = []
    for vals in qv:
        coeffs = _coset_ifft(vals)
        chunks += [coeffs[j * n:(j + 1) * n] for j in range(QUOTIENT_DEGREE_FACTOR)]
    q = O.commit(np.array(chunks, dtype=np.uint64), r, h, is_coeffs=True)
    ch.observe_cap(q["cap"])
    zeta = ch.get_extension_challenge()
    assert F.epow(zeta, n) != (1, 0), "Opening point is in the subgroup."
    commits = [cs, w, zpp, q]
    ks = [com["coeffs"].shape[0] for com in commits]
    batches = instance(c, zeta, ks)
    opened = [[tuple(int(v) for v in O.eval_ext2(commits[o]["coeffs"][i], np.array(pt, dtype=np.uint64))) for o, i in polys]
              for pt, polys in batches]
    for vals in opened:
        ch.observe_extension_elements(vals)
    op = F.prove_openings(commits, batches, ch, r, h, fri["arities"], fri["pow_bits"], fri["num_queries"], mul_by_x)
    return dict(wires_cap=w["cap"], plonk_zs_partial_products_cap=zpp["cap"], quotient_polys_cap=q["cap"],
                openings=split_openings(c, opened[0], opened[1], ks), opening_proof=op, circuit_digest=digest,
                constants_sigmas_cap=cs["cap"])


# ---------------------------------------------------------------------------------------------------- verifier
def verify(proof: dict, public_inputs: Sequence[int], c: V.Circuit, circuit_digest: Sequence[int], constants_sigmas_cap,
           fri: dict, mul_by_x: bool, ref=V) -> bool:
    """plonk/verifier.rs verify: True when the proof is accepted.  Only the circuit description of `c` is read (gates, selectors,
    k_is), never its witness."""
    r, h = fri["rate_bits"], fri["cap_height"]
    n, n_log = c.n, c.n_log
    o = proof["openings"]
    ch = F.Challenger()
    ch.observe_elements([int(v) for v in circuit_digest])
    pi_hash = [int(v) for v in O.hash_no_pad([int(x) % P for x in public_inputs])]
    ch.observe_elements(pi_hash)
    ch.observe_cap(proof["wires_cap"])
    betas = [ch.get_challenge() for _ in range(NUM_CHALLENGES)]
    gammas = [ch.get_challenge() for _ in range(NUM_CHALLENGES)]
    ch.observe_cap(proof["plonk_zs_partial_products_cap"])
    alphas = [ch.get_challenge() for _ in range(NUM_CHALLENGES)]
    ch.observe_cap(proof["quotient_polys_cap"])
    zeta = ch.get_extension_challenge()
    # the vanishing polynomial at zeta from the openings (eval_vanishing_poly over the extension)
    E = lambda vals: [Ext2(*v) for v in vals]
    num_prods = perm_ref.num_partial_products(V.NUM_ROUTED, QUOTIENT_DEGREE_FACTOR)
    pp = E(o["partial_products"])
    pp_rows = [pp[i * num_prods:(i + 1) * num_prods] for i in range(NUM_CHALLENGES)]
    cv = copy.copy(c)
    cv.pi_hash = pi_hash
    z = Ext2(*zeta)
    terms = _vanishing_terms_at(ref)(cv, z, E(o["constants"]), E(o["plonk_sigmas"]), E(o["wires"]), E(o["plonk_zs"]), pp_rows,
                                     E(o["plonk_zs_next"]), betas, gammas, QUOTIENT_DEGREE_FACTOR)
    z_h = z ** n - 1
    zeta_n = z ** n
    qs = E(o["quotient_polys"])
    for i in range(NUM_CHALLENGES):
        chunks = qs[i * QUOTIENT_DEGREE_FACTOR:(i + 1) * QUOTIENT_DEGREE_FACTOR]
        acc = Ext2(0)
        for q in reversed(chunks):
            acc = acc * zeta_n + q
        if V.reduce_with_powers(terms, alphas[i]) != z_h * acc:
            return False
    openings = fri_openings(o)
    for vals in openings:
        ch.observe_extension_elements(vals)
    caps = [np.asarray(constants_sigmas_cap, dtype=np.uint64).reshape(-1, 4)] + [
        np.asarray(proof[k], dtype=np.uint64).reshape(-1, 4)
        for k in ("wires_cap", "plonk_zs_partial_products_cap", "quotient_polys_cap")]
    ks = [len(o["constants"]) + len(o["plonk_sigmas"]), len(o["wires"]), len(o["plonk_zs"]) + len(o["partial_products"]),
          len(o["quotient_polys"])]
    batches = instance(c, zeta, ks)
    return F.verify(proof["opening_proof"], caps, batches, openings, ch, n_log, r, h, fri["arities"], fri["pow_bits"],
                    fri["num_queries"], mul_by_x)
