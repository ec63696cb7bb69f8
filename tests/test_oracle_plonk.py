"""The restated plonky2 prove() / verify() (tests/plonk_ref.py) on the CPU: vanishing_ref's gate code over the quadratic
extension agrees with the base field on embedded inputs, honest proofs are accepted, and every kind of tampering is refused."""
import copy
import random

import numpy as np
import pytest

import interpolation_ref as I
import plonk_ref as R
from oracle import vanishing_ref as V

P = 0xFFFFFFFF00000001
PIS = [5, 6, 7, 2**64 - 1]


def _gate_set():
    """all 15 gate kinds with the parameters the circuits use"""
    gates = dict(zip(I.recursion_circuit(5).gates, I.recursion_circuit(5).gate_params))
    gates[I.INTERPOLATION_HIGH_DEGREE] = (3,)
    return gates


def test_gate_constraints_over_the_extension_match_the_base_field():
    gates = _gate_set()
    assert len(gates) == 15
    rnd = random.Random(3)
    for kind, params in gates.items():
        for _ in range(2):
            wires = [rnd.randrange(P) for _ in range(V.NUM_WIRES)]
            consts = [rnd.randrange(P) for _ in range(V.NUM_GATE_CONSTANTS)]
            pi = [rnd.randrange(P) for _ in range(4)]
            base = I.gate_constraints(kind, wires, consts, pi, params)
            ext = I.gate_constraints(kind, [R.Ext2(w) for w in wires], [R.Ext2(c) for c in consts], pi, params)
            assert len(base) == I.gate_num_constraints(kind, params) == len(ext), kind
            assert [R.Ext2(v) for v in base] == [R.Ext2._of(v) for v in ext], kind


@pytest.mark.parametrize("interpolation", [(I.INTERPOLATION_LOW_DEGREE, 4), (I.INTERPOLATION_HIGH_DEGREE, 3)])
def test_vanishing_terms_over_the_extension_match_the_base_field(interpolation):
    """the whole of vanishing_terms_at, L_1's inversion included, on a base-field point embedded in the extension"""
    c = I.recursion_circuit(5, seed=4, interpolation=interpolation)
    rnd = random.Random(5)
    x = rnd.randrange(2, P)
    cols = lambda k: [rnd.randrange(P) for _ in range(k)]
    nc = c.num_selectors + V.NUM_GATE_CONSTANTS
    consts, sigmas, wires, zs, nzs = cols(nc), cols(V.NUM_ROUTED), cols(V.NUM_WIRES), cols(2), cols(2)
    pp = [cols(9), cols(9)]
    betas, gammas = cols(2), cols(2)
    base = I.vanishing_terms_at(c, x, consts, sigmas, wires, zs, pp, nzs, betas, gammas, 8)
    E = lambda v: [R.Ext2(a) for a in v]
    ext = R._vanishing_terms_at(I)(c, R.Ext2(x), E(consts), E(sigmas), E(wires), E(zs), [E(p) for p in pp], E(nzs), betas, gammas, 8)
    assert [R.Ext2(v) for v in base] == ext
    assert R.Ext2(12345, 678).inverse() * R.Ext2(12345, 678) == R.Ext2(1)


CASES = {
    "extended": lambda: (V.Circuit(5, seed=11, extended=True), V),
    "low_degree_4": lambda: (I.recursion_circuit(5, seed=12), I),
    "high_degree_3": lambda: (I.recursion_circuit(5, seed=13, interpolation=(I.INTERPOLATION_HIGH_DEGREE, 3)), I),
}


def _proved(name):
    c, ref = CASES[name]()
    c = R.with_public_inputs(c, PIS)
    fri = R.fri_args(c.n_log, pow_bits=8)
    proof = R.prove(c, PIS, fri, True, ref=ref)
    check = lambda p, pis=PIS: R.verify(p, pis, c, proof["circuit_digest"], proof["constants_sigmas_cap"], fri, True, ref=ref)
    return c, ref, fri, proof, check


@pytest.mark.parametrize("name", sorted(CASES))
def test_reference_proof_is_accepted(name):
    _, _, _, proof, check = _proved(name)
    assert check(proof)


def _bump(e):
    return ((e[0] + 1) % P, e[1])


def test_tampered_proofs_are_rejected():
    c, ref, fri, proof, check = _proved("low_degree_4")
    assert check(proof)

    def tampered(edit):
        p = copy.deepcopy(proof)
        edit(p)
        return p
    for field, i in (("wires", 7), ("quotient_polys", 3), ("plonk_zs_next", 1)):
        def edit(p, field=field, i=i):
            p["openings"][field][i] = _bump(p["openings"][field][i])
        assert not check(tampered(edit)), field

    def cap(p):
        p["wires_cap"] = p["wires_cap"].copy()
        p["wires_cap"][0, 0] = (int(p["wires_cap"][0, 0]) + 1) % P
    assert not check(tampered(cap))
    assert not check(proof, PIS[:-1] + [PIS[-1] - 1])

    def pow_witness(p):
        p["opening_proof"]["pow_witness"] += 1
    # (with 8 bits a changed witness can still qualify; the next candidates are tried until one does not)
    p = copy.deepcopy(proof)
    for _ in range(8):
        pow_witness(p)
        if not check(p):
            break
    else:
        pytest.fail("no changed proof-of-work witness was rejected")

    def leaf(p):
        row, sib = p["opening_proof"]["rounds"][0]["initial"][1]
        row = row.copy()
        row[3] = (int(row[3]) + 1) % P
        p["opening_proof"]["rounds"][0]["initial"][1] = (row, sib)
    assert not check(tampered(leaf))


@pytest.mark.parametrize("name", ["extended", "low_degree_4"])
def test_proof_of_a_changed_witness_is_rejected(name):
    c, ref = CASES[name]()
    c = R.with_public_inputs(c, PIS)
    fri = R.fri_args(c.n_log, pow_bits=8)
    wires = np.array(c.wires, dtype=np.uint64)
    wires[100][3] = (int(wires[100][3]) + 1) % P          # an unrouted wire of a Poseidon row: only a gate constraint sees it
    proof = R.prove(c, PIS, fri, True, ref=ref, wires=wires)
    assert not R.verify(proof, PIS, c, proof["circuit_digest"], proof["constants_sigmas_cap"], fri, True, ref=ref)
