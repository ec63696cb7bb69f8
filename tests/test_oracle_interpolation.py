"""HighDegreeInterpolationGate and LowDegreeInterpolationGate in tests/interpolation_ref.py (oracle/vanishing_ref.py extended
with the two gates): generated rows satisfy the constraints, the counts follow Gate::num_constraints, changed wires break them,
the evaluation value is what one FRI query step's fold computes (oracle/fri_ref.py), and the quotient identity closes for
circuits that hold the gates.  CPU only."""
import random

import numpy as np
import pytest

import interpolation_ref as I
from oracle import fri_ref as F
from oracle import perm_ref as PR
from oracle import vanishing_ref as V

P = V.P
HIGH, LOW = I.INTERPOLATION_HIGH_DEGREE, I.INTERPOLATION_LOW_DEGREE
CASES = [(HIGH, b) for b in range(1, 6)] + [(LOW, b) for b in range(1, 5)]


def build_instance(oracle, n_log, seed, interpolation, rate_bits=3):
    c = I.recursion_circuit(n_log, seed=seed, interpolation=interpolation)
    rnd = random.Random(seed + 1)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    zs_pp = PR.partial_products_and_zs([c.wires[j] for j in range(V.NUM_ROUTED)], c.sigmas, c.k_is, betas, gammas, 8)
    values = dict(cs=c.constants + c.sigmas, wires=c.wires, zpp=zs_pp)
    coeffs = {k: [oracle.ifft(np.array(col, np.uint64)) for col in cols] for k, cols in values.items()}
    ldes = {k: [oracle.coset_lde(col, rate_bits) for col in cols] for k, cols in coeffs.items()}
    return c, betas, gammas, alphas, coeffs, ldes


def coset_ifft(oracle, vals):
    co = oracle.ifft(np.array(vals, np.uint64))
    inv7 = pow(7, P - 2, P)
    s, out = 1, []
    for a in co:
        out.append(int(a) * s % P)
        s = s * inv7 % P
    return out


def quotient_closes(oracle, c, wires, betas, gammas, alphas, coeffs, ldes, zeta):
    """quotient values from `wires` (the circuit's other polynomials unchanged), interpolated, checked at zeta"""
    w_coeffs = [oracle.ifft(np.array(col, np.uint64)) for col in wires]
    w_lde = [oracle.coset_lde(col, 3) for col in w_coeffs]
    q = I.quotient_values(c, ldes["cs"], w_lde, ldes["zpp"], betas, gammas, alphas, 8, 3, 3)
    qc = [coset_ifft(oracle, col) for col in q]
    return I.check_quotient_identity(c, coeffs["cs"], w_coeffs, coeffs["zpp"], qc, betas, gammas, alphas, 8, zeta)


@pytest.mark.parametrize("kind,bits", CASES)
def test_interpolation_witness_satisfies_constraints(kind, bits):
    rnd = random.Random(100 * kind + bits)
    m = 1 << bits
    L = I.interpolation_layout(kind, bits)
    n_constraints = 2 * (m + 1) if kind == HIGH else 5 * m - 4
    assert I.gate_num_constraints(kind, (bits,)) == n_constraints
    assert L["num_wires"] == (5 + 4 * m if kind == HIGH else 7 * m - 1) <= V.NUM_WIRES
    assert I.gate_degree(kind, (bits,)) == (m if kind == HIGH else 2)
    for _ in range(3):
        w = I.gate_witness(kind, rnd, [0, 0], (bits,))
        out = I.gate_constraints(kind, w, [0, 0], [0] * 4, (bits,))
        assert len(out) == n_constraints and not any(out)
        wires_to_break = [L["coeff"](rnd.randrange(m)), L["coeff"](m - 1) + 1, L["value"](rnd.randrange(m)), L["eval_value"] + 1,
                          L["shift"]]
        if kind == LOW and m > 2:
            wires_to_break += [L["shift_pow"](rnd.randrange(2, m)), L["eval_pow"](rnd.randrange(2, m)) + 1]
        for j in wires_to_break:
            bad = list(w)
            bad[j] = (bad[j] + 1) % P
            assert any(I.gate_constraints(kind, bad, [0, 0], [0] * 4, (bits,))), j


def test_low_degree_uses_the_power_wires():
    """the same coefficients, shift and evaluation point with wrong power wires: HighDegree (which has none) is satisfied, the
    LowDegree constraint on the powers is not — the gate must read the wires, not recompute the powers"""
    rnd = random.Random(4)
    w = I.gate_witness(LOW, rnd, [0, 0], (4,))
    L = I.interpolation_layout(LOW, 4)
    w[L["shift_pow"](5)] = (w[L["shift_pow"](5)] + 3) % P
    out = I.gate_constraints(LOW, w, [0, 0], [0] * 4, (4,))
    assert out[5 - 2] and out[6 - 2]                           # shift^5 - shift^4 shift and shift^6 - shift^5 shift
    assert not any(out[14 + 32:])                              # the evaluation-point powers and value do not read it
    high = list(w[:I.interpolation_layout(HIGH, 4)["num_wires"]]) + [0] * 66
    assert not any(I.gate_constraints(HIGH, high, [0, 0], [0] * 4, (4,)))


@pytest.mark.parametrize("kind,bits", CASES)
def test_evaluation_value_is_the_fri_fold(kind, bits):
    """one FRI query step of arity 2^bits: the coset holding x, its evaluations stored bit-reversed, folded at beta.  A gate row
    with that coset's start as shift, the evaluations as values and beta as evaluation point has compute_evaluation's value
    (the fold the verifier of GPU proofs already checks) as its evaluation value"""
    rnd = random.Random(7 + bits)
    m = 1 << bits
    L = I.interpolation_layout(kind, bits)
    g = F.root(bits)
    for _ in range(3):
        x = 7 * pow(F.root(bits + 6), rnd.randrange(1 << (bits + 6)), P) % P
        idx = rnd.randrange(m)
        coset_start = x * pow(g, m - F.bitrev(idx, bits), P) % P
        w = [rnd.randrange(P) for _ in range(V.NUM_WIRES)]
        I.interpolation_witness(kind, bits, w, rnd, shift=coset_start)
        assert not any(I.gate_constraints(kind, w, [0, 0], [0] * 4, (bits,)))
        ext = lambda j: (w[j], w[j + 1])
        values = [ext(L["value"](i)) for i in range(m)]
        beta = ext(L["eval_point"])
        evals = F.reverse_index_bits(values)                   # as a FRI layer's leaf holds them
        assert values[F.bitrev(idx, bits)] == evals[idx]       # x is the idx-th leaf entry
        assert F.compute_evaluation(x, idx, bits, evals, beta) == ext(L["eval_value"])
        pts = [((coset_start * pow(g, i, P) % P, 0), values[i]) for i in range(m)]
        assert F.interpolate_at(pts, beta) == ext(L["eval_value"])


def test_recursion_gate_set():
    c = I.recursion_circuit(5, seed=3)
    assert len(c.gates) == 14 <= 16 and c.gates.count(LOW) == 1 and c.gate_params[c.gates.index(LOW)] == (4,)
    assert [I.gate_degree(g, p) for g, p in zip(c.gates, c.gate_params)] == sorted(I.gate_degree(g, p) for g, p in zip(c.gates, c.gate_params))
    assert set(c.gates) == set(V.Circuit(5, seed=3, extended=True).gates) | {LOW}
    # the interpolation row's shift is routed: its sigma points at a Poseidon output cell, not at itself
    row = c.row_gate.index(c.gates.index(LOW))
    assert c.sigmas[0][row] != c.k_is[0] * pow(V.root(5), row, P) % P
    # the gate with the most constraints still sizes the gate terms
    h = I.recursion_circuit(5, seed=1, interpolation=(HIGH, 3))
    assert h.gates[-1] == HIGH and I.gate_num_constraints(HIGH, (3,)) == 18


def test_timing_tool_recursion_set():
    """tools/quotient_timing.py times the same gate list, selectors and groups as recursion_circuit describes"""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("quotient_timing", os.path.join(V.ROOT, "tools", "quotient_timing.py"))
    T = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(T)
    gates, num_selectors = T.gate_sets()["recursion"]
    c = I.recursion_circuit(5, seed=3)
    assert num_selectors == c.num_selectors
    assert gates == [(g, c.selector_indices[i], c.groups[c.selector_indices[i]], c.gate_params[i]) for i, g in enumerate(c.gates)]


@pytest.mark.parametrize("interpolation", [(LOW, 4), (HIGH, 3)])
def test_quotient_identity_with_interpolation_rows(oracle, interpolation):
    kind, bits = interpolation
    c, betas, gammas, alphas, coeffs, ldes = build_instance(oracle, 5, 21, interpolation)
    assert kind in c.gates
    q = I.quotient_values(c, ldes["cs"], ldes["wires"], ldes["zpp"], betas, gammas, alphas, 8, 3, 3)
    qc = [coset_ifft(oracle, col) for col in q]
    for zeta in (987654321, 31337):
        assert I.check_quotient_identity(c, coeffs["cs"], coeffs["wires"], coeffs["zpp"], qc, betas, gammas, alphas, 8, zeta)
    row = c.row_gate.index(c.gates.index(kind))
    L = I.interpolation_layout(kind, bits)
    broken = [L["coeff"](3) + 1]
    if kind == LOW:
        broken += [L["shift_pow"](9), L["eval_pow"](7)]
    for j in broken:
        bad = [list(col) for col in c.wires]
        bad[j][row] = (bad[j][row] + 1) % P
        assert not quotient_closes(oracle, c, bad, betas, gammas, alphas, coeffs, ldes, 12345), j
