"""plonky2_u32's gates in tests/u32_ref.py (tests/interpolation_ref.py extended with the five gates): generated rows satisfy the
constraints and compute the integer semantics, the counts follow Gate::num_constraints, each constraint family catches its own
corruption, and the quotient identity closes for the ecdsa gate set.  CPU only."""
import random

import numpy as np
import pytest

import u32_ref as U
from oracle import perm_ref as PR
from oracle import vanishing_ref as V
from test_oracle_interpolation import coset_ifft

P = V.P
MAX32 = (1 << 32) - 1
# every gate over its parameter range (135 wires); U32AddMany over all arities with the ops its arity allows
CASES = ([(U.U32_ARITHMETIC, (ops,)) for ops in (1, 2, 3)] +
         [(U.U32_ADD_MANY, (a, ops)) for a in range(1, 17) for ops in sorted({1, 135 // (a + 21)})] +
         [(U.U32_SUBTRACTION, (ops,)) for ops in range(1, 7)] +
         [(U.U32_RANGE_CHECK, (nl,)) for nl in range(1, 8)] +
         [(U.COMPARISON, (nb, nc)) for nb in (1, 2, 3, 7, 8, 20, 32, 33, 63) for nc in range(1, nb + 1)
          if U.chunk_bits(nb, nc) <= 3 and U.num_wires(U.COMPARISON, (nb, nc)) <= 135])


def constraints(kind, params, w):
    return U.gate_constraints(kind, w, [0, 0], [0] * 4, params)


def row(kind, params, seed=0, inputs=None):
    rnd = random.Random(seed)
    w = [rnd.randrange(P) for _ in range(V.NUM_WIRES)]
    U.u32_witness(kind, params, w, rnd, inputs=inputs)
    return w


@pytest.mark.parametrize("kind,params", CASES)
def test_witness_satisfies_constraints(kind, params):
    want = {U.U32_ARITHMETIC: lambda p: 36 * p[0], U.U32_ADD_MANY: lambda p: 21 * p[1], U.U32_SUBTRACTION: lambda p: 19 * p[0],
            U.U32_RANGE_CHECK: lambda p: 17 * p[0], U.COMPARISON: lambda p: 6 + 5 * p[1] + U.chunk_bits(*p)}[kind](params)
    assert U.gate_num_constraints(kind, params) == want
    assert U.num_wires(kind, params) <= V.NUM_WIRES
    assert U.gate_degree(kind, params) == (1 << U.chunk_bits(*params) if kind == U.COMPARISON else 4)
    for seed in range(4):
        w = U.gate_witness(kind, random.Random(seed), [0, 0], params)
        out = constraints(kind, params, w)
        assert len(out) == want and not any(out)


def test_config_params():
    assert U.config_params(U.U32_ARITHMETIC) == (3,) and U.config_params(U.U32_SUBTRACTION) == (6,)
    assert U.config_params(U.U32_ADD_MANY, 16) == (16, 3) and U.config_params(U.U32_ADD_MANY, 3) == (3, 5)
    assert U.num_wires(U.COMPARISON, (32, 16)) == 5 + 80 + 2


def test_arithmetic_semantics():
    L = U.arithmetic_layout(3)
    cases = [(0, 0, 0), (MAX32, MAX32, MAX32), (MAX32, 1, 0), (1 << 31, 2, 1)]
    w = row(U.U32_ARITHMETIC, (3,), inputs=cases[:3])
    w4 = row(U.U32_ARITHMETIC, (3,), inputs=cases[3:] * 3)
    for ww, cs in ((w, cases[:3]), (w4, cases[3:] * 3)):
        assert not any(constraints(U.U32_ARITHMETIC, (3,), ww))
        for i, (m0, m1, ad) in enumerate(cs):
            assert ww[L["lo"](i)] + (ww[L["hi"](i)] << 32) == m0 * m1 + ad
            assert ww[L["lo"](i)] <= MAX32 and ww[L["hi"](i)] <= MAX32
    # the largest value: hi = 2^32 - 1, lo = 0, and the inverse is 0 where the generator puts 0
    assert (w[L["hi"](1)], w[L["lo"](1)], w[L["inverse"](1)]) == (MAX32, 0, 0)


def test_add_many_semantics():
    p = (16, 3)
    L = U.add_many_layout(*p)
    inputs = [([MAX32] * 16, 15), ([0] * 16, 0), (list(range(16)), 3)]
    w = row(U.U32_ADD_MANY, p, inputs=inputs)
    assert not any(constraints(U.U32_ADD_MANY, p, w))
    for i, (ads, cin) in enumerate(inputs):
        assert w[L["result"](i)] + (w[L["carry_out"](i)] << 32) == sum(ads) + cin
    assert w[L["carry_out"](0)] == 15 and w[L["result"](0)] == (16 * MAX32 + 15) % (1 << 32)


def test_subtraction_semantics():
    L = U.subtraction_layout(6)
    inputs = [(0, 0, 0), (0, 0, 1), (0, MAX32, 1), (MAX32, 0, 0), (5, 5, 0), (5, 6, 0)]
    w = row(U.U32_SUBTRACTION, (6,), inputs=inputs)
    assert not any(constraints(U.U32_SUBTRACTION, (6,), w))
    for i, (x, y, b) in enumerate(inputs):
        assert w[L["result"](i)] == (x - y - b) % (1 << 32)
        assert w[L["borrow_out"](i)] == int(x - y - b < 0)


def test_range_check_semantics():
    L = U.range_check_layout(3)
    w = row(U.U32_RANGE_CHECK, (3,), inputs=[0, MAX32, 0x12345678])
    assert not any(constraints(U.U32_RANGE_CHECK, (3,), w))
    assert [w[L["limb"](1, j)] for j in range(16)] == [3] * 16


@pytest.mark.parametrize("nb,nc", [(32, 16), (63, 21), (8, 4), (1, 1)])
def test_comparison_semantics(nb, nc):
    L = U.comparison_layout(nb, nc)
    top = (1 << nb) - 1
    pairs = [(0, 0), (top, top), (0, top), (top, 0), (5 % (top + 1), 5 % (top + 1))]
    if nb > 1:
        pairs += [(top - 1, top), (top, top - 1), (2, 3), (3, 2)]          # differ only in the lowest chunk
    for first, second in pairs:
        w = row(U.COMPARISON, (nb, nc), inputs=(first, second))
        assert not any(constraints(U.COMPARISON, (nb, nc), w)), (first, second)
        assert w[L["result"]] == int(first <= second)


# ---------------------------------------------------------------------------------------------------- corruption
def _bump_limb(w, limb, n_limbs, base):
    """limb j += base and limb j + 1 -= 1 (which was >= 1): the combined value is unchanged, limb j is out of range; returns j"""
    for j in range(n_limbs - 1):
        if w[limb(j + 1)] >= 1:
            w[limb(j)] += base
            w[limb(j + 1)] -= 1
            return j
    raise AssertionError("no limb to borrow from")


def test_out_of_range_limb_is_caught_by_its_range_constraint():
    # U32Arithmetic op 0 (constraints: canonicity, word, limbs 31..0, low, high)
    w = row(U.U32_ARITHMETIC, (3,), inputs=[(0x12345678, 0x9ABCDEF0, 77)] * 3)
    j = _bump_limb(w, lambda j: U.arithmetic_layout(3)["limb"](0, j), 32, 4)
    out = constraints(U.U32_ARITHMETIC, (3,), w)
    assert [t for t, v in enumerate(out) if v] == [2 + (31 - j)]
    # U32AddMany op 1 (word, limbs 17..0, result, carry)
    p = (16, 3)
    w = row(U.U32_ADD_MANY, p, inputs=[([MAX32] * 16, 15)] * 3)
    j = _bump_limb(w, lambda j: U.add_many_layout(*p)["limb"](1, j), 18, 4)
    assert [t for t, v in enumerate(constraints(U.U32_ADD_MANY, p, w)) if v] == [21 + 1 + (17 - j)]
    # U32Subtraction op 2 (word, limbs 15..0, combined, borrow bit)
    w = row(U.U32_SUBTRACTION, (6,), inputs=[(0x80000000, 1, 0)] * 6)
    j = _bump_limb(w, lambda j: U.subtraction_layout(6)["limb"](2, j), 16, 4)
    assert [t for t, v in enumerate(constraints(U.U32_SUBTRACTION, (6,), w)) if v] == [2 * 19 + 1 + (15 - j)]
    # U32RangeCheck input 1 (combined, limbs 0..15)
    w = row(U.U32_RANGE_CHECK, (2,), inputs=[7, 0x40000000])
    j = _bump_limb(w, lambda j: U.range_check_layout(2)["limb"](1, j), 16, 4)
    assert [t for t, v in enumerate(constraints(U.U32_RANGE_CHECK, (2,), w)) if v] == [17 + 1 + j]
    # Comparison: a first chunk of 2^cb (first chunk c is constraint 2 + 5c)
    L = U.comparison_layout(32, 16)
    w = row(U.COMPARISON, (32, 16), inputs=(0x40000000, 0x40000000))
    j = _bump_limb(w, L["first_chunk"], 16, 4)
    bad = [t for t, v in enumerate(constraints(U.COMPARISON, (32, 16), w)) if v]
    assert 2 + 5 * j in bad and 0 not in bad


def test_non_canonical_output_is_caught_by_the_canonicity_check():
    """m0 m1 + addend = v < 2^32 - 1 written as v + p = (2^32 - 1) 2^32 + (v + 1): word and limbs hold, canonicity does not"""
    L = U.arithmetic_layout(3)
    w = row(U.U32_ARITHMETIC, (3,), inputs=[(3, 5, 7)] * 3)
    v = 3 * 5 + 7
    alt = v + P
    w[L["hi"](0)], w[L["lo"](0)] = alt >> 32, alt % (1 << 32)
    assert w[L["hi"](0)] == MAX32 and w[L["lo"](0)] != 0
    for j, l in enumerate(U._limbs(alt, 32)):
        w[L["limb"](0, j)] = l
    for inverse in (0, 1, 12345):
        w[L["inverse"](0)] = inverse
        assert [t for t, x in enumerate(constraints(U.U32_ARITHMETIC, (3,), w)) if x] == [0]


def test_borrow_of_two_is_caught_by_the_bit_constraint():
    L = U.subtraction_layout(6)
    w = row(U.U32_SUBTRACTION, (6,), inputs=[(9, 4, 0)] * 6)
    w[L["borrow_out"](0)] = 2
    w[L["result"](0)] = (9 - 4 + 2 * (1 << 32)) % P          # the word equation still holds
    out = constraints(U.U32_SUBTRACTION, (6,), w)
    assert out[0] == 0 and out[18] != 0


def test_wrong_chunks_equal_and_flipped_result_are_caught():
    nb, nc = 32, 16
    L = U.comparison_layout(nb, nc)
    w = row(U.COMPARISON, (nb, nc), inputs=(0x1234, 0x1235))
    out_at = lambda ww: [t for t, v in enumerate(constraints(U.COMPARISON, (nb, nc), ww)) if v]
    for c, eq in ((0, 1), (5, 0)):                            # chunk 0 differs, chunk 5 is equal
        assert w[L["eq"](c)] == 1 - eq
        bad = list(w)
        bad[L["eq"](c)] = eq
        assert set(out_at(bad)) & {2 + 5 * c + 2, 2 + 5 * c + 3}
    bad = list(w)
    bad[L["result"]] = 1 - bad[L["result"]]
    assert out_at(bad) == [U.gate_num_constraints(U.COMPARISON, (nb, nc)) - 1]


# ---------------------------------------------------------------------------------------------------- circuits
def test_ecdsa_gate_set():
    c = U.ecdsa_circuit(5, seed=3)
    assert len(c.gates) == 20 <= 32 and c.gates.count(U.U32_ADD_MANY) == 2
    assert set(c.gates) == set(U.I.recursion_circuit(5, seed=3).gates) | set(U.U32_GATES)
    degs = [U.gate_degree(g, p) for g, p in zip(c.gates, c.gate_params)]
    assert degs == sorted(degs)
    for r in range(c.n):
        gi = c.row_gate[r]
        w = [c.wires[j][r] for j in range(V.NUM_WIRES)]
        assert not any(U.gate_constraints(c.gates[gi], w, [c.gate_consts[i][r] for i in range(2)], c.pi_hash, c.gate_params[gi])), r
    # the chained u32 wires are routed: their sigmas point at other cells
    cell = lambda j, r: c.k_is[j] * pow(V.root(5), r, P) % P
    ar, am, _, sub, rc, cmp_ = c.u32_rows
    for j, r in ((3, ar), (0, am), (4, am), (0, sub), (3, sub), (0, cmp_), (1, cmp_), (1, rc)):
        assert c.sigmas[j][r] != cell(j, r), (j, r)


def test_timing_tool_ecdsa_set():
    """tools/quotient_timing.py times the same gate list, selectors and groups as ecdsa_circuit describes"""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("quotient_timing", os.path.join(V.ROOT, "tools", "quotient_timing.py"))
    T = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(T)
    gates, num_selectors = T.gate_sets()["ecdsa"]
    c = U.ecdsa_circuit(5, seed=3)
    assert num_selectors == c.num_selectors
    assert gates == [(g, c.selector_indices[i], c.groups[c.selector_indices[i]], c.gate_params[i]) for i, g in enumerate(c.gates)]


def _instance(oracle, c, seed):
    rnd = random.Random(seed)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    zs_pp = PR.partial_products_and_zs([c.wires[j] for j in range(V.NUM_ROUTED)], c.sigmas, c.k_is, betas, gammas, 8)
    values = dict(cs=c.constants + c.sigmas, wires=c.wires, zpp=zs_pp)
    coeffs = {k: [oracle.ifft(np.array(col, np.uint64)) for col in cols] for k, cols in values.items()}
    ldes = {k: [oracle.coset_lde(col, 3) for col in cols] for k, cols in coeffs.items()}
    return betas, gammas, alphas, coeffs, ldes


def test_quotient_identity_for_the_ecdsa_circuit(oracle):
    c = U.ecdsa_circuit(5, seed=21)
    betas, gammas, alphas, coeffs, ldes = _instance(oracle, c, 22)
    q = U.quotient_values(c, ldes["cs"], ldes["wires"], ldes["zpp"], betas, gammas, alphas, 8, 3, 3)
    qc = [coset_ifft(oracle, col) for col in q]
    for zeta in (987654321, 31337):
        assert U.check_quotient_identity(c, coeffs["cs"], coeffs["wires"], coeffs["zpp"], qc, betas, gammas, alphas, 8, zeta)
    # one changed u32 wire: a U32Subtraction limb (unrouted), then the Comparison's chunks_equal
    sub_row, cmp_row = c.u32_rows[3], c.u32_rows[5]
    for j, r in ((U.subtraction_layout(6)["limb"](1, 3), sub_row), (U.comparison_layout(32, 16)["eq"](2), cmp_row)):
        bad = [list(col) for col in c.wires]
        bad[j][r] = (bad[j][r] + 1) % P
        w_coeffs = [oracle.ifft(np.array(col, np.uint64)) for col in bad]
        w_lde = [oracle.coset_lde(col, 3) for col in w_coeffs]
        qb = U.quotient_values(c, ldes["cs"], w_lde, ldes["zpp"], betas, gammas, alphas, 8, 3, 3)
        qbc = [coset_ifft(oracle, col) for col in qb]
        assert not U.check_quotient_identity(c, coeffs["cs"], w_coeffs, coeffs["zpp"], qbc, betas, gammas, alphas, 8, 12345), j
