"""TEST INFRASTRUCTURE: plonky2's interpolation gates on top of oracle/vanishing_ref.py.

Pure-Python restatement of
    plonky2 @ f99ed9c  plonky2/src/gates/interpolation.rs               HighDegreeInterpolationGate
                       plonky2/src/gates/low_degree_interpolation.rs    LowDegreeInterpolationGate
(wire layouts from memory like the rest of row N1b — parity unpinned; include/b200zkp.h states them), the gate that plonky2's
FRI verifier adds to every recursive circuit, one row per query step, to fold an arity-2^k coset.

oracle/vanishing_ref.py stays the restatement of the other thirteen gate kinds and of the vanishing polynomial.  This module
extends its gate functions (`gate_degree`, `gate_num_constraints`, `gate_constraints`, `gate_witness`) with the two kinds and
runs vanishing_ref's own `selector_groups`, `vanishing_terms_at`, `quotient_values` and `check_quotient_identity` with them:
the same code objects, looking up the gate functions here instead of there (`_with_interpolation`).  `recursion_circuit`
builds the gate set of a standard_recursion_config verifier circuit."""
from __future__ import annotations

import random
import types
from typing import List, Sequence

from oracle import vanishing_ref as V
from oracle.vanishing_ref import D, P, ext_add, ext_mul, ext_scale, ext_sub, root

INTERPOLATION_HIGH_DEGREE, INTERPOLATION_LOW_DEGREE = 14, 15          # ids shared with csrc/vanishing_kernels.cuh (13 is not assigned)
INTERPOLATION = (INTERPOLATION_HIGH_DEGREE, INTERPOLATION_LOW_DEGREE)
# the interpolation gate of a standard_recursion_config verifier: FRI folds with arity 16 > max_quotient_degree_factor 8
RECURSION_INTERPOLATION = (INTERPOLATION_LOW_DEGREE, 4)


# ---------------------------------------------------------------------------------------------------- the two gates
def interpolation_layout(kind: int, subgroup_bits: int):
    """gates/interpolation.rs, low_degree_interpolation.rs wire indices (m = 2^subgroup_bits points): shift 0, value(i) = ext at
    1 + D i, evaluation point 1 + D m, evaluation value 3 + D m, coeff(i) = ext at 5 + D m + D i; the first 5 + 2 m wires are
    routed.  LowDegree adds powers of the shift, shift_pow(i) for 2 <= i < m, and ext powers of the evaluation point,
    eval_pow(i) for 2 <= i < m, after the coefficients (shift_pow(1) is the shift, eval_pow(1) the evaluation point)."""
    m = 1 << subgroup_bits
    end_coeffs = 5 + 2 * D * m
    return dict(m=m, shift=0, value=lambda i: 1 + D * i, eval_point=1 + D * m, eval_value=3 + D * m,
                coeff=lambda i: 5 + D * m + D * i, end_coeffs=end_coeffs, routed=5 + 2 * m,
                shift_pow=lambda i: 0 if i == 1 else end_coeffs + i - 2,
                eval_pow=lambda i: 1 + D * m if i == 1 else end_coeffs + (m - 2) + D * (i - 2),
                num_wires=end_coeffs if kind == INTERPOLATION_HIGH_DEGREE else end_coeffs + (m - 2) * (1 + D))


def interpolation_constraints(kind: int, wires: Sequence[int], subgroup_bits: int, out: List[int]) -> None:
    """eval_unfiltered of HighDegreeInterpolationGate / LowDegreeInterpolationGate; appends to `out`"""
    L = interpolation_layout(kind, subgroup_bits)
    m = L["m"]
    ext = lambda j: (wires[j], wires[j + 1])
    g = root(subgroup_bits)
    coeffs = [ext(L["coeff"](i)) for i in range(m)]
    ev_point, ev_value = ext(L["eval_point"]), ext(L["eval_value"])
    if kind == INTERPOLATION_HIGH_DEGREE:
        shift = wires[L["shift"]]
        for i in range(m):
            x = shift * pow(g, i, P) % P
            computed = (0, 0)
            for c in reversed(coeffs):
                computed = ext_add(ext_scale(computed, x), c)
            out += list(ext_sub(ext(L["value"](i)), computed))
        computed = (0, 0)
        for c in reversed(coeffs):
            computed = ext_add(ext_mul(computed, ev_point), c)
        out += list(ext_sub(ev_value, computed))
        return
    # LowDegree: every power is a wire, constrained step by step, so each constraint has degree 2
    shift_pows = [1] + [wires[L["shift_pow"](i)] for i in range(1, m)]
    shift = shift_pows[1]
    for i in range(2, m):
        out.append((shift_pows[i - 1] * shift - shift_pows[i]) % P)
    altered = [ext_scale(c, sp) for c, sp in zip(coeffs, shift_pows)]      # altered(g^i) = interpolant(shift g^i)
    for i in range(m):
        x = pow(g, i, P)
        computed = (0, 0)
        for a in reversed(altered):
            computed = ext_add(ext_scale(computed, x), a)
        out += list(ext_sub(ext(L["value"](i)), computed))
    eval_pows = [None] + [ext(L["eval_pow"](i)) for i in range(1, m)]
    for i in range(2, m):
        out += list(ext_sub(ext_mul(eval_pows[i - 1], ev_point), eval_pows[i]))
    computed = coeffs[0]
    for i in range(1, m):
        computed = ext_add(computed, ext_mul(coeffs[i], eval_pows[i]))
    out += list(ext_sub(ev_value, computed))


def interpolation_witness(kind: int, subgroup_bits: int, w: List[int], rnd: random.Random, shift: int | None = None) -> None:
    """fill one interpolation row into `w`: a random shift (or `shift`), coefficients and evaluation point; the values on the
    coset shift <g>, the evaluation value and (LowDegree) the powers follow from them"""
    L = interpolation_layout(kind, subgroup_bits)
    m = L["m"]
    g = root(subgroup_bits)
    shift = rnd.randrange(1, P) if shift is None else shift
    coeffs = [(rnd.randrange(P), rnd.randrange(P)) for _ in range(m)]
    ev_point = (rnd.randrange(P), rnd.randrange(P))

    def put(j, e):
        w[j], w[j + 1] = e

    def interpolant(x):
        acc = (0, 0)
        for c in reversed(coeffs):
            acc = ext_add(ext_mul(acc, x), c)
        return acc

    w[L["shift"]] = shift
    for i, c in enumerate(coeffs):
        put(L["coeff"](i), c)
    for i in range(m):
        put(L["value"](i), interpolant((shift * pow(g, i, P) % P, 0)))
    put(L["eval_point"], ev_point)
    put(L["eval_value"], interpolant(ev_point))
    if kind == INTERPOLATION_LOW_DEGREE:
        sp, ep = shift, ev_point
        for i in range(2, m):
            sp, ep = sp * shift % P, ext_mul(ep, ev_point)
            w[L["shift_pow"](i)] = sp
            put(L["eval_pow"](i), ep)


# ---------------------------------------------------------------------------------------------------- the gate functions, extended
def gate_degree(kind: int, params=()) -> int:
    """Gate::degree()"""
    if kind == INTERPOLATION_HIGH_DEGREE:
        return 1 << params[0]
    if kind == INTERPOLATION_LOW_DEGREE:
        return 2
    return V.gate_degree(kind, params)


def gate_num_constraints(kind: int, params=()) -> int:
    """Gate::num_constraints()"""
    if kind == INTERPOLATION_HIGH_DEGREE:
        return D * ((1 << params[0]) + 1)
    if kind == INTERPOLATION_LOW_DEGREE:
        return 5 * (1 << params[0]) - 4
    return V.gate_num_constraints(kind, params)


def gate_constraints(kind: int, wires: Sequence[int], consts: Sequence[int], pi_hash: Sequence[int], params=()) -> List[int]:
    """eval_unfiltered of one gate type at one point"""
    if kind in INTERPOLATION:
        out: List[int] = []
        interpolation_constraints(kind, wires, params[0], out)
        return out
    return V.gate_constraints(kind, wires, consts, pi_hash, params)


def gate_witness(kind: int, rnd: random.Random, consts: Sequence[int], params=()) -> List[int]:
    """135 wires of one row of `kind` whose constraints vanish"""
    if kind in INTERPOLATION:
        w = [rnd.randrange(P) for _ in range(V.NUM_WIRES)]
        interpolation_witness(kind, params[0], w, rnd)
        return w
    return V.gate_witness(kind, rnd, consts, params)


# ---------------------------------------------------------------------------------------------------- vanishing_ref's code, these gates
_NAMESPACE = dict(vars(V), gate_degree=gate_degree, gate_num_constraints=gate_num_constraints, gate_constraints=gate_constraints)


def _with_interpolation(fn):
    """vanishing_ref's function `fn` (its code object unchanged) resolving module names in a copy of vanishing_ref's namespace
    in which the gate functions are the ones above"""
    g = types.FunctionType(fn.__code__, _NAMESPACE, fn.__name__, fn.__defaults__, fn.__closure__)
    _NAMESPACE[fn.__name__] = g
    return g


selector_groups = _with_interpolation(V.selector_groups)
vanishing_terms_at = _with_interpolation(V.vanishing_terms_at)
quotient_values = _with_interpolation(V.quotient_values)
check_quotient_identity = _with_interpolation(V.check_quotient_identity)


# ---------------------------------------------------------------------------------------------------- a recursion-shaped circuit
def recursion_circuit(n_log: int, seed: int = 0, n_poseidon: int | None = None, interpolation=RECURSION_INTERPOLATION) -> V.Circuit:
    """The gate set of a verifier circuit: vanishing_ref's extended circuit (13 gate kinds) plus one row of the interpolation
    gate `interpolation` = (kind, subgroup_bits) on a no-op row (default: what standard_recursion_config's arity 16
    instantiates).  The row's coset shift is copied from a Poseidon output: its cell joins that output's copy cycle, so the
    permutation argument covers a routed interpolation wire too.  Gates stay sorted by degree; the selector polynomials are
    recomputed for the longer list."""
    kind, bits = interpolation
    c = V.Circuit(n_log, seed=seed, n_poseidon=n_poseidon, extended=True)
    rnd = random.Random(seed + 1000)
    at = sum(1 for g, pr in zip(c.gates, c.gate_params) if gate_degree(g, pr) <= gate_degree(kind, (bits,)))
    c.gates.insert(at, kind)
    c.gate_params.insert(at, (bits,))
    noop = c.gates.index(V.NOOP)
    c.row_gate = [gi + 1 if gi >= at else gi for gi in c.row_gate]
    row = max(r for r in range(c.n) if c.row_gate[r] == noop)       # every cell of a no-op row is its own copy cycle
    pos_rows = [r for r in range(c.n) if c.row_gate[r] == c.gates.index(V.POSEIDON)]
    src, t = rnd.choice(pos_rows), rnd.randrange(V.WIDTH)
    w = [c.wires[j][row] for j in range(V.NUM_WIRES)]
    interpolation_witness(kind, bits, w, rnd, shift=c.wires[V.W_OUT + t][src])
    for j in range(V.NUM_WIRES):
        c.wires[j][row] = w[j]
    c.row_gate[row] = at
    # splice the shift cell (wire 0, row) into the cycle of (W_OUT + t, src), right after it
    cell_id = c.k_is[0] * pow(root(n_log), row, P) % P
    c.sigmas[0][row] = c.sigmas[V.W_OUT + t][src]
    c.sigmas[V.W_OUT + t][src] = cell_id
    c.selector_indices, c.groups = selector_groups(list(zip(c.gates, c.gate_params)), c.max_degree)
    c.num_selectors = len(c.groups)
    c.constants = [[c.row_gate[r] if grp[0] <= c.row_gate[r] < grp[1] else V.UNUSED_SELECTOR for r in range(c.n)] for grp in c.groups]
    c.constants += c.gate_consts
    return c
