"""TEST INFRASTRUCTURE: plonky2_u32's gates on top of tests/interpolation_ref.py.

Pure-Python restatement of the gates plonky2_u32 (the crate plonky2_ecdsa builds on, at the date of plonky2 @ f99ed9c) adds
to a circuit,
    gates/arithmetic_u32.rs    U32ArithmeticGate     lo + 2^32 hi = m0 m1 + addend
    gates/add_many_u32.rs      U32AddManyGate        result + 2^32 carry_out = sum of addends + carry_in
    gates/subtraction_u32.rs   U32SubtractionGate    result = x - y - borrow_in + 2^32 borrow_out
    gates/range_check_u32.rs   U32RangeCheckGate     each input is 16 two-bit limbs
    gates/comparison.rs        ComparisonGate        result = first <= second
(wire layouts and constraint orders from memory like the rest of row N1b — parity unpinned; include/b200zkp.h states them).

tests/interpolation_ref.py stays the restatement of the fifteen other gate kinds.  This module extends its gate functions
(`gate_degree`, `gate_num_constraints`, `gate_constraints`, `gate_witness`) with the five kinds and runs vanishing_ref's own
`selector_groups`, `vanishing_terms_at`, `quotient_values` and `check_quotient_identity` with them, through a copy of
vanishing_ref's namespace, as interpolation_ref does.  The constraints use only `+ - *` and `% P`, so plonk_ref.verify
evaluates them over the extension unchanged.  `ecdsa_circuit` builds the gate set of a verifier circuit built with the ecdsa
feature."""
from __future__ import annotations

import random
import types
from typing import List, Sequence

import interpolation_ref as I
from oracle import vanishing_ref as V
from oracle.vanishing_ref import P, root

U32_ARITHMETIC, U32_ADD_MANY, U32_SUBTRACTION, U32_RANGE_CHECK, COMPARISON = 16, 17, 18, 19, 20   # ids of csrc/vanishing_kernels.cuh
U32_GATES = (U32_ARITHMETIC, U32_ADD_MANY, U32_SUBTRACTION, U32_RANGE_CHECK, COMPARISON)
LIMB_BITS, LIMBS_PER_WORD = 2, 16
MAX_NUM_ADDENDS = 16
TWO32 = 1 << 32


# ---------------------------------------------------------------------------------------------------- layouts
def chunk_bits(num_bits: int, num_chunks: int) -> int:
    return -(-num_bits // num_chunks)


def num_wires(kind: int, params) -> int:
    if kind == U32_ARITHMETIC:
        return 38 * params[0]
    if kind == U32_ADD_MANY:
        return (params[0] + 21) * params[1]
    if kind == U32_SUBTRACTION:
        return 21 * params[0]
    if kind == U32_RANGE_CHECK:
        return 17 * params[0]
    nb, nc = params
    return 5 + 5 * nc + chunk_bits(nb, nc)


def config_params(kind: int, arg=None) -> tuple:
    """Gate::new_from_config for standard_recursion_config (135 wires, 80 routed): as many ops as fit both counts.  arg:
    num_addends (U32AddMany), num_input_limbs (U32RangeCheck) or (num_bits, num_chunks) (Comparison)"""
    fit = lambda wires_per_op, routed_per_op: min(V.NUM_WIRES // wires_per_op, V.NUM_ROUTED // routed_per_op)
    if kind == U32_ARITHMETIC:
        return (fit(38, 6),)
    if kind == U32_ADD_MANY:
        return (arg, fit(arg + 21, arg + 3))
    if kind == U32_SUBTRACTION:
        return (fit(21, 5),)
    if kind == U32_RANGE_CHECK:
        return (arg,)
    return tuple(arg)


def arithmetic_layout(num_ops: int):
    return dict(m0=lambda i: 6 * i, m1=lambda i: 6 * i + 1, addend=lambda i: 6 * i + 2, lo=lambda i: 6 * i + 3,
                hi=lambda i: 6 * i + 4, inverse=lambda i: 6 * i + 5, limb=lambda i, j: 6 * num_ops + 32 * i + j, limbs=32)


def add_many_layout(num_addends: int, num_ops: int):
    a = num_addends
    return dict(addend=lambda i, j: (a + 3) * i + j, carry_in=lambda i: (a + 3) * i + a, result=lambda i: (a + 3) * i + a + 1,
                carry_out=lambda i: (a + 3) * i + a + 2, limb=lambda i, j: (a + 3) * num_ops + 18 * i + j, limbs=18)


def subtraction_layout(num_ops: int):
    return dict(x=lambda i: 5 * i, y=lambda i: 5 * i + 1, borrow_in=lambda i: 5 * i + 2, result=lambda i: 5 * i + 3,
                borrow_out=lambda i: 5 * i + 4, limb=lambda i, j: 5 * num_ops + 16 * i + j, limbs=16)


def range_check_layout(num_input_limbs: int):
    return dict(input=lambda i: i, limb=lambda i, j: num_input_limbs + 16 * i + j, limbs=16)


def comparison_layout(num_bits: int, num_chunks: int):
    nc = num_chunks
    return dict(first=0, second=1, result=2, msd=3, first_chunk=lambda c: 4 + c, second_chunk=lambda c: 4 + nc + c,
                dummy=lambda c: 4 + 2 * nc + c, eq=lambda c: 4 + 3 * nc + c, inter=lambda c: 4 + 4 * nc + c,
                bit=lambda b: 4 + 5 * nc + b, cb=chunk_bits(num_bits, num_chunks))


# ---------------------------------------------------------------------------------------------------- constraints
def range_product(x, values: int):
    """prod_{v < values} (x - v)"""
    prod = 1
    for v in range(values):
        prod = prod * (x - v) % P
    return prod


def combine(limbs, base: int):
    """limbs little endian in `base`, folded from the top one down"""
    acc = 0
    for l in reversed(limbs):
        acc = (acc * base + l) % P
    return acc


def _limb_constraints(w, limb, op, n_limbs, out):
    """the limb range of limb j for j = n_limbs - 1 down to 0; returns (limbs below 16 combined, the others combined)"""
    for j in reversed(range(n_limbs)):
        out.append(range_product(w[limb(op, j)], 1 << LIMB_BITS))
    ls = [w[limb(op, j)] for j in range(n_limbs)]
    return combine(ls[:LIMBS_PER_WORD], 1 << LIMB_BITS), combine(ls[LIMBS_PER_WORD:], 1 << LIMB_BITS)


def u32_constraints(kind: int, w: Sequence, params, out: List) -> None:
    """eval_unfiltered of the five gates; appends to `out`"""
    if kind == U32_ARITHMETIC:
        (ops,) = params
        L = arithmetic_layout(ops)
        for i in range(ops):
            lo, hi = w[L["lo"](i)], w[L["hi"](i)]
            out.append((w[L["inverse"](i)] * (0xFFFFFFFF - hi) - 1) * lo % P)
            out.append((hi * TWO32 + lo - (w[L["m0"](i)] * w[L["m1"](i)] + w[L["addend"](i)])) % P)
            low, high = _limb_constraints(w, L["limb"], i, L["limbs"], out)
            out.append((low - lo) % P)
            out.append((high - hi) % P)
    elif kind == U32_ADD_MANY:
        a, ops = params
        L = add_many_layout(a, ops)
        for i in range(ops):
            computed = w[L["carry_in"](i)]
            for j in range(a):
                computed = computed + w[L["addend"](i, j)]
            result, carry = w[L["result"](i)], w[L["carry_out"](i)]
            out.append((carry * TWO32 + result - computed) % P)
            low, high = _limb_constraints(w, L["limb"], i, L["limbs"], out)
            out.append((low - result) % P)
            out.append((high - carry) % P)
    elif kind == U32_SUBTRACTION:
        (ops,) = params
        L = subtraction_layout(ops)
        for i in range(ops):
            borrow = w[L["borrow_out"](i)]
            out.append((w[L["result"](i)] - (w[L["x"](i)] - w[L["y"](i)] - w[L["borrow_in"](i)] + TWO32 * borrow)) % P)
            low, _ = _limb_constraints(w, L["limb"], i, L["limbs"], out)
            out.append((low - w[L["result"](i)]) % P)
            out.append(borrow * (1 - borrow) % P)
    elif kind == U32_RANGE_CHECK:
        (nl,) = params
        L = range_check_layout(nl)
        for i in range(nl):
            limbs = [w[L["limb"](i, j)] for j in range(L["limbs"])]
            out.append((combine(limbs, 1 << LIMB_BITS) - w[L["input"](i)]) % P)
            for l in limbs:
                out.append(range_product(l, 1 << LIMB_BITS))
    elif kind == COMPARISON:
        nb, nc = params
        L = comparison_layout(nb, nc)
        cb = L["cb"]
        first = [w[L["first_chunk"](c)] for c in range(nc)]
        second = [w[L["second_chunk"](c)] for c in range(nc)]
        out.append((combine(first, 1 << cb) - w[L["first"]]) % P)
        out.append((combine(second, 1 << cb) - w[L["second"]]) % P)
        so_far = 0
        for c in range(nc):
            out.append(range_product(first[c], 1 << cb))
            out.append(range_product(second[c], 1 << cb))
            diff = second[c] - first[c]
            eq, inter = w[L["eq"](c)], w[L["inter"](c)]
            out.append((diff * w[L["dummy"](c)] - (1 - eq)) % P)
            out.append(eq * diff % P)
            out.append((inter - eq * so_far) % P)
            so_far = (inter + (1 - eq) * diff) % P
        msd = w[L["msd"]]
        out.append((msd - so_far) % P)
        bits = [w[L["bit"](b)] for b in range(cb + 1)]
        for b in bits:
            out.append(b * (1 - b) % P)
        out.append(((1 << cb) + msd - combine(bits, 2)) % P)
        out.append((w[L["result"]] - bits[cb]) % P)
    else:
        raise ValueError(kind)


# ---------------------------------------------------------------------------------------------------- witnesses
def _limbs(value: int, n: int, bits: int = LIMB_BITS) -> List[int]:
    return [(value >> (bits * j)) & ((1 << bits) - 1) for j in range(n)]


def _inverse(x: int) -> int:
    return pow(x, P - 2, P) if x % P else 0


def u32_witness(kind: int, params, w: List[int], rnd: random.Random, inputs=None) -> None:
    """fill one row of `kind` into `w`: the generators' values for random u32 inputs (or `inputs`: per op (m0, m1, addend) /
    ([addends], carry_in) / (x, y, borrow_in); per limb the input word; (first, second) for Comparison)"""
    u32 = lambda: rnd.choice([0, 1, TWO32 - 1, rnd.randrange(TWO32)])
    if kind == U32_ARITHMETIC:
        (ops,) = params
        L = arithmetic_layout(ops)
        for i in range(ops):
            m0, m1, ad = inputs[i] if inputs else (u32(), u32(), u32())
            v = m0 * m1 + ad
            lo, hi = v % TWO32, v >> 32
            for k, x in (("m0", m0), ("m1", m1), ("addend", ad), ("lo", lo), ("hi", hi)):
                w[L[k](i)] = x
            w[L["inverse"](i)] = _inverse(0xFFFFFFFF - hi)
            for j, l in enumerate(_limbs(v, 32)):
                w[L["limb"](i, j)] = l
    elif kind == U32_ADD_MANY:
        a, ops = params
        L = add_many_layout(a, ops)
        for i in range(ops):
            addends, cin = inputs[i] if inputs else ([u32() for _ in range(a)], rnd.randrange(MAX_NUM_ADDENDS))
            v = sum(addends) + cin
            for j, x in enumerate(addends):
                w[L["addend"](i, j)] = x
            w[L["carry_in"](i)], w[L["result"](i)], w[L["carry_out"](i)] = cin, v % TWO32, v >> 32
            for j, l in enumerate(_limbs(v % TWO32, 16) + _limbs(v >> 32, 2)):
                w[L["limb"](i, j)] = l
    elif kind == U32_SUBTRACTION:
        (ops,) = params
        L = subtraction_layout(ops)
        for i in range(ops):
            x, y, bin_ = inputs[i] if inputs else (u32(), u32(), rnd.randrange(2))
            d = x - y - bin_
            borrow = 1 if d < 0 else 0
            result = d + TWO32 * borrow
            for k, v in (("x", x), ("y", y), ("borrow_in", bin_), ("result", result), ("borrow_out", borrow)):
                w[L[k](i)] = v
            for j, l in enumerate(_limbs(result, 16)):
                w[L["limb"](i, j)] = l
    elif kind == U32_RANGE_CHECK:
        (nl,) = params
        L = range_check_layout(nl)
        for i in range(nl):
            v = inputs[i] if inputs else u32()
            w[L["input"](i)] = v
            for j, l in enumerate(_limbs(v, 16)):
                w[L["limb"](i, j)] = l
    elif kind == COMPARISON:
        nb, nc = params
        L = comparison_layout(nb, nc)
        cb = L["cb"]
        top = (1 << nb) - 1
        first, second = inputs if inputs else (rnd.choice([0, top, rnd.randrange(1 << nb)]), rnd.choice([0, top, rnd.randrange(1 << nb)]))
        w[L["first"]], w[L["second"]] = first, second
        w[L["result"]] = int(first <= second)
        fc, sc = _limbs(first, nc, cb), _limbs(second, nc, cb)
        so_far = 0
        for c in range(nc):
            w[L["first_chunk"](c)], w[L["second_chunk"](c)] = fc[c], sc[c]
            w[L["eq"](c)] = int(fc[c] == sc[c])
            w[L["dummy"](c)] = 1 if fc[c] == sc[c] else _inverse(sc[c] - fc[c])
            if fc[c] != sc[c]:
                so_far = (sc[c] - fc[c]) % P
                w[L["inter"](c)] = 0
            else:
                w[L["inter"](c)] = so_far
        w[L["msd"]] = so_far
        for b, bit in enumerate(_limbs(((1 << cb) + so_far) % P, cb + 1, 1)):
            w[L["bit"](b)] = bit
    else:
        raise ValueError(kind)


# ---------------------------------------------------------------------------------------------------- the gate functions, extended
def gate_degree(kind: int, params=()) -> int:
    """Gate::degree()"""
    if kind == COMPARISON:
        return 1 << chunk_bits(*params)
    if kind in U32_GATES:
        return 1 << LIMB_BITS
    return I.gate_degree(kind, params)


def gate_num_constraints(kind: int, params=()) -> int:
    """Gate::num_constraints()"""
    if kind == U32_ARITHMETIC:
        return 36 * params[0]
    if kind == U32_ADD_MANY:
        return 21 * params[1]
    if kind == U32_SUBTRACTION:
        return 19 * params[0]
    if kind == U32_RANGE_CHECK:
        return 17 * params[0]
    if kind == COMPARISON:
        return 6 + 5 * params[1] + chunk_bits(*params)
    return I.gate_num_constraints(kind, params)


def gate_constraints(kind: int, wires: Sequence[int], consts: Sequence[int], pi_hash: Sequence[int], params=()) -> List[int]:
    """eval_unfiltered of one gate type at one point"""
    if kind in U32_GATES:
        out: List[int] = []
        u32_constraints(kind, wires, params, out)
        return out
    return I.gate_constraints(kind, wires, consts, pi_hash, params)


def gate_witness(kind: int, rnd: random.Random, consts: Sequence[int], params=()) -> List[int]:
    """135 wires of one row of `kind` whose constraints vanish"""
    if kind in U32_GATES:
        w = [rnd.randrange(P) for _ in range(V.NUM_WIRES)]
        u32_witness(kind, params, w, rnd)
        return w
    return I.gate_witness(kind, rnd, consts, params)


# ---------------------------------------------------------------------------------------------------- vanishing_ref's code, these gates
_NAMESPACE = dict(vars(V), gate_degree=gate_degree, gate_num_constraints=gate_num_constraints, gate_constraints=gate_constraints)


def _with_u32(fn):
    """vanishing_ref's function `fn` (its code object unchanged) resolving module names in a copy of vanishing_ref's namespace
    in which the gate functions are the ones above"""
    g = types.FunctionType(fn.__code__, _NAMESPACE, fn.__name__, fn.__defaults__, fn.__closure__)
    _NAMESPACE[fn.__name__] = g
    return g


selector_groups = _with_u32(V.selector_groups)
vanishing_terms_at = _with_u32(V.vanishing_terms_at)
quotient_values = _with_u32(V.quotient_values)
check_quotient_identity = _with_u32(V.check_quotient_identity)


# ---------------------------------------------------------------------------------------------------- circuits
def add_gate_rows(c: V.Circuit, rows) -> dict:
    """put rows [(kind, params, wires)] of new gate kinds on the last no-op rows of `c` (every cell of a no-op row is its own copy
    cycle); the gate list is re-sorted by degree (stable: a new kind follows the kinds of its degree already there) and the
    selector polynomials are recomputed.  Returns {index into rows: the row it went to}."""
    noop = c.gates.index(V.NOOP)
    free = [r for r in range(c.n) if c.row_gate[r] == noop]
    if len(rows) >= len(free):
        raise ValueError(f"{len(rows)} rows do not fit in the circuit's {len(free)} no-op rows")
    entries = list(zip(c.gates, c.gate_params))
    kinds = []
    for kind, params, _ in rows:
        if (kind, params) not in entries:
            entries.append((kind, params))
        kinds.append(entries.index((kind, params)))
    order = sorted(range(len(entries)), key=lambda e: gate_degree(*entries[e]))
    new_index = {old: k for k, old in enumerate(order)}
    c.gates = [entries[e][0] for e in order]
    c.gate_params = [entries[e][1] for e in order]
    c.row_gate = [new_index[g] for g in c.row_gate]
    placed = {}
    for t, ((_, _, w), e) in enumerate(zip(rows, kinds)):
        r = free[len(free) - len(rows) + t]
        for j in range(V.NUM_WIRES):
            c.wires[j][r] = w[j]
        c.row_gate[r] = new_index[e]
        placed[t] = r
    c.selector_indices, c.groups = selector_groups(list(zip(c.gates, c.gate_params)), c.max_degree)
    c.num_selectors = len(c.groups)
    c.constants = [[c.row_gate[r] if grp[0] <= c.row_gate[r] < grp[1] else V.UNUSED_SELECTOR for r in range(c.n)] for grp in c.groups]
    c.constants += c.gate_consts
    return placed


def copy_cells(c: V.Circuit, a, b) -> None:
    """a copy constraint between cells a = (wire, row) and b, both still their own copy cycles: sigma swaps them"""
    cell = lambda j, r: c.k_is[j] * pow(root(c.n_log), r, P) % P
    for j, r in (a, b):
        assert j < V.NUM_ROUTED and c.sigmas[j][r] == cell(j, r), "the cell must be routed and a fixed point of sigma"
    assert c.wires[a[0]][a[1]] == c.wires[b[0]][b[1]], "copy constraint between unequal cells"
    c.sigmas[a[0]][a[1]], c.sigmas[b[0]][b[1]] = cell(*b), cell(*a)


# the two U32AddManyGate arities of ecdsa_circuit (num_addends) and its ComparisonGate (list_le_u32_circuit's)
ECDSA_ADD_MANY_ARITIES = (3, 16)
ECDSA_COMPARISON = (32, 16)
ECDSA_RANGE_CHECK_LIMBS = 4


def ecdsa_u32_params():
    """(kind, params) of the six u32 rows ecdsa_circuit adds, in row order"""
    return [(U32_ARITHMETIC, config_params(U32_ARITHMETIC))] + \
           [(U32_ADD_MANY, config_params(U32_ADD_MANY, a)) for a in ECDSA_ADD_MANY_ARITIES] + \
           [(U32_SUBTRACTION, config_params(U32_SUBTRACTION)), (U32_RANGE_CHECK, config_params(U32_RANGE_CHECK, ECDSA_RANGE_CHECK_LIMBS)),
            (COMPARISON, config_params(COMPARISON, ECDSA_COMPARISON))]


def ecdsa_circuit(n_log: int, seed: int = 0, n_poseidon: int | None = None) -> V.Circuit:
    """interpolation_ref's recursion_circuit (14 gate kinds) plus one satisfied row of each plonky2_u32 gate, U32AddManyGate at two
    arities: 20 gate kinds, the set of a verifier circuit built with the ecdsa feature.  The u32 rows are chained by copy
    constraints, so the permutation argument covers routed u32 wires: U32Arithmetic's low output is an AddMany addend, that
    AddMany's result is the Subtraction's x, the Subtraction's result is the Comparison's first input, and a RangeCheck input
    limb is its second input.  n_poseidon defaults to n / 2 - 8, which leaves room for the u32 rows at 2^5."""
    n = 1 << n_log
    c = I.recursion_circuit(n_log, seed=seed, n_poseidon=max(1, n // 2 - 8) if n_poseidon is None else n_poseidon)
    rnd = random.Random(seed + 2000)
    specs = ecdsa_u32_params()
    rows = []
    for kind, params in specs:
        rows.append([rnd.randrange(P) for _ in range(V.NUM_WIRES)])
    (k_ar, p_ar), (_, p_am), (_, p_am16), (_, p_sub), (_, p_rc), (_, p_cmp) = specs
    u32_witness(U32_ARITHMETIC, p_ar, rows[0], rnd)
    lo = rows[0][arithmetic_layout(p_ar[0])["lo"](0)]
    am = add_many_layout(*p_am)
    u32_witness(U32_ADD_MANY, p_am, rows[1], rnd,
                inputs=[([lo] + [rnd.randrange(TWO32) for _ in range(p_am[0] - 1)], rnd.randrange(16))] +
                       [([rnd.randrange(TWO32) for _ in range(p_am[0])], rnd.randrange(16)) for _ in range(p_am[1] - 1)])
    u32_witness(U32_ADD_MANY, p_am16, rows[2], rnd)
    sub = subtraction_layout(p_sub[0])
    x = rows[1][am["result"](0)]
    u32_witness(U32_SUBTRACTION, p_sub, rows[3], rnd,
                inputs=[(x, rnd.randrange(TWO32), 1)] + [(rnd.randrange(TWO32), rnd.randrange(TWO32), rnd.randrange(2))
                                                        for _ in range(p_sub[0] - 1)])
    u32_witness(U32_RANGE_CHECK, p_rc, rows[4], rnd)
    second = rows[4][range_check_layout(p_rc[0])["input"](1)]
    u32_witness(COMPARISON, p_cmp, rows[5], rnd, inputs=(rows[3][sub["result"](0)], second))
    for (kind, params), w in zip(specs, rows):
        assert not any(gate_constraints(kind, w, [0, 0], [0] * 4, params)), kind
    placed = add_gate_rows(c, [(kind, params, w) for (kind, params), w in zip(specs, rows)])
    cmp_l = comparison_layout(*p_cmp)
    copy_cells(c, (arithmetic_layout(p_ar[0])["lo"](0), placed[0]), (am["addend"](0, 0), placed[1]))
    copy_cells(c, (am["result"](0), placed[1]), (sub["x"](0), placed[3]))
    copy_cells(c, (sub["result"](0), placed[3]), (cmp_l["first"], placed[5]))
    copy_cells(c, (range_check_layout(p_rc[0])["input"](1), placed[4]), (cmp_l["second"], placed[5]))
    c.u32_rows = [placed[t] for t in range(len(specs))]
    return c


def single_gate_circuit(n_log: int, kind: int, params, seed: int = 0) -> V.Circuit:
    """vanishing_ref's 5-gate circuit plus one row of one u32 gate"""
    c = V.Circuit(n_log, seed=seed, n_poseidon=max(1, (1 << n_log) // 4))
    rnd = random.Random(seed + 3000)
    w = gate_witness(kind, rnd, [0, 0], params)
    placed = add_gate_rows(c, [(kind, params, w)])
    c.u32_rows = [placed[0]]
    return c
