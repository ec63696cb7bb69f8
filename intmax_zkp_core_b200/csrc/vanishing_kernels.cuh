// Row N1b: the vanishing polynomial on the quotient coset, divided by Z_H — the reader of the three resident LDEs.
//
// Replaces plonky2 @ f99ed9c plonky2/src/plonk/prover.rs `compute_quotient_polys` (up to, not including, its coset_ifft,
// which is row N1c: b200zkp_dev_coset_intt) with plonk/vanishing_poly.rs `eval_vanishing_poly_base_batch` /
// `evaluate_gate_constraints_base_batch`, plonk_common.rs `ZeroPolyOnCoset`, `eval_l_1`, `reduce_with_powers`,
// gates/selectors.rs `compute_filter` and the eval_unfiltered of gates/{noop, constant, public_input, arithmetic_base,
// poseidon, poseidon_mds, base_sum, arithmetic_extension, multiplication_extension, reducing, reducing_extension,
// random_access, exponentiation, interpolation, low_degree_interpolation}.rs.  Reached from the reference through every prove() (/root/reference/src/rollup/circuits/mod.rs:1247,
// src/transaction/circuits/mod.rs:453, src/zkdsa/circuits/mod.rs:326); PoseidonGate is what
// /root/reference/src/poseidon/gadgets/mod.rs:7-22 instantiates.  Restated in oracle/vanishing_ref.py (parity unpinned: the
// crate source is not on this machine; the verifier's identity pins the restatement, tests/test_oracle_vanishing.py).
//
// One thread per point of the quotient coset 7 <w_Q>, Q = n 2^q.  The LDEs stay column-major in LEAF order: leaf t of the
// first Q leaves is the natural point i = bitrev(t) of the quotient coset (also when q < rate_bits: the sub-coset is a prefix
// of the leaf order), so consecutive threads read consecutive words of every column; only Z(g x) (C words) and the result
// (C words, natural order for the coset_ifft that follows) are scattered.  Terms are folded into sum_t alpha^t term_t as they
// are produced (alpha powers from a table), gate constraints per gate type first and then times the selector filter, so no
// per-thread array of constraints exists.  All values canonical.
#pragma once
#include "goldilocks.cuh"
#include "poseidon_gate_tables.cuh"

namespace vanish {

using gl::u32;
using gl::u64;

enum GateKind : u32 {
    GATE_NOOP = 0, GATE_CONSTANT = 1, GATE_PUBLIC_INPUT = 2, GATE_ARITHMETIC = 3, GATE_POSEIDON = 4,
    GATE_ARITHMETIC_EXTENSION = 5,   // 4 D wires per op: multiplicand 0, multiplicand 1, addend, output; constants c0, c1
    GATE_MUL_EXTENSION = 6,          // 3 D wires per op: multiplicand 0, multiplicand 1, output; constant c0
    GATE_BASE_SUM = 7,               // params (B, num_limbs): wire 0 = sum, limbs from wire 1 (little endian)
    GATE_REDUCING = 8,               // params (num_coeffs): output, alpha, old_acc (D wires each), base-field coefficients, accumulators
    GATE_REDUCING_EXTENSION = 9,     // params (num_coeffs): the same with extension-field coefficients
    GATE_RANDOM_ACCESS = 10,         // params (bits, num_copies, num_extra_constants)
    GATE_EXPONENTIATION = 11,        // params (num_power_bits): base, power bits, output, intermediate values
    GATE_POSEIDON_MDS = 12,          // 12 extension inputs, 12 extension outputs
    // (13 is not assigned)
    GATE_INTERPOLATION_HIGH_DEGREE = 14,   // params (subgroup_bits): m = 2^subgroup_bits points, degree m
    GATE_INTERPOLATION_LOW_DEGREE = 15,    // params (subgroup_bits): the same with power wires, degree 2
    GATE_U32_ARITHMETIC = 16,        // params (num_ops): lo + 2^32 hi = m0 m1 + addend, 32 two-bit limbs per op
    GATE_U32_ADD_MANY = 17,          // params (num_addends, num_ops): result + 2^32 carry_out = sum + carry_in, 18 limbs per op
    GATE_U32_SUBTRACTION = 18,       // params (num_ops): result = x - y - borrow_in + 2^32 borrow_out, 16 limbs per op
    GATE_U32_RANGE_CHECK = 19,       // params (num_input_limbs): 16 two-bit limbs per input
    GATE_COMPARISON = 20             // params (num_bits, num_chunks): result = first <= second, degree 2^chunk_bits
};
static constexpr u32 D = 2;          // quadratic extension F[X] / (X^2 - 7)
static constexpr u32 MAX_GATES = 32, MAX_CHALLENGES = 4;
static constexpr u32 UNUSED_SELECTOR = 0xFFFFFFFFu;
// PoseidonGate wire layout (gates/poseidon.rs)
static constexpr u32 W_IN = 0, W_OUT = 12, W_SWAP = 24, W_DELTA = 25, W_FULL0 = 29, W_PARTIAL = 65, W_FULL1 = 87;

// InterpolationGate layout (gates/interpolation.rs, low_degree_interpolation.rs), m = 2^subgroup_bits, ext(j) = wires j, j + 1:
// shift 0, value(i) ext(1 + D i), evaluation point ext(1 + D m), evaluation value ext(3 + D m), coeff(i) ext(5 + D m + D i), up
// to end_coeffs = 5 + 4 m; LowDegree only: shift^i at end_coeffs + i - 2 and ext eval_point^i at end_coeffs + m - 2 + D (i - 2)
// for 2 <= i < m

// plonky2_u32 layouts (gates/*_u32.rs, comparison.rs; include/b200zkp.h states them with their constraint order).  Limbs are 2
// bits, combined little endian in base 4.  U32Arithmetic op i: m0 6i, m1 6i+1, addend 6i+2, lo 6i+3, hi 6i+4, inverse 6i+5,
// limb j at 6 num_ops + 32i + j.  U32AddMany (a addends) op i: addend j (a+3)i + j, carry_in (a+3)i + a, result +1, carry_out
// +2, limb j at (a+3) num_ops + 18i + j (16 result limbs, 2 carry limbs).  U32Subtraction op i: x 5i, y 5i+1, borrow_in 5i+2,
// result 5i+3, borrow_out 5i+4, limb j at 5 num_ops + 16i + j.  U32RangeCheck: input i at i, its limb j at num_input_limbs +
// 16i + j.  Comparison (nc chunks of cb = ceil(num_bits / nc) bits): first 0, second 1, result 2, most-significant diff 3,
// first chunk c 4 + c, second chunk 4 + nc + c, equality dummy 4 + 2nc + c, chunks_equal 4 + 3nc + c, intermediate 4 + 4nc + c,
// bit b <= cb of 2^cb + msd at 4 + 5nc + b
static constexpr u32 U32_LIMBS_PER_WORD = 16;
GL_HD u32 comparison_chunk_bits(u32 num_bits, u32 num_chunks) { return num_chunks ? (num_bits + num_chunks - 1) / num_chunks : 0; }

struct GateDesc { u32 kind, selector_index, group_begin, group_end, p0, p1, p2; };

GL_HD bool gate_supported(u32 kind) {
    return kind <= GATE_POSEIDON_MDS || (kind >= GATE_INTERPOLATION_HIGH_DEGREE && kind <= GATE_COMPARISON);
}

// Gate::num_constraints() of standard_recursion_config instances (host and device)
GL_HD u32 gate_num_constraints(u32 kind, u32 num_routed, u32 num_gate_consts, u32 p0, u32 p1, u32 p2) {
    switch (kind) {
        case GATE_CONSTANT: return num_gate_consts;
        case GATE_PUBLIC_INPUT: return 4;
        case GATE_ARITHMETIC: return num_routed / 4;
        case GATE_POSEIDON: return 123;
        case GATE_ARITHMETIC_EXTENSION: return (num_routed / (4 * D)) * D;
        case GATE_MUL_EXTENSION: return (num_routed / (3 * D)) * D;
        case GATE_BASE_SUM: return 1 + p1;
        case GATE_REDUCING: case GATE_REDUCING_EXTENSION: return D * p0;
        case GATE_RANDOM_ACCESS: return p1 * (p0 + 2) + p2;
        case GATE_EXPONENTIATION: return p0 + 1;
        case GATE_POSEIDON_MDS: return 12 * D;
        case GATE_INTERPOLATION_HIGH_DEGREE: return D * ((1u << p0) + 1);
        case GATE_INTERPOLATION_LOW_DEGREE: return 5 * (1u << p0) - 4;
        case GATE_U32_ARITHMETIC: return 36 * p0;
        case GATE_U32_ADD_MANY: return 21 * p1;
        case GATE_U32_SUBTRACTION: return 19 * p0;
        case GATE_U32_RANGE_CHECK: return 17 * p0;
        case GATE_COMPARISON: return 6 + 5 * p1 + comparison_chunk_bits(p0, p1);
        default: return 0;
    }
}
// highest wire index the gate reads + 1 (argument check on the host)
GL_HD u32 gate_num_wires(u32 kind, u32 num_routed, u32 p0, u32 p1, u32 p2) {
    switch (kind) {
        case GATE_BASE_SUM: return 1 + p1;
        case GATE_REDUCING: return 3 * D + p0 + D * (p0 ? p0 - 1 : 0);
        case GATE_REDUCING_EXTENSION: return 3 * D + D * p0 + D * (p0 ? p0 - 1 : 0);
        case GATE_RANDOM_ACCESS: return (2 + (1u << p0)) * p1 + p2 + p0 * p1;
        case GATE_EXPONENTIATION: return 2 + 2 * p0;
        case GATE_POSEIDON_MDS: return 24 * D;
        case GATE_POSEIDON: return 135;
        case GATE_INTERPOLATION_HIGH_DEGREE: return 5 + 4 * (1u << p0);
        case GATE_INTERPOLATION_LOW_DEGREE: return 7 * (1u << p0) - 1;
        case GATE_U32_ARITHMETIC: return 38 * p0;
        case GATE_U32_ADD_MANY: return (p0 + 21) * p1;
        case GATE_U32_SUBTRACTION: return 21 * p0;
        case GATE_U32_RANGE_CHECK: return 17 * p0;
        case GATE_COMPARISON: return 5 + 5 * p1 + comparison_chunk_bits(p0, p1);
        default: return num_routed;
    }
}

struct E2 { u64 a, b; };
GL_FN E2 e2_mul(E2 x, E2 y) {
    return E2{gl::add(gl::mul(x.a, y.a), gl::mul(7, gl::mul(x.b, y.b))), gl::add(gl::mul(x.a, y.b), gl::mul(x.b, y.a))};
}
GL_FN E2 e2_add(E2 x, E2 y) { return E2{gl::add(x.a, y.a), gl::add(x.b, y.b)}; }
GL_FN E2 e2_sub(E2 x, E2 y) { return E2{gl::sub(x.a, y.a), gl::sub(x.b, y.b)}; }
GL_FN E2 e2_scale(E2 x, u64 c) { return E2{gl::mul(x.a, c), gl::mul(x.b, c)}; }

struct Params {
    const u64 *cs, *wires, *zpp;               // constants+sigmas, wires, Z+partial products: [columns][stride], leaf order
    u64 cs_stride, wires_stride, zpp_stride;
    u32 n_log, q_bits;                         // degree bits, quotient_degree_bits (the first n << q_bits leaves are read)
    u32 num_selectors, num_gate_consts, num_routed, num_challenges, num_prods, degree;
    u32 n_gates, n_terms;
    GateDesc gates[MAX_GATES];
    u64 betas[MAX_CHALLENGES], gammas[MAX_CHALLENGES], pi_hash[4];
    const u64* k_is;                           // [num_routed]
    const u64* alpha_pows;                     // [num_challenges][n_terms]
    const u64 *zh, *zh_inv;                    // [2^q_bits]: Z_H on the coset, 7^n w_(2^q)^i - 1, and its inverse (ZeroPolyOnCoset)
    const u64 *tw_lo, *tw_hi;                  // two-level powers of w_Q
    u32 tw_lo_bits;
    u64 n_inv;                                 // 1 / n
    u64* out;                                  // [num_challenges][out_stride], natural order
    u64 out_stride;
};

GL_FN u64 sbox(u64 x) {
    const u64 x2 = gl::mul(x, x), x4 = gl::mul(x2, x2), x3 = gl::mul(x2, x);
    return gl::mul(x3, x4);
}

// x^(p-2)
GL_FN u64 inverse(u64 x) {
    // p - 2 = 0xFFFFFFFEFFFFFFFF: square-and-multiply from the top bit
    u64 r = 1;
#pragma unroll 1
    for (int b = 63; b >= 0; b--) {
        r = gl::mul(r, r);
        if ((0xFFFFFFFEFFFFFFFFull >> b) & 1) r = gl::mul(r, x);
    }
    return r;
}

// state <- MDS state (circulant (17,15,41,16,2,28,13,13,39,18,34,20) + diag(8,0,..)), 128-bit accumulation, one reduction per word
GL_FN void mds_layer(u64 (&s)[12]) {
    constexpr u32 CIRC[12] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    u64 o[12];
#pragma unroll
    for (int r = 0; r < 12; r++) {
        unsigned __int128 acc = 0;
#pragma unroll
        for (int i = 0; i < 12; i++) acc += (unsigned __int128)s[(i + r) % 12] * CIRC[i];
        if (r == 0) acc += (unsigned __int128)s[0] * 8u;
        o[r] = gl::canon(gl::reduce128((u64)acc, (u64)(acc >> 64)));
    }
#pragma unroll
    for (int r = 0; r < 12; r++) s[r] = o[r];
}

// primitive 2^bits-th root of unity, the one the NTT uses: G^(2^(32 - bits)) for the generator G of the 2^32 subgroup
GL_FN u64 root_of_unity(u32 bits) {
    u64 g = 1753635133440165772ull;
#pragma unroll 1
    for (u32 k = bits; k < 32; k++) g = gl::mul(g, g);
    return g;
}

// prod_{v < 4} (x - v): the range check of a two-bit limb
GL_FN u64 limb_range(u64 x) { return gl::mul(gl::mul(x, gl::sub(x, 1)), gl::mul(gl::sub(x, 2), gl::sub(x, 3))); }

// running sums of one gate's constraints, one per challenge
struct Fold {
    u64 acc[MAX_CHALLENGES];
    const u64* pw;      // alpha_pows + index of the gate's first constraint
    u32 n_terms, C, t;
    GL_MFN void add(u64 v) {
#pragma unroll
        for (u32 c = 0; c < MAX_CHALLENGES; c++)
            if (c < C) acc[c] = gl::add(acc[c], gl::mul(v, gl::ldg(pw + (u64)c * n_terms + t)));
        t++;
    }
};

// gates/poseidon.rs eval_unfiltered: 123 constraints; wire j of this point at w[j * stride]
GL_FN void poseidon_gate(const u64* __restrict__ w, u64 stride, Fold& f) {
    using namespace poseidon_gate_tables;
    auto wire = [&](u32 j) { return w[(u64)j * stride]; };
    const u64 swap = wire(W_SWAP);
    f.add(gl::mul(swap, gl::sub(swap, 1)));
    u64 s[12];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const u64 lhs = wire(W_IN + i), rhs = wire(W_IN + 4 + i), delta = wire(W_DELTA + i);
        f.add(gl::sub(gl::mul(swap, gl::sub(rhs, lhs)), delta));
        s[i] = gl::add(lhs, delta);
        s[i + 4] = gl::sub(rhs, delta);
    }
#pragma unroll
    for (int i = 8; i < 12; i++) s[i] = wire(W_IN + i);
    u32 rnd = 0;
#pragma unroll 1
    for (int r = 0; r < 4; r++) {
#pragma unroll
        for (int i = 0; i < 12; i++) s[i] = gl::add(s[i], RC_ALL[rnd * 12 + i]);
        if (r) {
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const u64 s_in = wire(W_FULL0 + 12 * (r - 1) + i);
                f.add(gl::sub(s[i], s_in));
                s[i] = s_in;
            }
        }
#pragma unroll
        for (int i = 0; i < 12; i++) s[i] = sbox(s[i]);
        mds_layer(s);
        rnd++;
    }
    // partial rounds in the fast form whose word 0 is the gate's S-box input wire
#pragma unroll
    for (int i = 0; i < 12; i++) s[i] = gl::add(s[i], FAST_FIRST[i]);
    {
        u64 o[11];
#pragma unroll 1
        for (int r = 0; r < 11; r++) {
            u64 acc = 0;
#pragma unroll
            for (int i = 0; i < 11; i++) acc = gl::add(acc, gl::mul(FAST_INIT[r * 11 + i], s[1 + i]));
            o[r] = acc;
        }
#pragma unroll
        for (int r = 0; r < 11; r++) s[1 + r] = o[r];
    }
#pragma unroll 1
    for (int r = 0; r < 22; r++) {
        const u64 s_in = wire(W_PARTIAL + r);
        f.add(gl::sub(s[0], s_in));
        const u64 s0 = gl::add(sbox(s_in), FAST_POST[r]);
        u64 new0 = gl::mul(s0, 25);
#pragma unroll
        for (int i = 0; i < 11; i++) {
            new0 = gl::add(new0, gl::mul(FAST_VHAT[r * 11 + i], s[1 + i]));
            s[1 + i] = gl::add(s[1 + i], gl::mul(FAST_WHAT[r * 11 + i], s0));
        }
        s[0] = new0;
    }
    rnd += 22;
#pragma unroll 1
    for (int r = 0; r < 4; r++) {
#pragma unroll
        for (int i = 0; i < 12; i++) {
            s[i] = gl::add(s[i], RC_ALL[rnd * 12 + i]);
            const u64 s_in = wire(W_FULL1 + 12 * r + i);
            f.add(gl::sub(s[i], s_in));
            s[i] = sbox(s_in);
        }
        mds_layer(s);
        rnd++;
    }
#pragma unroll
    for (int i = 0; i < 12; i++) f.add(gl::sub(s[i], wire(W_OUT + i)));
}

// everything one thread does: leaf position t of the quotient coset (also stepped on the host by tests/emu)
GL_FN void quotient_point(const Params& p, u64 t) {
    const u32 Q_log = p.n_log + p.q_bits;
    const u64 Q = (u64)1 << Q_log;
    if (t >= Q) return;
    const u32 C = p.num_challenges;
    const u64 i = Q_log ? (gl::brev64(t) >> (64 - Q_log)) : 0;       // natural index on the quotient coset
    const u64 x = gl::mul(7, gl::mul(gl::ldg(p.tw_lo + (i & (((u64)1 << p.tw_lo_bits) - 1))), gl::ldg(p.tw_hi + (i >> p.tw_lo_bits))));
    const u64 i_next = (i + ((u64)1 << p.q_bits)) & (Q - 1);
    const u64 t_next = Q_log ? (gl::brev64(i_next) >> (64 - Q_log)) : 0;
    const u64* __restrict__ cs = p.cs + t;
    const u64* __restrict__ wr = p.wires + t;
    const u64* __restrict__ zp = p.zpp + t;
    const u32 n_const = p.num_selectors + p.num_gate_consts;

    u64 acc[MAX_CHALLENGES] = {0, 0, 0, 0};
    auto alpha = [&](u32 c, u32 term) { return gl::ldg(p.alpha_pows + (u64)c * p.n_terms + term); };

    // Z_H(x)^-1 and L_1(x) = Z_H(x) / (n (x - 1))
    const u64 zh_inv = gl::ldg(p.zh_inv + (i & (((u64)1 << p.q_bits) - 1)));
    const u64 zh = gl::ldg(p.zh + (i & (((u64)1 << p.q_bits) - 1)));
    const u64 l1 = gl::mul(gl::mul(zh, p.n_inv), inverse(gl::sub(x, 1)));      // x != 1 on the coset
    u32 term = 0;
    for (u32 c = 0; c < C; c++, term++) {
        const u64 z_x = zp[(u64)c * p.zpp_stride];
        const u64 v = gl::mul(l1, gl::sub(z_x, 1));
        for (u32 a = 0; a < C; a++) acc[a] = gl::add(acc[a], gl::mul(v, alpha(a, term)));
    }
    // permutation checks, chunk by chunk
    const u32 chunks = p.num_prods + 1;
    for (u32 c = 0; c < C; c++) {
        const u64 beta = p.betas[c], gamma = p.gammas[c];
        const u64 bx = gl::mul(beta, x);
        u64 prev = zp[(u64)c * p.zpp_stride];
        for (u32 l = 0; l < chunks; l++, term++) {
            const u64 next = (l + 1 < chunks) ? zp[(u64)(C + c * p.num_prods + l) * p.zpp_stride]
                                              : p.zpp[(u64)c * p.zpp_stride + t_next];
            u64 num = 1, den = 1;
            const u32 j1 = p.num_routed < (l + 1) * p.degree ? p.num_routed : (l + 1) * p.degree;
            for (u32 j = l * p.degree; j < j1; j++) {
                const u64 wj = wr[(u64)j * p.wires_stride];
                const u64 wg = gl::add(wj, gamma);
                num = gl::mul(num, gl::add(wg, gl::mul(bx, gl::ldg(p.k_is + j))));
                den = gl::mul(den, gl::add(wg, gl::mul(beta, cs[(u64)(n_const + j) * p.cs_stride])));
            }
            const u64 v = gl::sub(gl::mul(prev, num), gl::mul(next, den));
            for (u32 a = 0; a < C; a++) acc[a] = gl::add(acc[a], gl::mul(v, alpha(a, term)));
            prev = next;
        }
    }
    // gate constraints: every gate type at every point, times its selector filter
    const u64* __restrict__ gc = cs + (u64)p.num_selectors * p.cs_stride;      // gate constants
    for (u32 g = 0; g < p.n_gates; g++) {
        const GateDesc gd = p.gates[g];
        if (gd.kind == GATE_NOOP) continue;
        const u64 s = cs[(u64)gd.selector_index * p.cs_stride];
        u64 filter = 1;
        for (u32 q = gd.group_begin; q < gd.group_end; q++)
            if (q != g) filter = gl::mul(filter, gl::sub((u64)q, s));
        if (p.num_selectors > 1) filter = gl::mul(filter, gl::sub((u64)UNUSED_SELECTOR, s));
        Fold f;
        f.pw = p.alpha_pows + term; f.n_terms = p.n_terms; f.C = C; f.t = 0;
        auto wire = [&](u32 j) { return wr[(u64)j * p.wires_stride]; };
        auto ext = [&](u32 j) { return E2{wr[(u64)j * p.wires_stride], wr[(u64)(j + 1) * p.wires_stride]}; };
#pragma unroll
        for (u32 c = 0; c < MAX_CHALLENGES; c++) f.acc[c] = 0;
        switch (gd.kind) {
            case GATE_CONSTANT:                                       // gates/constant.rs
                for (u32 q = 0; q < p.num_gate_consts; q++) f.add(gl::sub(gc[(u64)q * p.cs_stride], wr[(u64)q * p.wires_stride]));
                break;
            case GATE_PUBLIC_INPUT:                                   // gates/public_input.rs
                for (u32 q = 0; q < 4; q++) f.add(gl::sub(wr[(u64)q * p.wires_stride], p.pi_hash[q]));
                break;
            case GATE_ARITHMETIC: {                                   // gates/arithmetic_base.rs, num_ops = num_routed / 4
                const u64 c0 = gc[0], c1 = gc[p.cs_stride];
                for (u32 q = 0; q < p.num_routed / 4; q++) {
                    const u64 m0 = wr[(u64)(4 * q) * p.wires_stride], m1 = wr[(u64)(4 * q + 1) * p.wires_stride];
                    const u64 ad = wr[(u64)(4 * q + 2) * p.wires_stride], o = wr[(u64)(4 * q + 3) * p.wires_stride];
                    f.add(gl::sub(o, gl::add(gl::mul(gl::mul(m0, m1), c0), gl::mul(ad, c1))));
                }
                break;
            }
            case GATE_POSEIDON:
                poseidon_gate(wr, p.wires_stride, f);
                break;
            case GATE_ARITHMETIC_EXTENSION: {                         // gates/arithmetic_extension.rs
                const u64 c0 = gc[0], c1 = gc[p.cs_stride];
                for (u32 q = 0; q < p.num_routed / (4 * D); q++) {
                    const u32 w0 = 4 * D * q;
                    const E2 r = e2_sub(ext(w0 + 3 * D), e2_add(e2_scale(e2_mul(ext(w0), ext(w0 + D)), c0), e2_scale(ext(w0 + 2 * D), c1)));
                    f.add(r.a); f.add(r.b);
                }
                break;
            }
            case GATE_MUL_EXTENSION: {                                // gates/multiplication_extension.rs
                const u64 c0 = gc[0];
                for (u32 q = 0; q < p.num_routed / (3 * D); q++) {
                    const u32 w0 = 3 * D * q;
                    const E2 r = e2_sub(ext(w0 + 2 * D), e2_scale(e2_mul(ext(w0), ext(w0 + D)), c0));
                    f.add(r.a); f.add(r.b);
                }
                break;
            }
            case GATE_BASE_SUM: {                                     // gates/base_sum.rs
                const u32 base = gd.p0, num_limbs = gd.p1;
                u64 computed = 0;
                for (u32 q = num_limbs; q-- > 0;) computed = gl::add(gl::mul(computed, base), wire(1 + q));
                f.add(gl::sub(computed, wire(0)));
                for (u32 q = 0; q < num_limbs; q++) {
                    const u64 l = wire(1 + q);
                    u64 prod = 1;
                    for (u32 v = 0; v < base; v++) prod = gl::mul(prod, gl::sub(l, (u64)v));
                    f.add(prod);
                }
                break;
            }
            case GATE_REDUCING:
            case GATE_REDUCING_EXTENSION: {                           // gates/reducing.rs, reducing_extension.rs
                const u32 nc = gd.p0, cw = gd.kind == GATE_REDUCING ? 1u : D;
                const E2 output = ext(0), alpha = ext(D);
                E2 acc = ext(2 * D);
                const u32 start_coeffs = 3 * D, start_accs = start_coeffs + nc * cw;
                for (u32 q = 0; q < nc; q++) {
                    const E2 coeff = gd.kind == GATE_REDUCING ? E2{wire(start_coeffs + q), 0} : ext(start_coeffs + D * q);
                    const E2 acc_q = (q + 1 == nc) ? output : ext(start_accs + D * q);
                    const E2 r = e2_sub(e2_add(e2_mul(acc, alpha), coeff), acc_q);
                    f.add(r.a); f.add(r.b);
                    acc = acc_q;
                }
                break;
            }
            case GATE_RANDOM_ACCESS: {                                // gates/random_access.rs
                const u32 bits = gd.p0, copies = gd.p1, extra = gd.p2, vec = 1u << bits;
                const u32 routed = (2 + vec) * copies + extra;
                for (u32 cp = 0; cp < copies; cp++) {
                    const u32 base_w = (2 + vec) * cp, bit_w = routed + cp * bits;
                    u64 rec = 0;
                    for (u32 q = 0; q < bits; q++) { const u64 b = wire(bit_w + q); f.add(gl::mul(b, gl::sub(b, 1))); }
                    for (u32 q = bits; q-- > 0;) rec = gl::add(gl::add(rec, rec), wire(bit_w + q));
                    f.add(gl::sub(rec, wire(base_w)));
                    // fold the list pair by pair, bit 0 first: item index bit q is decided by bit q.  Evaluated as a selection
                    // tree walked from the leaves without a per-thread array: level by level over the 2^bits items costs the same
                    // multiplications as plonky2's fold when done in place on a small register file of at most 64 items
                    u64 items[64];
                    for (u32 q = 0; q < vec; q++) items[q] = wire(base_w + 2 + q);
                    u32 len = vec;
                    for (u32 q = 0; q < bits; q++) {
                        const u64 b = wire(bit_w + q);
                        len >>= 1;
                        for (u32 v = 0; v < len; v++) items[v] = gl::add(items[2 * v], gl::mul(b, gl::sub(items[2 * v + 1], items[2 * v])));
                    }
                    f.add(gl::sub(items[0], wire(base_w + 1)));
                }
                for (u32 q = 0; q < extra; q++) f.add(gl::sub(gc[(u64)q * p.cs_stride], wire((2 + vec) * copies + q)));
                break;
            }
            case GATE_EXPONENTIATION: {                               // gates/exponentiation.rs
                const u32 nb = gd.p0;
                const u64 base = wire(0);
                u64 prev_inter = 1;
                for (u32 q = 0; q < nb; q++) {
                    const u64 prev = q == 0 ? 1 : gl::mul(prev_inter, prev_inter);
                    const u64 cur = wire(1 + (nb - 1 - q));
                    const u64 inter = wire(2 + nb + q);
                    f.add(gl::sub(gl::mul(prev, gl::add(gl::mul(cur, base), gl::sub(1, cur))), inter));
                    prev_inter = inter;
                }
                f.add(gl::sub(wire(1 + nb), prev_inter));
                break;
            }
            case GATE_POSEIDON_MDS: {                                 // gates/poseidon_mds.rs: the MDS layer, component by component
                u64 s0[12], s1[12];
                for (u32 q = 0; q < 12; q++) { s0[q] = wire(D * q); s1[q] = wire(D * q + 1); }
                mds_layer(s0);
                mds_layer(s1);
                for (u32 q = 0; q < 12; q++) {
                    f.add(gl::sub(wire(D * (12 + q)), s0[q]));
                    f.add(gl::sub(wire(D * (12 + q) + 1), s1[q]));
                }
                break;
            }
            case GATE_INTERPOLATION_HIGH_DEGREE:
            case GATE_INTERPOLATION_LOW_DEGREE: {                     // gates/interpolation.rs, low_degree_interpolation.rs
                // The coefficient wires are re-read from memory where they are used (not held: 2m words).  LowDegree uses its
                // power wires exactly where plonky2 does: off the trace the wires do not satisfy the power relations, so
                // recomputed powers would give different quotient values.
                const u32 m = 1u << gd.p0, w_coeffs = 5 + D * m, end_coeffs = w_coeffs + D * m;
                const bool low = gd.kind == GATE_INTERPOLATION_LOW_DEGREE;
                const u64 shift = wire(0), g_sub = root_of_unity(gd.p0);
                auto shift_pow = [&](u32 j) { return j == 0 ? (u64)1 : j == 1 ? shift : wire(end_coeffs + j - 2); };
                auto eval_pow = [&](u32 j) { return j == 1 ? ext(1 + D * m) : ext(end_coeffs + (m - 2) + D * (j - 2)); };
                if (low) {
#pragma unroll 1
                    for (u32 q = 2; q < m; q++) f.add(gl::sub(gl::mul(shift_pow(q - 1), shift), shift_pow(q)));
                }
                // value(i) - interpolant(shift g^i); LowDegree: with the coefficients c_j shift^j at the point g^i (Horner)
                u64 g_i = 1;
#pragma unroll 1
                for (u32 q = 0; q < m; q++) {
                    const u64 x_q = low ? g_i : gl::mul(shift, g_i);
                    E2 v{0, 0};
#pragma unroll 1
                    for (u32 j = m; j-- > 0;) {
                        const E2 c = low ? e2_scale(ext(w_coeffs + D * j), shift_pow(j)) : ext(w_coeffs + D * j);
                        v = e2_add(e2_scale(v, x_q), c);
                    }
                    const E2 r = e2_sub(ext(1 + D * q), v);
                    f.add(r.a); f.add(r.b);
                    g_i = gl::mul(g_i, g_sub);
                }
                // evaluation value - interpolant(evaluation point); LowDegree: c_0 + sum_j c_j eval_point^j with the power wires
                const E2 point = ext(1 + D * m);
                E2 v;
                if (low) {
                    E2 prev = point;
#pragma unroll 1
                    for (u32 q = 2; q < m; q++) {
                        const E2 cur = eval_pow(q), r = e2_sub(e2_mul(prev, point), cur);
                        f.add(r.a); f.add(r.b);
                        prev = cur;
                    }
                    v = ext(w_coeffs);
#pragma unroll 1
                    for (u32 j = 1; j < m; j++) v = e2_add(v, e2_mul(ext(w_coeffs + D * j), eval_pow(j)));
                } else {
                    v = E2{0, 0};
#pragma unroll 1
                    for (u32 j = m; j-- > 0;) v = e2_add(e2_mul(v, point), ext(w_coeffs + D * j));
                }
                const E2 r = e2_sub(ext(3 + D * m), v);
                f.add(r.a); f.add(r.b);
                break;
            }
            case GATE_U32_ARITHMETIC:
            case GATE_U32_ADD_MANY:
            case GATE_U32_SUBTRACTION: {                              // plonky2_u32 gates/{arithmetic,add_many,subtraction}_u32.rs
                // per op: the word equation (U32Arithmetic: the canonicity check first), the range of every limb from the top
                // one down, the limbs below 16 combined minus the low word, then the limbs above minus the high word
                // (U32Subtraction: borrow_out is a bit instead).  Limbs are read where they are used, never held.
                const u32 kind = gd.kind, a = gd.p0;
                const u32 ops = kind == GATE_U32_ADD_MANY ? gd.p1 : gd.p0;
                const u32 per = kind == GATE_U32_ARITHMETIC ? 6 : kind == GATE_U32_ADD_MANY ? a + 3 : 5;
                const u32 limbs = kind == GATE_U32_ARITHMETIC ? 2 * U32_LIMBS_PER_WORD : kind == GATE_U32_ADD_MANY ? U32_LIMBS_PER_WORD + 2 : U32_LIMBS_PER_WORD;
                const u64 two32 = (u64)1 << 32;
#pragma unroll 1
                for (u32 op = 0; op < ops; op++) {
                    const u32 w0 = per * op, l0 = per * ops + limbs * op;
                    u64 lo, hi;
                    if (kind == GATE_U32_ARITHMETIC) {
                        lo = wire(w0 + 3); hi = wire(w0 + 4);
                        f.add(gl::mul(gl::sub(gl::mul(wire(w0 + 5), gl::sub(0xFFFFFFFFull, hi)), 1), lo));
                        f.add(gl::sub(gl::add(gl::mul(hi, two32), lo), gl::add(gl::mul(wire(w0), wire(w0 + 1)), wire(w0 + 2))));
                    } else if (kind == GATE_U32_ADD_MANY) {
                        lo = wire(w0 + a + 1); hi = wire(w0 + a + 2);
                        u64 sum = wire(w0 + a);
#pragma unroll 1
                        for (u32 j = 0; j < a; j++) sum = gl::add(sum, wire(w0 + j));
                        f.add(gl::sub(gl::add(gl::mul(hi, two32), lo), sum));
                    } else {
                        lo = wire(w0 + 3); hi = wire(w0 + 4);
                        f.add(gl::sub(lo, gl::add(gl::sub(gl::sub(wire(w0), wire(w0 + 1)), wire(w0 + 2)), gl::mul(hi, two32))));
                    }
                    u64 comb_lo = 0, comb_hi = 0;
#pragma unroll 1
                    for (u32 j = limbs; j-- > 0;) {
                        const u64 l = wire(l0 + j);
                        f.add(limb_range(l));
                        if (j < U32_LIMBS_PER_WORD) comb_lo = gl::add(gl::mul(comb_lo, 4), l);
                        else comb_hi = gl::add(gl::mul(comb_hi, 4), l);
                    }
                    f.add(gl::sub(comb_lo, lo));
                    f.add(kind == GATE_U32_SUBTRACTION ? gl::mul(hi, gl::sub(1, hi)) : gl::sub(comb_hi, hi));
                }
                break;
            }
            case GATE_U32_RANGE_CHECK: {                              // plonky2_u32 gates/range_check_u32.rs
                const u32 nl = gd.p0;
#pragma unroll 1
                for (u32 q = 0; q < nl; q++) {
                    const u32 l0 = nl + U32_LIMBS_PER_WORD * q;
                    u64 comb = 0;
#pragma unroll 1
                    for (u32 j = U32_LIMBS_PER_WORD; j-- > 0;) comb = gl::add(gl::mul(comb, 4), wire(l0 + j));
                    f.add(gl::sub(comb, wire(q)));
#pragma unroll 1
                    for (u32 j = 0; j < U32_LIMBS_PER_WORD; j++) f.add(limb_range(wire(l0 + j)));
                }
                break;
            }
            case GATE_COMPARISON: {                                   // plonky2_u32 gates/comparison.rs
                const u32 nc = gd.p1, cb = comparison_chunk_bits(gd.p0, gd.p1);
                const u64 chunk_size = (u64)1 << cb;
                u64 first = 0, second = 0;
#pragma unroll 1
                for (u32 c = nc; c-- > 0;) {
                    first = gl::add(gl::mul(first, chunk_size), wire(4 + c));
                    second = gl::add(gl::mul(second, chunk_size), wire(4 + nc + c));
                }
                f.add(gl::sub(first, wire(0)));
                f.add(gl::sub(second, wire(1)));
                u64 msd = 0;                                          // the most significant difference so far
#pragma unroll 1
                for (u32 c = 0; c < nc; c++) {
                    const u64 x = wire(4 + c), y = wire(4 + nc + c);
                    u64 px = 1, py = 1;
#pragma unroll 1
                    for (u64 v = 0; v < chunk_size; v++) { px = gl::mul(px, gl::sub(x, v)); py = gl::mul(py, gl::sub(y, v)); }
                    f.add(px);
                    f.add(py);
                    const u64 diff = gl::sub(y, x), eq = wire(4 + 3 * nc + c), inter = wire(4 + 4 * nc + c);
                    f.add(gl::sub(gl::mul(diff, wire(4 + 2 * nc + c)), gl::sub(1, eq)));
                    f.add(gl::mul(eq, diff));
                    f.add(gl::sub(inter, gl::mul(eq, msd)));
                    msd = gl::add(inter, gl::mul(gl::sub(1, eq), diff));
                }
                const u64 msd_wire = wire(3);
                f.add(gl::sub(msd_wire, msd));
                u64 bits = 0;
#pragma unroll 1
                for (u32 b = 0; b <= cb; b++) {
                    const u64 bit = wire(4 + 5 * nc + b);
                    f.add(gl::mul(bit, gl::sub(1, bit)));
                    bits = gl::add(bits, gl::mul(bit, (u64)1 << b));
                }
                f.add(gl::sub(gl::add(chunk_size, msd_wire), bits));
                f.add(gl::sub(wire(2), wire(4 + 5 * nc + cb)));
                break;
            }
            default: break;
        }
        for (u32 a = 0; a < C; a++) acc[a] = gl::add(acc[a], gl::mul(filter, f.acc[a]));
    }
    for (u32 c = 0; c < C; c++) p.out[(u64)c * p.out_stride + i] = gl::mul(acc[c], zh_inv);
}

#ifndef B200ZKP_HOST_EMU
__global__ void __launch_bounds__(128)
quotient_values_kernel(const Params p) { quotient_point(p, (u64)blockIdx.x * blockDim.x + threadIdx.x); }
#endif

}  // namespace vanish
