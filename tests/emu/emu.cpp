// TEST HARNESS (not product): compiles the CUDA kernel bodies of intmax_zkp_core_b200/csrc with g++ under
// B200ZKP_HOST_EMU and steps the "threads" of each CTA in a loop, so the index logic of the NTT passes, the
// Poseidon permutation arithmetic and the digest layout can be checked on a machine without a GPU.
// The product library never defines B200ZKP_HOST_EMU and has no CPU path.
#define B200ZKP_HOST_EMU 1
#define __restrict__
#include <cstring>
#include <vector>

#include "../../intmax_zkp_core_b200/csrc/merkle_kernels.cuh"
#include "../../intmax_zkp_core_b200/csrc/perm_kernels.cuh"
#include "../../intmax_zkp_core_b200/csrc/vanishing_kernels.cuh"
#include "../../intmax_zkp_core_b200/csrc/host_plan.hpp"

using gl::u32;
using gl::u64;

static void run_pass(const ntt::PassParams& p, u32 B, u32 n_blk) {
    u64 T = (u64)ntt::tile_elems_for((int)B) >> B;
    u64 total_batches = (u64)p.ncols << (p.n_log - B);
    u64 blocks = (total_batches + T - 1) / T;
    for (u32 y = 0; y < n_blk; y++)
        for (u64 blk = 0; blk < blocks; blk++) {
#define EMU_PASS(BB)                                                                                           \
    case BB:                                                                                                   \
        switch (ntt::pass_mode(p)) {                                                                           \
            case ntt::MODE_MID_NATURAL: ntt::pass_body<BB, ntt::MODE_MID_NATURAL>(p, (u32)blk, y); break;      \
            case ntt::MODE_MID_BITREV: ntt::pass_body<BB, ntt::MODE_MID_BITREV>(p, (u32)blk, y); break;        \
            case ntt::MODE_FINAL_BITREV: ntt::pass_body<BB, ntt::MODE_FINAL_BITREV>(p, (u32)blk, y); break;    \
            default: ntt::pass_body<BB, ntt::MODE_FINAL_NATURAL>(p, (u32)blk, y); break;                       \
        }                                                                                                      \
        break;
            switch (B) { EMU_PASS(1) EMU_PASS(2) EMU_PASS(3) EMU_PASS(4) EMU_PASS(5) EMU_PASS(6) EMU_PASS(7) EMU_PASS(8) EMU_PASS(9) EMU_PASS(10) }
#undef EMU_PASS
        }
}

struct Tables {
    std::vector<u64> w[2][ntt::MAX_PASS_BITS + 1];
    Tables() { for (int d = 0; d < 2; d++) for (u32 B = 1; B <= (u32)ntt::MAX_PASS_BITS; B++) w[d][B] = hostgl::small_root_table(B, d); }
};
static Tables g_tab;

// host replicas of the device table builders (build_twiddle_image_kernel / build_powers_kernel)
static std::vector<u64> twiddle_image(u32 n_log, int dir, bool bitrev_pos, const ntt::TwiddleImageShape& sh, u64 f) {
    u64 w = hostgl::root(n_log);
    if (dir) w = hostgl::inv(w);
    u64 count = (u64)1 << (sh.B + sh.C_log);
    std::vector<u64> img(count);
    for (u64 i = 0; i < count; i++) {
        u32 pos = (u32)(i >> sh.C_log);
        u64 c = i & (((u64)1 << sh.C_log) - 1);
        u32 k1 = bitrev_pos ? hostgl::bitrev(pos, sh.B) : pos;
        u64 t = hostgl::pw(w, (c * k1) << sh.shift);
        img[i] = f ? hostgl::mul(t, f) : t;
    }
    return img;
}

// scale_bases: one shift per block (nullptr: no scaling)
static void transform(const u64* in, u64 in_stride, u64* out, u64 out_stride, u64* scratch, u32 n_log, u32 ncols,
                      int dir, bool bitrev_out, const std::vector<u64>* scale_bases, bool inverse_scale,
                      u32 n_blk = 1, u64 out_blk_stride = 0) {
    if (n_log == 0) {
        for (u32 y = 0; y < n_blk; y++)
            for (u32 c = 0; c < ncols; c++) out[y * out_blk_stride + c * out_stride] = gl::canon(in[c * in_stride]);
        return;
    }
    u64 n = (u64)1 << n_log;
    u64* wt[ntt::MAX_PASS_BITS + 1];
    for (u32 B = 0; B <= (u32)ntt::MAX_PASS_BITS; B++) wt[B] = B ? g_tab.w[dir][B].data() : nullptr;
    ntt::TwiddleImageShape shapes[ntt::MAX_PASSES];
    u32 n_img = ntt::twiddle_images(n_log, shapes);
    u64 n_inv = hostgl::inv(n % hostgl::P);
    std::vector<std::vector<u64>> imgs(n_img);
    ntt::TransformTables tb{};
    tb.wtab = wt;
    for (u32 i = 0; i < n_img; i++) {
        imgs[i] = twiddle_image(n_log, dir, bitrev_out, shapes[i], (dir == 1 && i == 0) ? n_inv : 0);
        tb.twimg[i] = imgs[i].data();
    }
    std::vector<u64> sc;
    if (scale_bases) {
        sc.resize((size_t)n * scale_bases->size());
        for (size_t y = 0; y < scale_bases->size(); y++) {
            u64 x = 1;
            for (u64 i = 0; i < n; i++) { sc[y * n + i] = x; x = hostgl::mul(x, (*scale_bases)[y]); }
        }
        tb.scale = sc.data();
        tb.scale_blk_stride = n;
    }
    ntt::Plan plan;
    ntt::make_plan(&plan, in, in_stride, out, out_stride, scratch, n_log, ncols, tb, bitrev_out,
                   inverse_scale ? n_inv : 0, true, 0, out_blk_stride);
    for (u32 pi = 0; pi < plan.n_passes; pi++) run_pass(plan.pass[pi], plan.bits[pi], n_blk);
}

// ---- second-generation passes (ntt_ct_kernels.cuh): the thread bodies stepped on the host (generic staging path; the TMA
// staging of the device build moves the same [row][T] image)
static void run_ct_pass(const ntc::PassParams& p, u32 B, int kind, u64 grid) {
    static std::vector<u64> smem(16 * 1024);
    for (u64 bid = 0; bid < grid; bid++) {
#define EMU_CT(BB)                                                                                                       \
    case BB:                                                                                                             \
        if (kind == ntc::KIND_STRIDED) ntc::strided_body<BB, false, int>(p, nullptr, nullptr, smem.data(), (u32)bid);     \
        else if (kind == ntc::KIND_STRIDED_LOOP) ntc::strided_body<BB, true, int>(p, nullptr, nullptr, smem.data(), (u32)bid); \
        else if (kind == ntc::KIND_PULL_LOOP) ntc::strided_body<BB, true, int, true>(p, nullptr, nullptr, smem.data(), (u32)bid); \
        else if (kind == ntc::KIND_FINAL_INPLACE) ntc::final_body<BB, false>(p, smem.data(), (u32)bid);                  \
        else ntc::final_body<BB, true>(p, smem.data(), (u32)bid);                                                        \
        break;
        switch (B) { EMU_CT(5) EMU_CT(6) EMU_CT(7) EMU_CT(8) }
#undef EMU_CT
    }
}

extern "C" {
// values [k][n] -> coeffs [k][n] through the block-twiddle passes; returns 0 when this generation does not cover n_log
int emu_ct_intt(const u64* in, u64* out, u32 n_log, u32 k) {
    u64 n = (u64)1 << n_log;
    u64 n_inv = hostgl::inv(n % hostgl::P);
    if (!ntc::covers(n_log)) return 0;
    std::vector<u64> z = ntc::ztab_host(n_log, 1, 1, n_inv), scratch((size_t)k * n);
    std::vector<u64> zf = ntc::zfinal_host(n_log, z, true);
    z.resize(ntc::ztab_entries(n_log));
    ntc::Plan plan;
    if (!ntc::make_plan(&plan, in, n, out, n, scratch.data(), n_log, k, 1, 0, true, z.data(), zf.data(), n_inv, false)) return 0;
    for (u32 pi = 0; pi < plan.n_passes; pi++) run_ct_pass(plan.pass[pi], plan.bits[pi], plan.kind[pi], plan.grid[pi]);
    return 1;
}
// coeffs [k][n] -> leaves of coset blocks [b0, b1) of every column, [k][(b1 - b0) * n] in leaf order
int emu_ct_lde(const u64* coeffs, u64* lde, u32 n_log, u32 k, u32 rate_bits, u32 b0, u32 b1) {
    u64 n = (u64)1 << n_log;
    if (!ntc::covers(n_log)) return 0;
    std::vector<u64> z, zf;
    for (u32 b = b0; b < b1; b++) {
        std::vector<u64> zb = ntc::ztab_host(n_log, hostgl::coset_shift_of_block(n_log, rate_bits, b), 0, 0);
        std::vector<u64> fb = ntc::zfinal_host(n_log, zb, false);
        z.insert(z.end(), zb.begin(), zb.begin() + ntc::ztab_entries(n_log));
        zf.insert(zf.end(), fb.begin(), fb.end());
    }
    ntc::Plan plan;
    if (!ntc::make_plan(&plan, coeffs, n, lde, (u64)(b1 - b0) * n, nullptr, n_log, k, b1 - b0, n, false, z.data(), zf.data(), 0, false)) return 0;
    for (u32 pi = 0; pi < plan.n_passes; pi++) run_ct_pass(plan.pass[pi], plan.bits[pi], plan.kind[pi], plan.grid[pi]);
    return 1;
}
// partitioned LDE (sharded.inl): the k columns are dealt to G ranks in groups of G * w (column c: rank (c % (G w)) / w, local
// column (c / (G w)) * w + c % w; src[q] = rank q's local columns, [.][n]).  sel = 0: physical columns [col0, col0 + count);
// sel = 1: the first `count` columns of rank src_rank from group col0 / (G w) on.  pull: gathered from src into coeffs_copy
// [k][n] on the way; else read from coeffs_copy.  Coset blocks [b0, b1) into lde [k][(b1 - b0) * n].
int emu_ct_lde_cols(const u64* const* src, u32 G, u32 w, u32 k, u32 col0, u32 count, u32 sel, u32 src_rank, int pull, u64* coeffs_copy,
                    u64* lde, u32 n_log, u32 rate_bits, u32 b0, u32 b1) {
    u64 n = (u64)1 << n_log;
    if (!ntc::covers(n_log)) return 0;
    std::vector<u64> z, zf;
    for (u32 b = b0; b < b1; b++) {
        std::vector<u64> zb = ntc::ztab_host(n_log, hostgl::coset_shift_of_block(n_log, rate_bits, b), 0, 0);
        std::vector<u64> fb = ntc::zfinal_host(n_log, zb, false);
        z.insert(z.end(), zb.begin(), zb.begin() + ntc::ztab_entries(n_log));
        zf.insert(zf.end(), fb.begin(), fb.end());
    }
    ntc::ColumnSet cs;
    cs.run = w; cs.period = G * w; cs.col0 = col0; cs.limit = k; cs.count = count; cs.sel = sel; cs.src_rank = src_rank; cs.pull = pull != 0;
    for (u32 q = 0; q < G && q < (u32)ntc::MAX_SRC; q++) cs.src[q] = src[q];
    cs.src_col_stride = n; cs.copy_out = coeffs_copy; cs.copy_col_stride = n;
    ntc::Plan plan;
    if (!ntc::make_plan(&plan, coeffs_copy, n, lde, (u64)(b1 - b0) * n, nullptr, n_log, 0, b1 - b0, n, false, z.data(), zf.data(), 0, false, &cs)) return 0;
    for (u32 pi = 0; pi < plan.n_passes; pi++) run_ct_pass(plan.pass[pi], plan.bits[pi], plan.kind[pi], plan.grid[pi]);
    return 1;
}
// the plan the library makes (use_tma asked for) for an inverse transform (natural_out) or an LDE of n_blk coset blocks with
// columns out_stride apart, over 16-byte aligned buffers it never touches: -1 when make_plan refuses it, else bit pi set when
// pass pi keeps TMA staging
int emu_ct_plan_tma(u32 n_log, u32 k, u64 out_stride, u32 n_blk, int natural_out) {
    alignas(16) static u64 in[2], out[2], scratch[2], ztab[2], zfinal[2];
    const u64 n = (u64)1 << n_log;
    ntc::Plan plan;
    if (!ntc::make_plan(&plan, in, n, out, out_stride, natural_out ? scratch : nullptr, n_log, k, n_blk, natural_out ? 0 : n,
                        natural_out != 0, ztab, zfinal, 0, true))
        return -1;
    int mask = 0;
    for (u32 pi = 0; pi < plan.n_passes; pi++) if (plan.pass[pi].use_tma) mask |= 1 << pi;
    return mask;
}
// row N1b: vanish::quotient_point stepped over every leaf of the quotient coset; LDEs [columns][Q] in leaf order,
// gates: n_gates x (kind, selector_index, group_begin, group_end, p0, p1, p2); out [C][Q] natural order
void emu_quotient_values(const u64* cs, const u64* wires, const u64* zpp, u32 n_log, u32 q_bits, u32 num_selectors, u32 C, u32 degree,
                         const u32* gates, u32 n_gates, const u64* k_is, const u64* betas, const u64* gammas, const u64* alphas,
                         const u64* pi_hash, u64* out) {
    vanish::Params p{};
    const u32 R = 80, Q_log = n_log + q_bits;
    const u64 Q = (u64)1 << Q_log, n = (u64)1 << n_log;
    p.cs = cs; p.wires = wires; p.zpp = zpp; p.cs_stride = p.wires_stride = p.zpp_stride = Q;
    p.n_log = n_log; p.q_bits = q_bits; p.num_selectors = num_selectors; p.num_gate_consts = 2; p.num_routed = R;
    p.num_challenges = C; p.degree = degree; p.num_prods = (R + degree - 1) / degree - 1; p.n_gates = n_gates;
    u32 max_c = 0;
    for (u32 i = 0; i < n_gates; i++) {
        const u32* gi = gates + 7 * i;
        p.gates[i] = vanish::GateDesc{gi[0], gi[1], gi[2], gi[3], gi[4], gi[5], gi[6]};
        const u32 nc = vanish::gate_num_constraints(gi[0], R, 2, gi[4], gi[5], gi[6]);
        if (nc > max_c) max_c = nc;
    }
    p.n_terms = C + C * (p.num_prods + 1) + max_c;
    std::vector<u64> apw((size_t)C * p.n_terms), zh(1u << q_bits), zhi(1u << q_bits), lo, hi;
    for (u32 c = 0; c < C; c++) { u64 x = 1; for (u32 t = 0; t < p.n_terms; t++) { apw[(size_t)c * p.n_terms + t] = x; x = hostgl::mul(x, alphas[c]); } p.betas[c] = betas[c]; p.gammas[c] = gammas[c]; }
    const u64 shift_n = hostgl::pw(7, n), wq = q_bits ? hostgl::root(q_bits) : 1;
    u64 wp = 1;
    for (u32 i = 0; i < (1u << q_bits); i++) { { const u64 xn = hostgl::mul(shift_n, wp); zh[i] = xn ? xn - 1 : hostgl::P - 1; } zhi[i] = hostgl::inv(zh[i]); wp = hostgl::mul(wp, wq); }
    p.tw_lo_bits = hostgl::two_level_powers(hostgl::root(Q_log), Q_log, &lo, &hi);
    p.tw_lo = lo.data(); p.tw_hi = hi.data();
    for (int i = 0; i < 4; i++) p.pi_hash[i] = pi_hash[i];
    p.k_is = k_is; p.alpha_pows = apw.data(); p.zh = zh.data(); p.zh_inv = zhi.data();
    p.n_inv = hostgl::inv(n % hostgl::P);
    p.out = out; p.out_stride = Q;
    for (u64 t = 0; t < Q; t++) vanish::quotient_point(p, t);
}
u64 emu_inverse(u64 x) { return perm::inverse(x); }
// rows of the permutation argument (perm::row_chunk_products): running[(c * chunks + l) * n + i]
void emu_perm_rows(const u64* wires, const u64* sigmas, const u64* k_is, const u64* betas, const u64* gammas, u32 n_log, u32 R,
                   u32 degree, u32 C, u64* running) {
    perm::Params p;
    p.n = (u64)1 << n_log;
    p.wires = wires; p.wires_stride = p.n; p.sigmas = sigmas; p.sigmas_stride = p.n;
    p.k_is = k_is; p.betas = betas; p.gammas = gammas; p.omega = hostgl::root(n_log);
    p.R = R; p.degree = degree; p.chunks = (R + degree - 1) / degree; p.C = C;
    for (u32 c = 0; c < C; c++)
        for (u64 i = 0; i < p.n; i++) perm::row_chunk_products(p, i, c, running);
}
void emu_permute(u64* s) { u64 t[12]; memcpy(t, s, sizeof t); poseidon::permute(t); memcpy(s, t, sizeof t); }
void emu_sponge(const u64* leaf, u64 col_stride, u32 len, u32 noop_short, u64* out4) {
    u64 s[12];
    merkle::sponge_leaf(leaf, col_stride, len, noop_short, s);
    memcpy(out4, s, 32);
}
// the sponge of one leaf absorbed in pieces cut at `cuts` (multiples of the rate), the state carried between the pieces
void emu_sponge_pieces(const u64* leaf, u64 col_stride, u32 len, const u32* cuts, u32 n_cuts, u64* out4) {
    u64 s[12] = {0};
    u32 begin = 0;
    for (u32 i = 0; i <= n_cuts; i++) {
        const u32 end = i < n_cuts ? cuts[i] : len;
        u64 carried[12];
        memcpy(carried, s, sizeof s);       // (what leaf_absorb_kernel stores and reloads)
        memcpy(s, carried, sizeof s);
        merkle::sponge_absorb(leaf, col_stride, begin, end, s);
        begin = end;
    }
    memcpy(out4, s, 32);
}
u64 emu_node_slot(u32 sub_log, u64 subtree, u32 layer, u64 m) {
    merkle::TreeShape t; t.sub_log = sub_log; t.sub_digests = 2 * (((u64)1 << sub_log) - 1);
    return merkle::node_slot(t, subtree, layer, m);
}
// values [k][n] -> coeffs [k][n]
void emu_intt(const u64* in, u64* out, u32 n_log, u32 k) {
    u64 n = (u64)1 << n_log;
    std::vector<u64> scratch((size_t)k * n);
    transform(in, n, out, n, scratch.data(), n_log, k, 1, false, nullptr, true);
}
void emu_ntt(const u64* in, u64* out, u32 n_log, u32 k) {
    u64 n = (u64)1 << n_log;
    std::vector<u64> scratch((size_t)k * n);
    transform(in, n, out, n, scratch.data(), n_log, k, 0, false, nullptr, false);
}
// coeffs [k][n] -> lde [k][N] in leaf order
void emu_lde(const u64* coeffs, u64* lde, u32 n_log, u32 k, u32 rate_bits) {
    u64 n = (u64)1 << n_log, N = n << rate_bits;
    std::vector<u64> bases;
    for (u32 b = 0; b < (1u << rate_bits); b++) bases.push_back(hostgl::coset_shift_of_block(n_log, rate_bits, b));
    // all coset blocks in one "launch" per pass, exactly as the library does (blockIdx.y = block)
    transform(coeffs, n, lde, N, nullptr, n_log, k, 0, true, &bases, false, 1u << rate_bits, n);
}
}
