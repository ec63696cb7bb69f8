// Openings (SURVEY.md section 8f, row N3, first piece): evaluate every polynomial of a batch at one point of the
// quadratic extension F_p[X]/(X^2 - 7).
//
// Replaces the evaluation loop of plonky2 `OpeningSet::new` / `eval_commitment`:
//     c.polynomials.par_iter().map(|p| p.to_extension().eval(z))          (plonky2/src/plonk/proof.rs, @ f99ed9c)
// with `QuadraticExtension<GoldilocksField>` arithmetic (field/src/extension/quadratic.rs, W = 7), reached from the
// reference through every prove() (e.g. /root/reference/src/rollup/circuits/mod.rs:1247).  The coefficients are already
// in HBM after the commitment, so the prover no longer has to copy 8nk bytes back just to open them.
//
// p(z) = sum_t z^t * Q_t(z^256),  Q_t(y) = sum_j c[256 j + t] y^j : thread t of a CTA runs Horner in y over its strided
// (coalesced) coefficients; columns are cut into segments so the grid fills the GPU; a second tiny kernel adds the
// segment partials  sum_s z^(s * seg_len) * P_s.
//
// One launch pair evaluates a list of entries e = (column, point): the whole of OpeningSet::new (every polynomial of four
// batches at zeta, the Zs at g zeta) is one list.  Without a table (entries == nullptr) entry e is the column
// base + e * col_stride at the point z0, which is what the one-batch, one-point callers pass by value.
#pragma once
#include "goldilocks.cuh"

namespace evalk {

using gl::u32;
using gl::u64;

struct Ext2 { u64 a, b; };   // a + b X, X^2 = 7, both canonical

GL_FN Ext2 ext_mul(Ext2 x, Ext2 y) {
    u64 t0 = gl::mul(x.a, y.a), t1 = gl::mul(x.b, y.b);
    u64 t2 = gl::mul(x.a, y.b), t3 = gl::mul(x.b, y.a);
    Ext2 r;
    r.a = gl::add(t0, gl::mul(t1, 7));
    r.b = gl::add(t2, t3);
    return r;
}
GL_FN Ext2 ext_add(Ext2 x, Ext2 y) { Ext2 r; r.a = gl::add(x.a, y.a); r.b = gl::add(x.b, y.b); return r; }
GL_FN Ext2 ext_pow(Ext2 x, u64 e) {
    Ext2 r; r.a = 1; r.b = 0;
    while (e) { if (e & 1) r = ext_mul(r, x); x = ext_mul(x, x); e >>= 1; }
    return r;
}

static constexpr int EVAL_THREADS = 256;

struct EvalEntry { const u64* col; u64 point; };   // a column of n coefficients and the index of its point

#ifndef B200ZKP_HOST_EMU
struct EvalList {
    const EvalEntry* entries;   // nullptr: column base + e * col_stride at z0
    const Ext2* points;
    const u64* base;
    u64 col_stride;
    Ext2 z0;
};

GL_FN void eval_entry(const EvalList& L, u64 e, const u64** col, Ext2* z) {
    if (L.entries) { const EvalEntry en = L.entries[e]; *col = en.col; *z = L.points[en.point]; }
    else { *col = L.base + e * L.col_stride; *z = L.z0; }
}

// grid (segments, entries); partial[e][seg] = sum_{i in segment} c[i] z^(i - seg_start)
__global__ void __launch_bounds__(EVAL_THREADS)
eval_segments_kernel(EvalList L, u64 n, u64 seg_len, Ext2* __restrict__ partial) {
    __shared__ Ext2 red[EVAL_THREADS];
    const u32 t = threadIdx.x;
    const u64 seg = blockIdx.x, e = blockIdx.y;
    const u64 i0 = seg * seg_len;
    const u64 i1 = (i0 + seg_len < n) ? i0 + seg_len : n;
    const u64* c;
    Ext2 z;
    eval_entry(L, e, &c, &z);
    const Ext2 y = ext_pow(z, EVAL_THREADS);
    // this thread's coefficients: i0 + t, i0 + t + 256, ...; Horner from the top
    Ext2 acc; acc.a = 0; acc.b = 0;
    if (i0 + t < i1) {
        u64 cnt = (i1 - i0 - t + EVAL_THREADS - 1) / EVAL_THREADS;
        for (u64 j = cnt; j-- > 0;) {
            acc = ext_mul(acc, y);
            acc.a = gl::add(acc.a, gl::canon(c[i0 + t + j * EVAL_THREADS]));
        }
        acc = ext_mul(acc, ext_pow(z, t));
    }
    red[t] = acc;
    __syncthreads();
    for (u32 s = EVAL_THREADS / 2; s > 0; s >>= 1) {
        if (t < s) red[t] = ext_add(red[t], red[t + s]);
        __syncthreads();
    }
    if (t == 0) partial[e * gridDim.x + seg] = red[0];
}

// out[e] = sum_s z_e^(s * seg_len) * partial[e][s]
__global__ void eval_combine_kernel(EvalList L, const Ext2* __restrict__ partial, u32 n_seg, u64 seg_len, u32 m, Ext2* __restrict__ out) {
    u32 e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const u64* c;
    Ext2 z;
    eval_entry(L, e, &c, &z);
    Ext2 step = ext_pow(z, seg_len);
    Ext2 acc; acc.a = 0; acc.b = 0;
    for (u32 s = n_seg; s-- > 0;) acc = ext_add(ext_mul(acc, step), partial[(u64)e * n_seg + s]);
    out[e] = acc;
}
#endif

}  // namespace evalk
