// C ABI implementation (include/b200zkp.h): contexts, twiddle caches, pass scheduling, handles.
// Product code: no CPU fallback, nothing from oracle/ is included, linked or executed here.
#include "../../include/b200zkp.h"
#include "../../include/b200zkp_test.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <optional>
#include <string>
#include <tuple>
#include <vector>

#include "merkle_kernels.cuh"
#include "ntt_kernels.cuh"
#include "eval_kernels.cuh"
#include "fri_kernels.cuh"
#include "perm_kernels.cuh"
#include "vanishing_kernels.cuh"
#include "random_kernels.cuh"
#include "host_plan.hpp"

using gl::u32;
using gl::u64;

// ------------------------------------------------------------------------------------------------
static inline u64 gl_host_canon(u64 a) { return a >= hostgl::P ? a - hostgl::P : a; }

struct TwoLevel {
    u64* lo = nullptr;
    u64* hi = nullptr;
    u32 lo_bits = 0;
};

struct b200zkp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::mutex mu;
    std::string err;
    u64 launches = 0;
    u64* wtab[2][ntt::MAX_PASS_BITS + 1] = {};          // [dir][B] w_{2^B}^(+-e)
    std::map<u32, TwoLevel> tw[2];                      // [dir][n_log] -> w_n^(+-e)
    // direct tables read by the pass kernels
    struct Images { const u64* img[ntt::MAX_PASSES] = {}; };
    std::map<std::tuple<u32, int, bool>, Images> twimg; // (n_log, dir, bitrev_out) -> twiddle image per pass
    std::map<std::pair<u32, u32>, const u64*> coset_scale;   // (n_log, rate_bits) -> [2^rate_bits][n] shift powers
    std::map<std::pair<u64, u32>, const u64*> power_scale;   // (shift, bits) -> shift^i, i < 2^bits (coset transforms)
    // second-generation passes (ntt_ct_kernels.cuh): block-twiddle tables Z, [n_blk][n] each
    struct ZTables { const u64* strided = nullptr; const u64* final_ = nullptr; };   // see ntc::ztab_entries / zfinal_words
    std::map<std::pair<u32, u32>, ZTables> ztab_lde;    // (n_log, rate_bits) -> forward transform on every leaf block's coset
    std::map<u32, ZTables> ztab_inv;                    // n_log -> inverse transform (s = 1), last level carries n^-1
    u32 ct_smem_set = 0;                                // kernels whose dynamic shared memory limit has been raised on this device
    u32 sm_count = 0;                                   // (queried on first use)
    // mailbox: 64 KB of mapped pinned host memory the small host-buffer calls (single hashes, the Fiat-Shamir transcript)
    // read and write directly from the kernel: no cudaMemcpy on those paths, one launch + one stream synchronise per call
    void* mailbox = nullptr;
    void* mailbox_dev = nullptr;
    u64* round_add = nullptr;                           // poseidon_tables::ROUND_ADD in global memory (latency-form kernels)
    std::multimap<size_t, void*> pool;                  // cached device allocations (DevBuf::reset), at most pool_max_bytes
    size_t pool_bytes = 0;
    size_t live_bytes = 0;                              // handed out by DevBuf::alloc and not yet returned (b200zkp_ctx_buffer_bytes)
    size_t pool_max_bytes = (size_t)16 << 30;         // reset to 1/8 of the device memory in ctx_create
    std::vector<void*> table_allocs;                    // the cached tables above and round_add, freed with the ctx
    // second, higher-priority stream: host uploads and copy-back beside the main stream (ensure_stream2)
    cudaStream_t stream2 = nullptr;
    std::vector<cudaEvent_t> sync_events;
    // optional per-stage timing (bench.py): CUDA event pairs recorded on the ctx stream
    bool timing = false;
    std::vector<cudaEvent_t> ev_free;
    struct Span { int stage; cudaEvent_t a, b; };
    std::vector<Span> spans;
};

struct StageTimer {
    b200zkp_ctx* c;
    int stage;
    cudaEvent_t a = nullptr;
    static cudaEvent_t get(b200zkp_ctx* c) {
        cudaEvent_t e = nullptr;
        if (!c->ev_free.empty()) { e = c->ev_free.back(); c->ev_free.pop_back(); }
        else if (cudaEventCreate(&e) != cudaSuccess) { (void)cudaGetLastError(); e = nullptr; }
        return e;
    }
    StageTimer(b200zkp_ctx* ctx, int st) : c(ctx), stage(st) {
        if (c->timing && (a = get(c))) cudaEventRecord(a, c->stream);
    }
    ~StageTimer() {
        if (!a) return;
        cudaEvent_t b = get(c);
        if (b) { cudaEventRecord(b, c->stream); c->spans.push_back({stage, a, b}); }
        else c->ev_free.push_back(a);
    }
};

struct Guard {
    b200zkp_ctx* c;
    explicit Guard(b200zkp_ctx* ctx) : c(ctx) { c->mu.lock(); cudaSetDevice(c->device); }
    ~Guard() { c->mu.unlock(); }
};

// Sets ctx->stream for the life of the scope and puts the previous stream back on every exit.
struct StreamScope {
    b200zkp_ctx* c;
    cudaStream_t saved;
    StreamScope(b200zkp_ctx* ctx, cudaStream_t s) : c(ctx), saved(ctx->stream) { c->stream = s; }
    ~StreamScope() { c->stream = saved; }
};

// (clears the thread's last error, so that a failure is reported by its own call only)
#define CUDA_TRY(ctx, expr)                                                                   \
    do {                                                                                      \
        cudaError_t e__ = (expr);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                 \
            (void)cudaGetLastError();                                                         \
            return e__ == cudaErrorMemoryAllocation ? B200ZKP_ERR_OOM : B200ZKP_ERR_CUDA;     \
        }                                                                                     \
    } while (0)
#define TRY(expr) do { int rc__ = (expr); if (rc__ != 0) return rc__; } while (0)
#define BAD(ctx, msg) do { (ctx)->err = (msg); return B200ZKP_ERR_BAD_ARG; } while (0)
#define LAUNCH_CHECK(ctx) do { (ctx)->launches++; CUDA_TRY(ctx, cudaGetLastError()); } while (0)

static void pool_drop(b200zkp_ctx* ctx) {
    for (auto& kv : ctx->pool) cudaFree(kv.second);
    ctx->pool.clear();
    ctx->pool_bytes = 0;
}

// One pooled device allocation, returned to the ctx's cache when its owner goes away; take the ctx lock around both.
// A returned buffer may be handed to later work on ctx->stream without a synchronisation, so a buffer that another stream
// touched (stream2, the communicator's side or hash stream, NCCL) must have that stream drained or joined into ctx->stream
// before its owner is destroyed.
class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : ctx_(o.ctx_), p_(o.p_), bytes_(o.bytes_) { o.p_ = nullptr; o.bytes_ = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { reset(); ctx_ = o.ctx_; p_ = o.p_; bytes_ = o.bytes_; o.p_ = nullptr; o.bytes_ = 0; }
        return *this;
    }
    ~DevBuf() { reset(); }

    u64* get() const { return (u64*)p_; }
    size_t bytes() const { return bytes_; }

    // 0 bytes: nullptr and success
    int alloc(b200zkp_ctx* ctx, size_t bytes) {
        reset();
        ctx_ = ctx;
        if (bytes == 0) return 0;
        void* p = nullptr;
        auto it = ctx->pool.find(bytes);
        if (it != ctx->pool.end()) {
            p = it->second; ctx->pool_bytes -= it->first; ctx->pool.erase(it);
        } else {
            cudaError_t e = cudaMalloc(&p, bytes);
            if (e == cudaErrorMemoryAllocation) {
                // drop the cache and retry once
                (void)cudaGetLastError();
                pool_drop(ctx);
                e = cudaMalloc(&p, bytes);
            }
            if (e != cudaSuccess) {
                ctx->err = std::string("cudaMalloc: ") + cudaGetErrorString(e);
                (void)cudaGetLastError();
                return e == cudaErrorMemoryAllocation ? B200ZKP_ERR_OOM : B200ZKP_ERR_CUDA;
            }
        }
        p_ = p; bytes_ = bytes;
        ctx->live_bytes += bytes;
        return 0;
    }
    // grows only (the contents are not kept)
    int ensure(b200zkp_ctx* ctx, size_t bytes) { return bytes_ >= bytes ? 0 : alloc(ctx, bytes); }

    void reset() {
        if (!p_) return;
        ctx_->live_bytes -= bytes_;
        // cached for the next request of the same size; an opening proof cycles through ~40 distinct sizes.  The cache is
        // capped by bytes so that a freed 2^20 x 135 batch (10.7 GB) goes back to the driver instead of starving torch or a
        // second ctx on the same GPU; b200zkp_ctx_trim empties it on request
        if (ctx_->pool.size() < 256 && ctx_->pool_bytes + bytes_ <= ctx_->pool_max_bytes) {
            ctx_->pool.emplace(bytes_, p_);
            ctx_->pool_bytes += bytes_;
        } else {
            cudaFree(p_);    // (cudaFree synchronises the device: pending work on the buffer has finished when it returns)
        }
        p_ = nullptr; bytes_ = 0;
    }

  private:
    b200zkp_ctx* ctx_ = nullptr;
    void* p_ = nullptr;
    size_t bytes_ = 0;
};

struct b200zkp_batch {
    b200zkp_ctx* ctx;
    u32 n_log, k, rate_bits, cap_height, salt;
    DevBuf coeffs, lde, digests, cap;
};

struct b200zkp_tree {
    b200zkp_ctx* ctx;
    u64 n_leaves;
    u32 leaf_len, cap_height;
    DevBuf digests, cap;
};

static int d2h(b200zkp_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!bytes) return 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
static int h2d(b200zkp_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!bytes) return 0;
    CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

// the second stream of the ctx, created on first use at the highest priority
static int ensure_stream2(b200zkp_ctx* ctx) {
    if (ctx->stream2) return 0;
    int lo = 0, hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, hi) != cudaSuccess) {
        (void)cudaGetLastError();
        ctx->stream2 = nullptr;
        ctx->err = "cannot create the copy stream";
        return B200ZKP_ERR_CUDA;
    }
    return 0;
}

// *lg = log2(n); false unless n is a power of two
static bool log2_exact(u64 n, u32* lg) {
    if (n == 0 || (n & (n - 1))) return false;
    u32 l = 0;
    while (((u64)1 << l) < n) l++;
    *lg = l;
    return true;
}

// device memory kept for the life of the ctx
static int table_alloc(b200zkp_ctx* ctx, u64 count, u64** out) {
    CUDA_TRY(ctx, cudaMalloc((void**)out, count * sizeof(u64)));
    ctx->table_allocs.push_back(*out);
    return 0;
}

static int upload(b200zkp_ctx* ctx, const std::vector<u64>& h, u64** d) {
    TRY(table_alloc(ctx, h.size(), d));
    TRY(h2d(ctx, *d, h.data(), h.size() * sizeof(u64)));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// *out = the table cached under `key`, built by build(&table) on first use (a failed build caches nothing)
template <typename Map, typename Build>
static int get_or_build(Map& cache, const typename Map::key_type& key, typename Map::mapped_type* out, Build build) {
    auto it = cache.find(key);
    if (it == cache.end()) {
        typename Map::mapped_type t{};
        TRY(build(&t));
        it = cache.emplace(key, t).first;
    }
    *out = it->second;
    return 0;
}

static int get_tw(b200zkp_ctx* ctx, int dir, u32 n_log, TwoLevel* out) {
    return get_or_build(ctx->tw[dir], n_log, out, [&](TwoLevel* t) -> int {
        const u64 w = hostgl::root(n_log);
        std::vector<u64> lo, hi;
        t->lo_bits = hostgl::two_level_powers(dir ? hostgl::inv(w) : w, n_log, &lo, &hi);
        TRY(upload(ctx, lo, &t->lo));
        return upload(ctx, hi, &t->hi);
    });
}

// dst[i] = base^i, i < 2^bits.  The two-level input lives only for the build: the stream is synchronised before it goes
// back to the pool, so the build is safe on whichever stream ctx->stream is.
static int fill_powers(b200zkp_ctx* ctx, u64 base, u32 bits, u64* dst) {
    std::vector<u64> lo, hi;
    const u32 lo_bits = hostgl::two_level_powers(base, bits, &lo, &hi);
    DevBuf d_lo, d_hi;
    TRY(d_lo.alloc(ctx, lo.size() * 8));
    TRY(d_hi.alloc(ctx, hi.size() * 8));
    TRY(h2d(ctx, d_lo.get(), lo.data(), d_lo.bytes()));
    TRY(h2d(ctx, d_hi.get(), hi.data(), d_hi.bytes()));
    const u64 n = (u64)1 << bits;
    ntt::build_powers_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dst, n, d_lo.get(), d_hi.get(), lo_bits);
    LAUNCH_CHECK(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// powers shift^i, i < 2^bits (scale table of a coset transform)
static int get_power_scale(b200zkp_ctx* ctx, u64 shift, u32 bits, const u64** out) {
    return get_or_build(ctx->power_scale, std::make_pair(shift, bits), out, [&](const u64** t) -> int {
        u64* d = nullptr;
        TRY(table_alloc(ctx, (u64)1 << bits, &d));
        *t = d;
        return fill_powers(ctx, shift, bits, d);
    });
}

// [2^rate_bits][n]: row b holds the powers of the coset shift of leaf block b, s_b = 7 * w_N^bitrev(b, rate_bits)
static int get_coset_scale(b200zkp_ctx* ctx, u32 n_log, u32 rate_bits, const u64** out) {
    return get_or_build(ctx->coset_scale, std::make_pair(n_log, rate_bits), out, [&](const u64** t) -> int {
        const u64 n = (u64)1 << n_log;
        u64* d = nullptr;
        TRY(table_alloc(ctx, n << rate_bits, &d));
        for (u32 b = 0; b < (1u << rate_bits); b++)
            TRY(fill_powers(ctx, hostgl::coset_shift_of_block(n_log, rate_bits, b), n_log, d + (u64)b * n));
        *t = d;
        return 0;
    });
}

template <int B>
static void launch_pass_b(const ntt::PassParams& p, dim3 grid, cudaStream_t s) {
    switch (ntt::pass_mode(p)) {
        case ntt::MODE_MID_NATURAL: ntt::ntt_pass_kernel<B, ntt::MODE_MID_NATURAL><<<grid, ntt::threads_for(B), 0, s>>>(p); break;
        case ntt::MODE_MID_BITREV: ntt::ntt_pass_kernel<B, ntt::MODE_MID_BITREV><<<grid, ntt::threads_for(B), 0, s>>>(p); break;
        case ntt::MODE_FINAL_BITREV: ntt::ntt_pass_kernel<B, ntt::MODE_FINAL_BITREV><<<grid, ntt::threads_for(B), 0, s>>>(p); break;
        default: ntt::ntt_pass_kernel<B, ntt::MODE_FINAL_NATURAL><<<grid, ntt::threads_for(B), 0, s>>>(p); break;
    }
}
static int launch_pass(b200zkp_ctx* ctx, const ntt::PassParams& p, u32 B, u32 n_blk) {
    u64 T = (u64)ntt::tile_elems_for((int)B) >> B;
    u64 total_batches = (u64)p.ncols << (p.n_log - B);
    u64 blocks = (total_batches + T - 1) / T;
    if (blocks == 0 || n_blk == 0) return 0;
    if (blocks > 0x7fffffffull || n_blk > 65535) BAD(ctx, "transform too large for one launch");
    dim3 grid((unsigned)blocks, n_blk);
    switch (B) {
        case 1: launch_pass_b<1>(p, grid, ctx->stream); break;
        case 2: launch_pass_b<2>(p, grid, ctx->stream); break;
        case 3: launch_pass_b<3>(p, grid, ctx->stream); break;
        case 4: launch_pass_b<4>(p, grid, ctx->stream); break;
        case 5: launch_pass_b<5>(p, grid, ctx->stream); break;
        case 6: launch_pass_b<6>(p, grid, ctx->stream); break;
        case 7: launch_pass_b<7>(p, grid, ctx->stream); break;
        case 8: launch_pass_b<8>(p, grid, ctx->stream); break;
        case 9: launch_pass_b<9>(p, grid, ctx->stream); break;
        case 10: launch_pass_b<10>(p, grid, ctx->stream); break;
        default: BAD(ctx, "internal: bad pass width");
    }
    LAUNCH_CHECK(ctx);
    return 0;
}

static int launch_canon_copy(b200zkp_ctx* ctx, const u64* src, u64* dst, u64 count) {
    if (!count) return 0;
    ntt::canon_copy_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(src, dst, count);
    LAUNCH_CHECK(ctx);
    return 0;
}

// twiddle images of every non-final pass of a 2^n_log transform (built on the device, cached per ctx);
// the inverse direction carries n^-1 in the first image
static int get_twiddle_images(b200zkp_ctx* ctx, u32 n_log, int dir, bool bitrev_out, b200zkp_ctx::Images* out) {
    return get_or_build(ctx->twimg, std::make_tuple(n_log, dir, bitrev_out), out, [&](b200zkp_ctx::Images* im) -> int {
        ntt::TwiddleImageShape shapes[ntt::MAX_PASSES];
        u32 n_img = ntt::twiddle_images(n_log, shapes);
        if (!n_img) return 0;
        TwoLevel tw{};
        TRY(get_tw(ctx, dir, n_log, &tw));
        u64 n_inv = hostgl::inv(((u64)1 << n_log) % hostgl::P);
        for (u32 pi = 0; pi < n_img; pi++) {
            u64 count = (u64)1 << (shapes[pi].B + shapes[pi].C_log);
            u64* d = nullptr;
            TRY(table_alloc(ctx, count, &d));
            u64 f = (dir == 1 && pi == 0) ? n_inv : 0;
            ntt::build_twiddle_image_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(
                d, shapes[pi].B, shapes[pi].C_log, shapes[pi].shift, bitrev_out ? 1u : 0u, f, tw.lo, tw.hi, tw.lo_bits);
            LAUNCH_CHECK(ctx);
            im->img[pi] = d;
        }
        return 0;
    });
}

// ---- second-generation passes: Z tables, tensor maps, launches
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn tensor_map_encoder() {
    static TensorMapEncodeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            (void)cudaGetLastError();
            p = nullptr;
        }
        return (TensorMapEncodeFn)p;
    }();
    return fn;
}

// 5-D view (c, row, a, coset block, column) of one side of a strided pass; box = one tile [2^B rows][T]
static bool encode_tile_map(CUtensorMap* map, const u64* base, u32 B, u32 S, u32 C_log, u32 n_blk, u64 blk_stride, u32 ncols,
                            u64 col_stride) {
    TensorMapEncodeFn enc = tensor_map_encoder();
    if (!enc) return false;
    const u64 C = (u64)1 << C_log, rows = (u64)1 << B, A = (u64)1 << S;
    cuuint64_t dims[5] = {C, rows, A, n_blk ? n_blk : 1, ncols};
    cuuint64_t strides[4] = {C * 8, C * rows * 8, (blk_stride ? blk_stride : C * rows * A) * 8, col_stride * 8};
    cuuint32_t box[5] = {(cuuint32_t)(ntc::TILE >> B), (cuuint32_t)rows, 1, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

template <int B>
static int launch_ct_b(b200zkp_ctx* ctx, int kind, const ntc::PassParams& p, u64 grid, const CUtensorMap& tm_in, const CUtensorMap& tm_out,
                       const ntc::PullMaps* tm_src, const CUtensorMap* tm_copy, u32 pull_ctas_per_sm) {
    const void* fn = nullptr;
    u32 smem = 0;
    switch (kind) {
        case ntc::KIND_STRIDED: fn = (const void*)ntc::ct_pass_kernel<B, ntc::KIND_STRIDED>; smem = ntc::StridedSmem<B, false>::bytes; break;
        case ntc::KIND_STRIDED_LOOP: fn = (const void*)ntc::ct_pass_kernel<B, ntc::KIND_STRIDED_LOOP>; smem = ntc::StridedSmem<B, true>::bytes; break;
        case ntc::KIND_FINAL_INPLACE: fn = (const void*)ntc::ct_pass_kernel<B, ntc::KIND_FINAL_INPLACE>; smem = ntc::FinalSmem<B>::bytes; break;
        case ntc::KIND_PULL_LOOP: fn = (const void*)ntc::ct_pull_kernel<B>; smem = ntc::PullSmem<B>::bytes; break;
        default: fn = (const void*)ntc::ct_pass_kernel<B, ntc::KIND_FINAL_NATURAL>; smem = ntc::FinalSmem<B>::bytes; break;
    }
    const u32 bit = 1u << ((B - ntc::MIN_BITS) * 5 + kind);
    if (smem > 48 * 1024 && !(ctx->ct_smem_set & bit)) {
        CUDA_TRY(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctx->ct_smem_set |= bit;
    }
    void* args[5] = {(void*)&p, (void*)&tm_in, (void*)&tm_out, nullptr, nullptr};
    u32 total = (u32)grid;
    if (kind == ntc::KIND_PULL_LOOP) {
        // persistent: a few CTAs per SM walk all `total` tiles
        args[1] = (void*)tm_src; args[2] = (void*)&tm_out; args[3] = (void*)tm_copy; args[4] = (void*)&total;
        if (!ctx->sm_count) {
            int sms = 0;
            CUDA_TRY(ctx, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
            ctx->sm_count = (u32)std::max(1, sms);
        }
        grid = std::min<u64>(grid, (u64)std::max(1u, pull_ctas_per_sm) * ctx->sm_count);
    }
    CUDA_TRY(ctx, cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(ntc::THREADS), args, smem, ctx->stream));
    ctx->launches++;
    return 0;
}

// later_stream (optional): the passes after the first run there, behind an event recorded after the first pass on the ctx
// stream (a partitioned LDE: the NVLink-bound gather pass of the next column group runs beside them); pull_ctas_per_sm:
// width of the persistent gather launch
static int run_ct_plan(b200zkp_ctx* ctx, ntc::Plan& plan, cudaStream_t later_stream = nullptr, cudaEvent_t first_done = nullptr,
                       u32 pull_ctas_per_sm = 4) {
    cudaStream_t const first_stream = ctx->stream;
    std::optional<StreamScope> later;
    for (u32 pi = 0; pi < plan.n_passes; pi++) {
        if (pi == 1 && later_stream && later_stream != first_stream) {
            CUDA_TRY(ctx, cudaEventRecord(first_done, first_stream));
            CUDA_TRY(ctx, cudaStreamWaitEvent(later_stream, first_done, 0));
            later.emplace(ctx, later_stream);
        }
        ntc::PassParams& p = plan.pass[pi];
        const u32 B = plan.bits[pi];
        const int kind = plan.kind[pi];
        if (plan.grid[pi] > 0x7fffffffull) BAD(ctx, "transform too large for one launch");
        alignas(64) CUtensorMap tm_in, tm_out, tm_copy;
        alignas(64) ntc::PullMaps tm_src;
        memset(&tm_in, 0, sizeof tm_in); memset(&tm_out, 0, sizeof tm_out); memset(&tm_copy, 0, sizeof tm_copy);
        const bool pull = kind == ntc::KIND_PULL_LOOP;
        if (pull) memset(&tm_src, 0, sizeof tm_src);
        // physical columns the maps must cover (a column set addresses columns [0, col_limit) of the buffers)
        const u32 map_cols = p.col_run ? p.col_limit : p.ncols;
        if (p.use_tma) {
            // the staged side of a coset loop has a single block; every other side walks the blocks of its buffer
            const bool loop = kind == ntc::KIND_STRIDED_LOOP || pull;
            bool ok = encode_tile_map(&tm_out, p.out, B, p.S, p.C_log, p.n_blk, p.out_blk_stride, map_cols, p.out_col_stride);
            if (ok && pull) {
                ok = encode_tile_map(&tm_copy, p.copy_out, B, p.S, p.C_log, 1, 0, map_cols, p.copy_col_stride);
                // a source's matrix holds col_run local columns per group of col_period columns of the commitment
                const u32 src_cols = ((p.col_limit + p.col_period - 1) / p.col_period) * p.col_run;
                for (u32 q = 0; ok && q < p.col_period / p.col_run; q++)
                    ok = encode_tile_map(&tm_src.m[q], p.src[q], B, p.S, p.C_log, 1, 0, src_cols, p.in_col_stride);
            } else if (ok) {
                ok = encode_tile_map(&tm_in, p.in, B, p.S, p.C_log, loop ? 1 : p.n_blk, loop ? 0 : p.in_blk_stride, map_cols, p.in_col_stride);
            }
            if (!ok) p.use_tma = 0;
        }
        switch (B) {
            case 5: TRY(launch_ct_b<5>(ctx, kind, p, plan.grid[pi], tm_in, tm_out, &tm_src, &tm_copy, pull_ctas_per_sm)); break;
            case 6: TRY(launch_ct_b<6>(ctx, kind, p, plan.grid[pi], tm_in, tm_out, &tm_src, &tm_copy, pull_ctas_per_sm)); break;
            case 7: TRY(launch_ct_b<7>(ctx, kind, p, plan.grid[pi], tm_in, tm_out, &tm_src, &tm_copy, pull_ctas_per_sm)); break;
            case 8: TRY(launch_ct_b<8>(ctx, kind, p, plan.grid[pi], tm_in, tm_out, &tm_src, &tm_copy, pull_ctas_per_sm)); break;
            default: BAD(ctx, "internal: bad pass width");
        }
    }
    return 0;
}

// Z tables of `n_blk` cosets s_b <w_n>: shifts[b] on the host; built on the device and kept for the life of the ctx.
// The squared shifts are a build input only: the stream is synchronised before they go back to the pool.
static int build_ztab(b200zkp_ctx* ctx, u32 n_log, int dir, const std::vector<u64>& shifts, u64 last_scale, bool natural,
                      b200zkp_ctx::ZTables* out) {
    TwoLevel tw{};
    TRY(get_tw(ctx, dir, n_log, &tw));
    std::vector<u64> spow((size_t)shifts.size() * n_log);
    for (size_t b = 0; b < shifts.size(); b++) {
        u64 x = shifts[b] % hostgl::P;
        for (u32 e = 0; e < n_log; e++) { spow[b * n_log + e] = x; x = hostgl::mul(x, x); }
    }
    DevBuf d_spow;
    TRY(d_spow.alloc(ctx, spow.size() * 8));
    TRY(h2d(ctx, d_spow.get(), spow.data(), d_spow.bytes()));
    const u64 count = ntc::ztab_entries(n_log), words = ntc::zfinal_words(n_log);
    u64 *d = nullptr, *f = nullptr;
    TRY(table_alloc(ctx, count * shifts.size(), &d));
    TRY(table_alloc(ctx, words * shifts.size(), &f));
    ntc::build_ztab_kernel<<<dim3((unsigned)((count + 255) / 256), (unsigned)shifts.size()), 256, 0, ctx->stream>>>(
        d, count, n_log, d_spow.get(), tw.lo, tw.hi, tw.lo_bits, last_scale);
    LAUNCH_CHECK(ctx);
    ntc::build_zfinal_kernel<<<dim3((unsigned)((words + 255) / 256), (unsigned)shifts.size()), 256, 0, ctx->stream>>>(
        f, words, n_log, ntc::last_pass_bits(n_log), natural ? 1u : 0u, d_spow.get(), tw.lo, tw.hi, tw.lo_bits, last_scale);
    LAUNCH_CHECK(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    out->strided = d;
    out->final_ = f;
    return 0;
}

static int get_ztab_lde(b200zkp_ctx* ctx, u32 n_log, u32 rate_bits, b200zkp_ctx::ZTables* out) {
    return get_or_build(ctx->ztab_lde, std::make_pair(n_log, rate_bits), out, [&](b200zkp_ctx::ZTables* t) {
        std::vector<u64> shifts;
        for (u32 b = 0; b < (1u << rate_bits); b++) shifts.push_back(hostgl::coset_shift_of_block(n_log, rate_bits, b));
        return build_ztab(ctx, n_log, 0, shifts, 0, /*natural=*/false, t);
    });
}

static int get_ztab_inv(b200zkp_ctx* ctx, u32 n_log, b200zkp_ctx::ZTables* out) {
    return get_or_build(ctx->ztab_inv, n_log, out, [&](b200zkp_ctx::ZTables* t) {
        return build_ztab(ctx, n_log, 1, std::vector<u64>{1}, hostgl::inv(((u64)1 << n_log) % hostgl::P), /*natural=*/true, t);
    });
}

// One multi-pass transform over `ncols` columns, for `n_blk` blocks at once (blockIdx.y: the coset blocks of an
// LDE share the input and differ in scale table and output offset).
//   bitrev_out: in-place DIF order (LDE leaf order); else natural order (needs scratch when P > 1)
static int run_transform(b200zkp_ctx* ctx, const u64* in, u64 in_stride, u64* out, u64 out_stride,
                         u64* scratch, u32 n_log, u32 ncols, int dir, bool bitrev_out,
                         const u64* scale, u64 scale_blk_stride, bool inverse_scale, bool canon_in,
                         u32 n_blk = 1, u64 out_blk_stride = 0) {
    if (ncols == 0) return 0;
    if (n_log == 0) {
        // single point: the transform is the identity (scale^0 = 1)
        for (u32 blk = 0; blk < n_blk; blk++)
            for (u32 c = 0; c < ncols; c++)   // rare path (n = 1): tiny launches keep strides general
                TRY(launch_canon_copy(ctx, in + c * in_stride, out + blk * out_blk_stride + c * out_stride, 1));
        return 0;
    }
    if (n_log > 32) BAD(ctx, "n_log exceeds the field's two-adicity (32)");
    if (!bitrev_out && n_log > (u32)ntt::MAX_PASS_BITS && !scratch) BAD(ctx, "scratch buffer required for multi-pass natural-order transforms");
    b200zkp_ctx::Images im;
    TRY(get_twiddle_images(ctx, n_log, dir, bitrev_out, &im));
    ntt::TransformTables tb{};
    tb.wtab = ctx->wtab[dir];
    for (u32 i = 0; i < ntt::MAX_PASSES; i++) tb.twimg[i] = im.img[i];
    tb.scale = scale;
    tb.scale_blk_stride = scale_blk_stride;
    u64 n_inv = hostgl::inv(((u64)1 << n_log) % hostgl::P);
    ntt::Plan plan;
    ntt::make_plan(&plan, in, in_stride, out, out_stride, scratch, n_log, ncols, tb, bitrev_out,
                   inverse_scale ? n_inv : 0, canon_in, /*in_blk_stride=*/0, out_blk_stride);
    for (u32 pi = 0; pi < plan.n_passes; pi++) TRY(launch_pass(ctx, plan.pass[pi], plan.bits[pi], n_blk));
    return 0;
}

// ------------------------------------------------------------------------------------------------
extern "C" const char* b200zkp_version(void) { return "b200zkp 0.1 (sm_100a)"; }

extern "C" int b200zkp_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return B200ZKP_ERR_CUDA; }
    return n;
}

static int ctx_init_tables(b200zkp_ctx* ctx) {
    TRY(table_alloc(ctx, 360, &ctx->round_add));
    CUDA_TRY(ctx, cudaMemcpyFromSymbolAsync(ctx->round_add, poseidon_tables::ROUND_ADD, 360 * sizeof(u64), 0,
                                            cudaMemcpyDeviceToDevice, ctx->stream));
    for (int dir = 0; dir < 2; dir++)
        for (u32 B = 1; B <= (u32)ntt::MAX_PASS_BITS; B++) TRY(upload(ctx, hostgl::small_root_table(B, dir), &ctx->wtab[dir][B]));
    return 0;
}

extern "C" int b200zkp_ctx_create(int device, void* stream, b200zkp_ctx** out) {
    if (!out) return B200ZKP_ERR_BAD_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { (void)cudaGetLastError(); return B200ZKP_ERR_CUDA; }
    if (device < 0 || device >= n) return B200ZKP_ERR_BAD_ARG;
    if (cudaSetDevice(device) != cudaSuccess) { (void)cudaGetLastError(); return B200ZKP_ERR_CUDA; }
    b200zkp_ctx* ctx = new (std::nothrow) b200zkp_ctx();
    if (!ctx) return B200ZKP_ERR_OOM;
    ctx->device = device;
    if (stream) { ctx->stream = (cudaStream_t)stream; ctx->own_stream = false; }
    else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            (void)cudaGetLastError(); delete ctx; return B200ZKP_ERR_CUDA;
        }
        ctx->own_stream = true;
    }
    size_t mem_free = 0, mem_total = 0;
    if (cudaMemGetInfo(&mem_free, &mem_total) == cudaSuccess && mem_total) ctx->pool_max_bytes = mem_total / 8;
    else (void)cudaGetLastError();
    int rc = ctx_init_tables(ctx);
    if (rc != 0) { b200zkp_ctx_destroy(ctx); return rc; }
    *out = ctx;
    return 0;
}

extern "C" void b200zkp_ctx_destroy(b200zkp_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    pool_drop(ctx);
    for (void* p : ctx->table_allocs) cudaFree(p);
    for (auto& sp : ctx->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    for (auto e : ctx->ev_free) cudaEventDestroy(e);
    for (auto e : ctx->sync_events) cudaEventDestroy(e);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->mailbox) cudaFreeHost(ctx->mailbox);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* b200zkp_last_error(const b200zkp_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
extern "C" uint64_t b200zkp_ctx_launch_count(const b200zkp_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int b200zkp_ctx_synchronize(b200zkp_ctx* ctx) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);      // ctx->stream is swapped temporarily by the two-stream pipelines: read it under the lock
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int b200zkp_ctx_set_pool_limit(b200zkp_ctx* ctx, uint64_t bytes) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    ctx->pool_max_bytes = (size_t)bytes;
    if (ctx->pool_bytes > ctx->pool_max_bytes) {
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        pool_drop(ctx);
    }
    return 0;
}

extern "C" int b200zkp_ctx_trim(b200zkp_ctx* ctx) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    pool_drop(ctx);
    return 0;
}

extern "C" int b200zkp_ctx_buffer_bytes(b200zkp_ctx* ctx, uint64_t* live, uint64_t* cached) {
    if (!ctx || !live || !cached) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    *live = ctx->live_bytes;
    *cached = ctx->pool_bytes;
    return 0;
}

extern "C" int b200zkp_ctx_set_timing(b200zkp_ctx* ctx, int enabled) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    ctx->timing = enabled != 0;
    return 0;
}

// Synchronises the stream, adds up the recorded spans per stage and clears them.
extern "C" int b200zkp_ctx_stage_ms(b200zkp_ctx* ctx, double ms[B200ZKP_N_STAGES], uint32_t counts[B200ZKP_N_STAGES]) {
    if (!ctx || !ms) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < B200ZKP_N_STAGES; i++) { ms[i] = 0; if (counts) counts[i] = 0; }
    for (auto& sp : ctx->spans) {
        float t = 0;
        if (cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess && sp.stage >= 0 && sp.stage < B200ZKP_N_STAGES) {
            ms[sp.stage] += t;
            if (counts) counts[sp.stage]++;
        }
        ctx->ev_free.push_back(sp.a);
        ctx->ev_free.push_back(sp.b);
    }
    (void)cudaGetLastError();
    ctx->spans.clear();
    return 0;
}

extern "C" int b200zkp_host_alloc(size_t bytes, void** out) {
    if (!out) return B200ZKP_ERR_BAD_ARG;
    cudaError_t e = cudaMallocHost(out, bytes);
    if (e != cudaSuccess) { (void)cudaGetLastError(); *out = nullptr; return e == cudaErrorMemoryAllocation ? B200ZKP_ERR_OOM : B200ZKP_ERR_CUDA; }
    return 0;
}
extern "C" void b200zkp_host_free(void* p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------------ device stages

static int dev_intt_locked(b200zkp_ctx* ctx, const u64* values, u64 in_stride, u64* coeffs, u64 out_stride,
                           u64* scratch, u32 n_log, u32 k) {
    if (scratch && k && ntc::covers(n_log)) {
        // 2^11 points and more: block-twiddle passes (ntt_ct_kernels.cuh), natural order out through the scratch buffer
        b200zkp_ctx::ZTables z;
        TRY(get_ztab_inv(ctx, n_log, &z));
        ntc::Plan plan;
        if (ntc::make_plan(&plan, values, in_stride, coeffs, out_stride, scratch, n_log, k, 1, 0, /*natural_out=*/true, z.strided,
                           z.final_, hostgl::inv(((u64)1 << n_log) % hostgl::P), /*use_tma=*/true)) {
            StageTimer tm(ctx, B200ZKP_STAGE_INTT);
            return run_ct_plan(ctx, plan);
        }
    }
    StageTimer tm(ctx, B200ZKP_STAGE_INTT);
    return run_transform(ctx, values, in_stride, coeffs, out_stride, scratch, n_log, k, /*dir=*/1,
                         /*bitrev_out=*/false, nullptr, 0, /*inverse_scale=*/true, /*canon_in=*/true);
}

extern "C" int b200zkp_dev_intt(b200zkp_ctx* ctx, const uint64_t* values, uint64_t in_stride, uint64_t* coeffs,
                                uint64_t out_stride, uint64_t* scratch, uint32_t n_log, uint32_t k) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!values || !coeffs) BAD(ctx, "null buffer");
    return dev_intt_locked(ctx, (const u64*)values, in_stride, (u64*)coeffs, out_stride, (u64*)scratch, n_log, k);
}

static int dev_lde_locked(b200zkp_ctx* ctx, const u64* coeffs, u64 coeff_stride, u64* lde, u64 lde_stride,
                          u32 n_log, u32 k, u32 rate_bits, u32 b0, u32 b1) {
    if (rate_bits > 8 || n_log + rate_bits > 32) BAD(ctx, "rate_bits / n_log out of range");
    if (b0 > b1 || b1 > (1u << rate_bits)) BAD(ctx, "bad coset block range");
    u64 n = (u64)1 << n_log;
    if (k && b1 > b0 && ntc::covers(n_log)) {
        // block-twiddle passes: the coset shift lives in the twiddles, the first pass stages a coefficient tile once for all blocks
        b200zkp_ctx::ZTables z;
        TRY(get_ztab_lde(ctx, n_log, rate_bits, &z));
        ntc::Plan plan;
        if (ntc::make_plan(&plan, coeffs, coeff_stride, lde, lde_stride, nullptr, n_log, k, b1 - b0, n, /*natural_out=*/false,
                           z.strided + (u64)b0 * ntc::ztab_entries(n_log), z.final_ + (u64)b0 * ntc::zfinal_words(n_log), 0, /*use_tma=*/true)) {
            StageTimer tm(ctx, B200ZKP_STAGE_LDE);
            return run_ct_plan(ctx, plan);
        }
    }
    const u64* cs = nullptr;
    TRY(get_coset_scale(ctx, n_log, rate_bits, &cs));
    StageTimer tm(ctx, B200ZKP_STAGE_LDE);
    // all coset blocks in one launch per pass (blockIdx.y): block b reads the same coefficients, scales them
    // by the powers of its shift and writes leaves [(b - b0) * n, (b - b0 + 1) * n) of every column
    return run_transform(ctx, coeffs, coeff_stride, lde, lde_stride, nullptr, n_log, k, /*dir=*/0, /*bitrev_out=*/true,
                         cs + (u64)b0 * n, n, /*inverse_scale=*/false, /*canon_in=*/true, b1 - b0, n);
}

// Coset transforms of a column set of a partitioned LDE (sharded.inl): `cols` names cols.count columns of the local LDE;
// with cols.pull the first pass gathers the coefficients from the sources' exchange windows (peer memory) on the way.
// Returns B200ZKP_ERR_UNSUPPORTED (nothing launched) when the block-twiddle passes do not cover the shape.
static int dev_lde_cols_locked(b200zkp_ctx* ctx, const ntc::ColumnSet& cols, const u64* coeffs, u64 coeff_stride, u64* lde,
                               u64 lde_stride, u32 n_log, u32 rate_bits, u32 b0, u32 b1, cudaStream_t later_stream = nullptr,
                               cudaEvent_t first_done = nullptr, u32 pull_ctas_per_sm = 4) {
    if (rate_bits > 8 || n_log + rate_bits > 32) BAD(ctx, "rate_bits / n_log out of range");
    if (b0 >= b1 || b1 > (1u << rate_bits)) BAD(ctx, "bad coset block range");
    const u64 n = (u64)1 << n_log;
    if (!ntc::covers(n_log)) return B200ZKP_ERR_UNSUPPORTED;
    b200zkp_ctx::ZTables z;
    TRY(get_ztab_lde(ctx, n_log, rate_bits, &z));
    ntc::Plan plan;
    if (!ntc::make_plan(&plan, coeffs, coeff_stride, lde, lde_stride, nullptr, n_log, 0, b1 - b0, n, /*natural_out=*/false,
                        z.strided + (u64)b0 * ntc::ztab_entries(n_log), z.final_ + (u64)b0 * ntc::zfinal_words(n_log), 0, /*use_tma=*/true, &cols))
        return B200ZKP_ERR_UNSUPPORTED;
    if (later_stream) return run_ct_plan(ctx, plan, later_stream, first_done, pull_ctas_per_sm);   // (the caller times the whole pipeline)
    StageTimer tm(ctx, B200ZKP_STAGE_LDE);
    return run_ct_plan(ctx, plan, nullptr, nullptr, pull_ctas_per_sm);
}

extern "C" int b200zkp_dev_lde(b200zkp_ctx* ctx, const uint64_t* coeffs, uint64_t coeff_stride, uint64_t* lde,
                               uint64_t lde_stride, uint32_t n_log, uint32_t k, uint32_t rate_bits,
                               uint32_t block_begin, uint32_t block_end) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!coeffs || !lde) BAD(ctx, "null buffer");
    return dev_lde_locked(ctx, (const u64*)coeffs, coeff_stride, (u64*)lde, lde_stride, n_log, k, rate_bits,
                          block_begin, block_end);
}

static int dev_salt_locked(b200zkp_ctx* ctx, const u64* salt, u64* lde_salt, u64 lde_stride, u32 n_log,
                           u32 rate_bits, u32 b0, u32 b1) {
    // leaf j = natural row bitrev(j, N_log); leaf block b covers j in [b*n, (b+1)*n):
    // natural index = bitrev(jl, n_log) * 2^r + bitrev(b, r).  One strided bit-reversed copy per block.
    u32 N_log = n_log + rate_bits;
    if (b0 == 0 && b1 == (1u << rate_bits)) {
        u64 cnt = (u64)B200ZKP_SALT_SIZE << N_log;
        ntt::bitrev_copy_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, ctx->stream>>>(
            salt, lde_salt, N_log, B200ZKP_SALT_SIZE, (u64)1 << N_log, lde_stride);
        LAUNCH_CHECK(ctx);
        return 0;
    }
    ctx->err = "salted commitments are only supported unsharded";
    return B200ZKP_ERR_UNSUPPORTED;
}

extern "C" int b200zkp_dev_salt(b200zkp_ctx* ctx, const uint64_t* salt, uint64_t* lde_salt_cols,
                                uint64_t lde_stride, uint32_t n_log, uint32_t rate_bits, uint32_t block_begin,
                                uint32_t block_end) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!salt || !lde_salt_cols) BAD(ctx, "null buffer");
    return dev_salt_locked(ctx, (const u64*)salt, (u64*)lde_salt_cols, lde_stride, n_log, rate_bits, block_begin, block_end);
}

// F::rand_vec: elements [first, first + count) of the ChaCha20 stream (key, nonce), one thread per block (random_kernels.cuh)
extern "C" int b200zkp_dev_random_field(b200zkp_ctx* ctx, const uint8_t key[32], const uint8_t nonce[12], uint64_t first,
                                        uint64_t count, uint64_t* out_dev) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!count) return 0;
    if (!key || !nonce || !out_dev) BAD(ctx, "null key, nonce or output");
    if (!rnd::range_ok(first, count)) BAD(ctx, "the range needs a ChaCha20 block counter of 2^32 or more (first + count > 2^34)");
    rnd::ChaChaKey k;
    for (int i = 0; i < 8; i++)
        k.key[i] = (u32)key[4 * i] | (u32)key[4 * i + 1] << 8 | (u32)key[4 * i + 2] << 16 | (u32)key[4 * i + 3] << 24;
    for (int i = 0; i < 3; i++)
        k.nonce[i] = (u32)nonce[4 * i] | (u32)nonce[4 * i + 1] << 8 | (u32)nonce[4 * i + 2] << 16 | (u32)nonce[4 * i + 3] << 24;
    const u64 n_blocks = rnd::blocks_of_range(first, count);
    rnd::random_field_kernel<<<(unsigned)((n_blocks + 255) / 256), 256, 0, ctx->stream>>>(k, first, count, n_blocks, (u64*)out_dev);
    LAUNCH_CHECK(ctx);
    return 0;
}

static int merkle_shape(b200zkp_ctx* ctx, u64 n_leaves, u32 cap_height, const void* leaves, const void* digests, const void* cap,
                        merkle::TreeShape* shape) {
    u32 lg = 0;
    if (!log2_exact(n_leaves, &lg)) BAD(ctx, "number of leaves must be a power of two");
    if (cap_height > lg) BAD(ctx, "cap_height exceeds log2(number of leaves)");
    if (!leaves || !cap) BAD(ctx, "null buffer");
    shape->sub_log = lg - cap_height;
    shape->sub_digests = 2 * (((u64)1 << shape->sub_log) - 1);
    if (shape->sub_log > 0 && !digests) BAD(ctx, "null digests buffer");
    return 0;
}

// Block size of the hash kernels: 512 threads when the launch fills the GPU anyway, smaller CTAs for small trees so
// that every SM gets work (the kernels are compiled for up to 512 threads at 64 registers).
static unsigned hash_block_threads(u64 n_items) {
    unsigned t = B200ZKP_HASH_THREADS;
    while (t > 32 && n_items / t < 2 * 148) t >>= 1;
    return t;
}

// Leaf batches, tree levels and hash batches of at most this many items use the latency form of the permutation
// (merkle_kernels.cuh), which wins while the work cannot fill the GPU; sweeps of both thresholds: profiles/r2z_*_sweep.log.
static constexpr u64 COOP_MAX_NODES = 2048;

static int launch_leaf_hash(b200zkp_ctx* ctx, const u64* leaves, u64 row_stride, u64 col_stride, u32 leaf_len, u64 row0,
                            u64 n_rows, const merkle::TreeShape& shape, u64* digests, u64* cap) {
    if (!n_rows) return 0;
    StageTimer tm(ctx, B200ZKP_STAGE_LEAF_HASH);
    if (n_rows <= COOP_MAX_NODES) {
        merkle::leaf_hash_coop_kernel<<<(unsigned)((n_rows * 16 + 127) / 128), 128, 0, ctx->stream>>>(
            leaves, row_stride, col_stride, leaf_len, row0, n_rows, shape, digests, cap, 1u, ctx->round_add);
        LAUNCH_CHECK(ctx);
        return 0;
    }
    unsigned threads = hash_block_threads(n_rows);
    u64 blocks = (n_rows + threads - 1) / threads;
    merkle::leaf_hash_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(leaves, row_stride, col_stride, leaf_len,
                                                                                         row0, n_rows, shape, digests, cap, 1u);
    LAUNCH_CHECK(ctx);
    return 0;
}

static int launch_tree_levels(b200zkp_ctx* ctx, u64 n_leaves, const merkle::TreeShape& shape, u64* digests, u64* cap) {
    StageTimer tm(ctx, B200ZKP_STAGE_TREE);
    // layers with at most 2^TOP_PARENTS_LOG parents per cap subtree: one launch for all of them (merkle_top_kernel)
    const u32 top_layer0 = shape.sub_log > merkle::TOP_PARENTS_LOG ? shape.sub_log - merkle::TOP_PARENTS_LOG : 0;
    const u64 n_subtrees = n_leaves >> shape.sub_log;
    const bool fused_top = shape.sub_log > 0 && n_subtrees <= 65535;
    for (u32 layer = 0; layer < shape.sub_log; layer++) {
        if (fused_top && layer == top_layer0) {
            const u32 par0 = 1u << (shape.sub_log - layer - 1);          // parents per subtree at the first fused layer
            const unsigned threads = std::max(32u, std::min(1024u, par0 * 16));
            merkle::merkle_top_kernel<<<(unsigned)n_subtrees, threads, 0, ctx->stream>>>(digests, cap, shape, layer, ctx->round_add);
            LAUNCH_CHECK(ctx);
            break;
        }
        u64 n_parents = n_leaves >> (layer + 1);
        if (n_parents <= COOP_MAX_NODES) {
            // too few nodes to fill the GPU: one node per 16 lanes, ~4x less latency per level
            merkle::merkle_level_coop_kernel<<<(unsigned)((n_parents * 16 + 127) / 128), 128, 0, ctx->stream>>>(
                digests, cap, shape, layer, n_parents, ctx->round_add);
        } else {
            unsigned threads = hash_block_threads(n_parents);
            u64 blocks = (n_parents + threads - 1) / threads;
            merkle::merkle_level_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(digests, cap, shape, layer, n_parents);
        }
        LAUNCH_CHECK(ctx);
    }
    return 0;
}

static int dev_merkle_locked(b200zkp_ctx* ctx, const u64* leaves, u64 row_stride, u64 col_stride, u32 leaf_len,
                             u64 n_leaves, u32 cap_height, u64* digests, u64* cap) {
    merkle::TreeShape shape;
    TRY(merkle_shape(ctx, n_leaves, cap_height, leaves, digests, cap, &shape));
    TRY(launch_leaf_hash(ctx, leaves, row_stride, col_stride, leaf_len, 0, n_leaves, shape, digests, cap));
    return launch_tree_levels(ctx, n_leaves, shape, digests, cap);
}

static int get_sync_event(b200zkp_ctx* ctx, size_t i, cudaEvent_t* out) {
    while (ctx->sync_events.size() <= i) {
        cudaEvent_t e;
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->sync_events.push_back(e);
    }
    *out = ctx->sync_events[i];
    return 0;
}

// Coset LDE of leaf blocks [b0, b1) + Merkle forest over those leaves
static int dev_lde_merkle_locked(b200zkp_ctx* ctx, const u64* coeffs, u64 coeff_stride, u64* lde, u64 lde_stride, u32 n_log,
                                 u32 k, u32 rate_bits, u32 b0, u32 b1, u32 leaf_len, u32 cap_height, u64* digests, u64* cap) {
    if (rate_bits > 8 || n_log + rate_bits > 32) BAD(ctx, "rate_bits / n_log out of range");
    if (b0 >= b1 || b1 > (1u << rate_bits)) BAD(ctx, "bad coset block range");
    u64 n_leaves = (u64)(b1 - b0) << n_log;
    merkle::TreeShape shape;
    TRY(merkle_shape(ctx, n_leaves, cap_height, lde, digests, cap, &shape));
    TRY(dev_lde_locked(ctx, coeffs, coeff_stride, lde, lde_stride, n_log, k, rate_bits, b0, b1));
    TRY(launch_leaf_hash(ctx, lde, 1, lde_stride, leaf_len, 0, n_leaves, shape, digests, cap));
    return launch_tree_levels(ctx, n_leaves, shape, digests, cap);
}

extern "C" int b200zkp_dev_merkle(b200zkp_ctx* ctx, const uint64_t* leaves, uint64_t row_stride,
                                  uint64_t col_stride, uint32_t leaf_len, uint64_t n_leaves, uint32_t cap_height,
                                  uint64_t* digests, uint64_t* cap) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return dev_merkle_locked(ctx, (const u64*)leaves, row_stride, col_stride, leaf_len, n_leaves, cap_height,
                             (u64*)digests, (u64*)cap);
}

extern "C" int b200zkp_dev_lde_merkle(b200zkp_ctx* ctx, const uint64_t* coeffs, uint64_t coeff_stride, uint64_t* lde,
                                      uint64_t lde_stride, uint32_t n_log, uint32_t k, uint32_t rate_bits, uint32_t block_begin,
                                      uint32_t block_end, uint32_t cap_height, uint64_t* digests, uint64_t* cap) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!coeffs || !lde) BAD(ctx, "null buffer");
    return dev_lde_merkle_locked(ctx, (const u64*)coeffs, coeff_stride, (u64*)lde, lde_stride, n_log, k, rate_bits, block_begin,
                                 block_end, k, cap_height, (u64*)digests, (u64*)cap);
}

// plonky2's asserts on the shape of a PolynomialBatch
static int check_commit_shape(b200zkp_ctx* ctx, u32 n_log, u32 k, u32 rate_bits, u32 cap_height) {
    if (k == 0) BAD(ctx, "empty polynomial batch");
    if (n_log + rate_bits > 32 || rate_bits > 8) BAD(ctx, "n_log + rate_bits exceeds two-adicity");
    if (cap_height > n_log + rate_bits) BAD(ctx, "cap_height exceeds log2(LDE size)");
    return 0;
}

static int dev_commit_locked(b200zkp_ctx* ctx, const u64* in, int is_coeffs, u32 n_log, u32 k, u32 rate_bits,
                             u32 cap_height, const u64* salt, u64* coeffs, u64* lde, u64* digests, u64* cap) {
    TRY(check_commit_shape(ctx, n_log, k, rate_bits, cap_height));
    if (!in || !coeffs || !lde || !cap) BAD(ctx, "null buffer");
    u64 n = (u64)1 << n_log, N = n << rate_bits;
    u32 row = k + (salt ? B200ZKP_SALT_SIZE : 0);
    if (is_coeffs) TRY(launch_canon_copy(ctx, in, coeffs, (u64)k * n));
    else TRY(dev_intt_locked(ctx, in, n, coeffs, n, /*scratch=*/lde, n_log, k));   // the LDE buffer is free until step 2
    if (salt) TRY(dev_salt_locked(ctx, salt, lde + (u64)k * N, N, n_log, rate_bits, 0, 1u << rate_bits));
    return dev_lde_merkle_locked(ctx, coeffs, n, lde, N, n_log, k, rate_bits, 0, 1u << rate_bits, row, cap_height, digests, cap);
}

extern "C" int b200zkp_dev_commit(b200zkp_ctx* ctx, const uint64_t* in, int is_coeffs, uint32_t n_log, uint32_t k,
                                  uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, uint64_t* coeffs,
                                  uint64_t* lde, uint64_t* digests, uint64_t* cap) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return dev_commit_locked(ctx, (const u64*)in, is_coeffs, n_log, k, rate_bits, cap_height, (const u64*)salt,
                             (u64*)coeffs, (u64*)lde, (u64*)digests, (u64*)cap);
}

static int dev_transpose_rows_locked(b200zkp_ctx* ctx, const u64* cm, u64 col_stride, u32 cols, u64 row0,
                                     u64 n_rows, u64* rm) {
    if (!n_rows || !cols) return 0;
    dim3 grid((unsigned)((n_rows + 31) / 32), (cols + 31) / 32), block(32, 8);
    merkle::transpose_to_rows_kernel<<<grid, block, 0, ctx->stream>>>(cm, col_stride, cols, row0, n_rows, rm);
    LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int b200zkp_dev_transpose_to_rows(b200zkp_ctx* ctx, const uint64_t* cm, uint64_t col_stride,
                                             uint32_t cols, uint64_t row0, uint64_t n_rows, uint64_t* rm) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!cm || !rm) BAD(ctx, "null buffer");
    return dev_transpose_rows_locked(ctx, (const u64*)cm, col_stride, cols, row0, n_rows, (u64*)rm);
}

// ------------------------------------------------------------------------------------------------ PolynomialBatch
// host destinations of a copy-back commit (any may be null)
struct CopyBack {
    u64* coeffs = nullptr;   // k * n
    u64* leaves = nullptr;   // N * (k + salt), row-major
    u64* digests = nullptr;  // 4 * 2(N - 2^h)
    u64* cap = nullptr;      // 4 * 2^h
};

static int commit_host(b200zkp_ctx* ctx, const u64* in, int is_coeffs, u32 n_log, u32 k, u32 rate_bits,
                       u32 cap_height, const u64* salt, b200zkp_batch** out, const CopyBack* cb = nullptr) {
    if (!out && !cb) BAD(ctx, "null out");
    if (out) *out = nullptr;
    TRY(check_commit_shape(ctx, n_log, k, rate_bits, cap_height));
    if (!in) BAD(ctx, "null input");
    u64 n = (u64)1 << n_log, N = n << rate_bits;
    u32 row = k + (salt ? B200ZKP_SALT_SIZE : 0);
    std::unique_ptr<b200zkp_batch> b(new (std::nothrow) b200zkp_batch());
    if (!b) return B200ZKP_ERR_OOM;
    b->ctx = ctx; b->n_log = n_log; b->k = k; b->rate_bits = rate_bits; b->cap_height = cap_height;
    b->salt = salt ? B200ZKP_SALT_SIZE : 0;
    DevBuf d_in, d_salt, stage;
    TRY(b->coeffs.alloc(ctx, (size_t)k * n * 8));
    TRY(b->lde.alloc(ctx, (size_t)row * N * 8));
    TRY(b->digests.alloc(ctx, (size_t)2 * (N - ((u64)1 << cap_height)) * 32));
    TRY(b->cap.alloc(ctx, ((size_t)32) << cap_height));
    TRY(d_in.alloc(ctx, (size_t)k * n * 8));
    TRY(d_salt.alloc(ctx, salt ? (size_t)B200ZKP_SALT_SIZE * N * 8 : 0));
    // declared after the buffers, so it runs before they go back to the pool on every exit: nothing may still be writing them
    struct Drain {
        b200zkp_ctx* c;
        ~Drain() { cudaStreamSynchronize(c->stream); if (c->stream2) cudaStreamSynchronize(c->stream2); (void)cudaGetLastError(); }
    } drain{ctx};
    // Column-chunked upload pipeline: chunk c+1 crosses PCIe on the copy stream while chunk c is inverse-transformed
    // and extended on the main stream (columns are independent until the leaf hash), so the 8nk-byte H2D hides behind
    // the transforms when the caller's buffer is pinned.
    TRY(ensure_stream2(ctx));
    const u32 n_chunks = (k >= 16 && d_in.bytes() >= ((size_t)64 << 20)) ? 8 : 1;
    const u32 per = (k + n_chunks - 1) / n_chunks;
    cudaEvent_t e_free;
    TRY(get_sync_event(ctx, 0, &e_free));
    // d_in / lde may be recycled buffers still in use by earlier work on the main stream
    CUDA_TRY(ctx, cudaEventRecord(e_free, ctx->stream));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, e_free, 0));
    if (salt) CUDA_TRY(ctx, cudaMemcpyAsync(d_salt.get(), salt, d_salt.bytes(), cudaMemcpyHostToDevice, ctx->stream2));
    std::vector<cudaEvent_t> up(n_chunks);
    for (u32 c = 0; c < n_chunks; c++) {
        u32 c0 = std::min(k, c * per), c1 = std::min(k, (c + 1) * per);
        TRY(get_sync_event(ctx, 1 + c, &up[c]));
        if (c1 > c0) CUDA_TRY(ctx, cudaMemcpyAsync(d_in.get() + (u64)c0 * n, in + (u64)c0 * n, (size_t)(c1 - c0) * n * 8, cudaMemcpyHostToDevice, ctx->stream2));
        CUDA_TRY(ctx, cudaEventRecord(up[c], ctx->stream2));
    }
    for (u32 c = 0; c < n_chunks; c++) {
        u32 c0 = std::min(k, c * per), c1 = std::min(k, (c + 1) * per);
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, up[c], 0));
        if (c1 == c0) continue;
        const u64* src = d_in.get() + (u64)c0 * n;
        u64* cf = b->coeffs.get() + (u64)c0 * n;
        u64* ld = b->lde.get() + (u64)c0 * N;
        if (is_coeffs) TRY(launch_canon_copy(ctx, src, cf, (u64)(c1 - c0) * n));
        else TRY(dev_intt_locked(ctx, src, n, cf, n, /*scratch=*/ld, n_log, c1 - c0));     // this chunk's LDE columns are still free
        if (cb && cb->coeffs) {
            // copy-back: this chunk's coefficients go home while the later chunks are still being transformed
            cudaEvent_t e_cf;
            TRY(get_sync_event(ctx, 2 + n_chunks + c, &e_cf));
            CUDA_TRY(ctx, cudaEventRecord(e_cf, ctx->stream));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, e_cf, 0));
            CUDA_TRY(ctx, cudaMemcpyAsync(cb->coeffs + (u64)c0 * n, cf, (size_t)(c1 - c0) * n * 8, cudaMemcpyDeviceToHost, ctx->stream2));
        }
        TRY(dev_lde_locked(ctx, cf, n, ld, N, n_log, c1 - c0, rate_bits, 0, 1u << rate_bits));
    }
    if (salt) TRY(dev_salt_locked(ctx, d_salt.get(), b->lde.get() + (u64)k * N, N, n_log, rate_bits, 0, 1u << rate_bits));
    // Copy-back (strict drop-in) mode: coefficients and row-major leaves leave the device on the copy stream while the
    // main stream hashes — the 8N(k+salt)-byte D2H (PCIe bound) overlaps the leaf hash instead of following it.
    if (cb && (cb->coeffs || cb->leaves)) {
        cudaEvent_t e_lde;
        TRY(get_sync_event(ctx, 1 + n_chunks, &e_lde));
        CUDA_TRY(ctx, cudaEventRecord(e_lde, ctx->stream));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, e_lde, 0));
        if (cb->leaves) {
            u64 chunk_rows = std::min<u64>(N, std::max<u64>(1, ((u64)256 << 20) / ((u64)row * 8)));
            TRY(stage.alloc(ctx, (size_t)chunk_rows * row * 8));
            StreamScope on_copy(ctx, ctx->stream2);     // transposes are issued on the copy stream (same order as their D2H)
            for (u64 r0 = 0; r0 < N; r0 += chunk_rows) {
                u64 nr = std::min(chunk_rows, N - r0);
                TRY(dev_transpose_rows_locked(ctx, b->lde.get(), N, row, r0, nr, stage.get()));
                CUDA_TRY(ctx, cudaMemcpyAsync(cb->leaves + r0 * row, stage.get(), (size_t)nr * row * 8, cudaMemcpyDeviceToHost, ctx->stream2));
            }
        }
    }
    TRY(dev_merkle_locked(ctx, b->lde.get(), /*row_stride=*/1, /*col_stride=*/N, row, N, cap_height, b->digests.get(), b->cap.get()));
    if (cb && cb->digests && b->digests.bytes())
        CUDA_TRY(ctx, cudaMemcpyAsync(cb->digests, b->digests.get(), b->digests.bytes(), cudaMemcpyDeviceToHost, ctx->stream));
    if (cb && cb->cap) CUDA_TRY(ctx, cudaMemcpyAsync(cb->cap, b->cap.get(), b->cap.bytes(), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream2));
    if (out) *out = b.release();
    return 0;
}

extern "C" int b200zkp_commit_copy_back(b200zkp_ctx* ctx, const uint64_t* in, int is_coeffs, uint32_t n_log, uint32_t k,
                                        uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, uint64_t* coeffs_out,
                                        uint64_t* leaves_out, uint64_t* digests_out, uint64_t* cap_out, b200zkp_batch** out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    CopyBack cb;
    cb.coeffs = (u64*)coeffs_out; cb.leaves = (u64*)leaves_out; cb.digests = (u64*)digests_out; cb.cap = (u64*)cap_out;
    return commit_host(ctx, (const u64*)in, is_coeffs, n_log, k, rate_bits, cap_height, (const u64*)salt, out, &cb);
}

extern "C" int b200zkp_commit_from_values(b200zkp_ctx* ctx, const uint64_t* values, uint32_t n_log, uint32_t k,
                                          uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt,
                                          b200zkp_batch** out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return commit_host(ctx, (const u64*)values, 0, n_log, k, rate_bits, cap_height, (const u64*)salt, out);
}
extern "C" int b200zkp_commit_from_coeffs(b200zkp_ctx* ctx, const uint64_t* coeffs, uint32_t n_log, uint32_t k,
                                          uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt,
                                          b200zkp_batch** out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return commit_host(ctx, (const u64*)coeffs, 1, n_log, k, rate_bits, cap_height, (const u64*)salt, out);
}

// PolynomialBatch::from_values / from_coeffs on a matrix already in HBM: dev_commit_locked writing into the handle's buffers
extern "C" int b200zkp_batch_from_device(b200zkp_ctx* ctx, const uint64_t* in_dev, int is_coeffs, uint32_t n_log, uint32_t k,
                                         uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt_dev, b200zkp_batch** out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!out) BAD(ctx, "null out");
    *out = nullptr;
    TRY(check_commit_shape(ctx, n_log, k, rate_bits, cap_height));
    if (!in_dev) BAD(ctx, "null buffer");
    u64 N = (u64)1 << (n_log + rate_bits);
    std::unique_ptr<b200zkp_batch> b(new (std::nothrow) b200zkp_batch());
    if (!b) return B200ZKP_ERR_OOM;
    b->ctx = ctx; b->n_log = n_log; b->k = k; b->rate_bits = rate_bits; b->cap_height = cap_height;
    b->salt = salt_dev ? B200ZKP_SALT_SIZE : 0;
    TRY(b->coeffs.alloc(ctx, ((size_t)k * 8) << n_log));
    TRY(b->lde.alloc(ctx, (size_t)(k + b->salt) * N * 8));
    TRY(b->digests.alloc(ctx, (size_t)2 * (N - ((u64)1 << cap_height)) * 32));
    TRY(b->cap.alloc(ctx, ((size_t)32) << cap_height));
    int rc = dev_commit_locked(ctx, (const u64*)in_dev, is_coeffs, n_log, k, rate_bits, cap_height, (const u64*)salt_dev,
                               b->coeffs.get(), b->lde.get(), b->digests.get(), b->cap.get());
    if (rc) {
        // the buffers go back to the pool: nothing may still be writing them
        cudaStreamSynchronize(ctx->stream);
        if (ctx->stream2) cudaStreamSynchronize(ctx->stream2);
        (void)cudaGetLastError();
        return rc;
    }
    *out = b.release();
    return 0;
}

extern "C" void b200zkp_batch_free(b200zkp_batch* b) {
    if (!b) return;
    Guard g(b->ctx);
    cudaStreamSynchronize(b->ctx->stream);
    delete b;
}

extern "C" int b200zkp_batch_shape(const b200zkp_batch* b, uint32_t shape[5]) {
    if (!b || !shape) return B200ZKP_ERR_BAD_ARG;
    shape[0] = b->n_log; shape[1] = b->k; shape[2] = b->rate_bits; shape[3] = b->cap_height; shape[4] = b->salt;
    return 0;
}

extern "C" int b200zkp_batch_cap(b200zkp_batch* b, uint64_t* out) {
    if (!b || !out) return B200ZKP_ERR_BAD_ARG;
    Guard g(b->ctx);
    return d2h(b->ctx, out, b->cap.get(), b->cap.bytes());
}
extern "C" int b200zkp_batch_coeffs(b200zkp_batch* b, uint64_t* out) {
    if (!b || !out) return B200ZKP_ERR_BAD_ARG;
    Guard g(b->ctx);
    return d2h(b->ctx, out, b->coeffs.get(), b->coeffs.bytes());
}
extern "C" int b200zkp_batch_digests(b200zkp_batch* b, uint64_t* out) {
    if (!b) return B200ZKP_ERR_BAD_ARG;
    Guard g(b->ctx);
    if (b->digests.bytes() && !out) BAD(b->ctx, "null out");
    return d2h(b->ctx, out, b->digests.get(), b->digests.bytes());
}

// leaves leave the device row-major: transpose in chunks through a bounded staging buffer
extern "C" int b200zkp_batch_leaves(b200zkp_batch* b, uint64_t* out) {
    if (!b || !out) return B200ZKP_ERR_BAD_ARG;
    b200zkp_ctx* ctx = b->ctx;
    Guard g(ctx);
    u64 N = (u64)1 << (b->n_log + b->rate_bits);
    u32 row = b->k + b->salt;
    u64 chunk_rows = std::min<u64>(N, std::max<u64>(1, ((u64)256 << 20) / ((u64)row * 8)));
    DevBuf stage;
    TRY(stage.alloc(ctx, (size_t)chunk_rows * row * 8));
    for (u64 r0 = 0; r0 < N; r0 += chunk_rows) {
        u64 nr = std::min(chunk_rows, N - r0);
        TRY(dev_transpose_rows_locked(ctx, b->lde.get(), N, row, r0, nr, stage.get()));
        TRY(d2h(ctx, out + r0 * row, stage.get(), (size_t)nr * row * 8));
    }
    return 0;
}

// MerkleTree::get + prove on the device, asynchronous: idx, rows [n_idx][row_len] and siblings [n_idx][depth][4] are
// device buffers (rows or siblings may be null); element (row, c) of a leaf is lde[c * col_stride + row].  Each index is
// reduced modulo n_leaves (a power of two), so no index reads out of range.
static int dev_gather_locked(b200zkp_ctx* ctx, const u64* lde, u64 col_stride, u32 row_len, const u64* digests, u64 n_leaves,
                             u32 depth, const u64* idx, u64 n_idx, u64* rows, u64* siblings) {
    const u64 n_rows = rows ? n_idx * row_len : 0, n_sib = siblings ? n_idx * depth : 0;
    if (n_rows) {
        merkle::gather_rows_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, ctx->stream>>>(lde, col_stride, row_len, idx, n_idx, rows,
                                                                                            n_leaves - 1);
        LAUNCH_CHECK(ctx);
    }
    if (n_sib) {
        merkle::TreeShape shape; shape.sub_log = depth; shape.sub_digests = 2 * (((u64)1 << depth) - 1);
        merkle::gather_siblings_kernel<<<(unsigned)((n_sib + 255) / 256), 256, 0, ctx->stream>>>(digests, shape, idx, n_idx, siblings,
                                                                                               n_leaves - 1);
        LAUNCH_CHECK(ctx);
    }
    return 0;
}

// the same for host indices and host outputs, synchronous; an index >= N is an error
static int gather_locked(b200zkp_ctx* ctx, const u64* lde, u64 N, u32 row, const u64* digests, u32 depth,
                         const u64* idx, u64 n_idx, u64* rows, u64* siblings) {
    if (!n_idx) return 0;
    for (u64 i = 0; i < n_idx; i++) if (idx[i] >= N) BAD(ctx, "leaf index out of range");
    DevBuf d_idx, d_rows, d_sib;
    TRY(d_idx.alloc(ctx, n_idx * 8));
    TRY(d_rows.alloc(ctx, rows ? n_idx * row * 8 : 0));
    TRY(d_sib.alloc(ctx, siblings ? n_idx * depth * 32 : 0));
    TRY(h2d(ctx, d_idx.get(), idx, d_idx.bytes()));
    TRY(dev_gather_locked(ctx, lde, N, row, digests, N, depth, d_idx.get(), n_idx, d_rows.get(), d_sib.get()));
    if (d_rows.bytes()) CUDA_TRY(ctx, cudaMemcpyAsync(rows, d_rows.get(), d_rows.bytes(), cudaMemcpyDeviceToHost, ctx->stream));
    if (d_sib.bytes()) CUDA_TRY(ctx, cudaMemcpyAsync(siblings, d_sib.get(), d_sib.bytes(), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int b200zkp_batch_rows(b200zkp_batch* b, const uint64_t* idx, uint64_t n_idx, uint64_t* rows,
                                  uint64_t* siblings) {
    if (!b || (!idx && n_idx)) return B200ZKP_ERR_BAD_ARG;
    Guard g(b->ctx);
    u32 N_log = b->n_log + b->rate_bits;
    return gather_locked(b->ctx, b->lde.get(), (u64)1 << N_log, b->k + b->salt, b->digests.get(), N_log - b->cap_height,
                         (const u64*)idx, n_idx, (u64*)rows, (u64*)siblings);
}

extern "C" int b200zkp_batch_lde_values(b200zkp_batch* b, uint64_t index, uint64_t step, uint64_t* out) {
    if (!b || !out) return B200ZKP_ERR_BAD_ARG;
    Guard g(b->ctx);
    u32 N_log = b->n_log + b->rate_bits;
    u64 N = (u64)1 << N_log;
    u64 nat = index * step;
    if (nat >= N) BAD(b->ctx, "index * step out of range");
    u64 leaf = 0;
    for (u32 i = 0; i < N_log; i++) leaf |= ((nat >> i) & 1) << (N_log - 1 - i);
    // salt columns are last, so the first k entries of the row are the polynomial values
    return gather_locked(b->ctx, b->lde.get(), N, b->k, b->digests.get(), 0, &leaf, 1, (u64*)out, nullptr);
}

extern "C" int b200zkp_batch_device_ptrs(b200zkp_batch* b, const uint64_t** coeffs, const uint64_t** lde,
                                         const uint64_t** digests, const uint64_t** cap) {
    if (!b) return B200ZKP_ERR_BAD_ARG;
    if (coeffs) *coeffs = (const uint64_t*)b->coeffs.get();
    if (lde) *lde = (const uint64_t*)b->lde.get();
    if (digests) *digests = (const uint64_t*)b->digests.get();
    if (cap) *cap = (const uint64_t*)b->cap.get();
    return 0;
}

// MerkleTree::get + prove on caller-owned device buffers (a rank's leaf shard of a sharded commitment): asynchronous.
extern "C" int b200zkp_dev_gather(b200zkp_ctx* ctx, const uint64_t* lde, uint64_t col_stride, uint32_t row_len,
                                  const uint64_t* digests, uint64_t n_leaves, uint32_t cap_height, const uint64_t* idx_dev,
                                  uint64_t n_idx, uint64_t* rows_dev, uint64_t* siblings_dev) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!n_idx) return 0;
    if (!idx_dev) BAD(ctx, "null index buffer");
    u32 lg = 0;
    if (!log2_exact(n_leaves, &lg)) BAD(ctx, "number of leaves must be a power of two");
    if (cap_height > lg) BAD(ctx, "cap_height exceeds log2(number of leaves)");
    const u32 depth = lg - cap_height;
    if (rows_dev && !lde) BAD(ctx, "null leaf buffer");
    if (siblings_dev && depth && !digests) BAD(ctx, "null digests buffer");
    return dev_gather_locked(ctx, (const u64*)lde, col_stride, row_len, (const u64*)digests, n_leaves, depth, (const u64*)idx_dev, n_idx,
                             (u64*)rows_dev, (u64*)siblings_dev);
}

// ------------------------------------------------------------------------------------------------ openings (N3)
// the two launches of every opening evaluation: m entries of L, each a column of n = 2^n_log coefficients -> d_out[m]
static int eval_list_locked(b200zkp_ctx* ctx, const evalk::EvalList& L, u32 m, u32 n_log, evalk::Ext2* d_out) {
    if (!m) return 0;
    u64 n = (u64)1 << n_log;
    // segments: enough CTAs to fill the GPU (~4 per SM), at least 1024 coefficients each
    u64 want = (4 * 148 + m - 1) / m;
    u64 n_seg = 1;
    while (n_seg < want && (n / (n_seg * 2)) >= 1024) n_seg *= 2;
    u64 seg_len = n / n_seg;
    DevBuf d_part;
    TRY(d_part.alloc(ctx, (size_t)m * n_seg * sizeof(evalk::Ext2)));
    dim3 grid((unsigned)n_seg, m);
    evalk::eval_segments_kernel<<<grid, evalk::EVAL_THREADS, 0, ctx->stream>>>(L, n, seg_len, (evalk::Ext2*)d_part.get());
    LAUNCH_CHECK(ctx);
    evalk::eval_combine_kernel<<<(m + 127) / 128, 128, 0, ctx->stream>>>(L, (const evalk::Ext2*)d_part.get(), (u32)n_seg, seg_len, m, d_out);
    LAUNCH_CHECK(ctx);
    return 0;
}

static int dev_eval_ext2_locked(b200zkp_ctx* ctx, const u64* coeffs, u64 col_stride, u32 n_log, u32 k, const u64 zeta[2],
                                u64* d_out /* k*2 */) {
    if (!k) return 0;
    if (n_log > 32) BAD(ctx, "n_log out of range");
    evalk::EvalList L{};
    L.base = coeffs; L.col_stride = col_stride;
    L.z0.a = gl_host_canon(zeta[0]); L.z0.b = gl_host_canon(zeta[1]);
    return eval_list_locked(ctx, L, k, n_log, (evalk::Ext2*)d_out);
}

extern "C" int b200zkp_dev_eval_ext2(b200zkp_ctx* ctx, const uint64_t* coeffs, uint64_t col_stride, uint32_t n_log, uint32_t k,
                                     const uint64_t zeta[2], uint64_t* out_dev) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!coeffs || !zeta || !out_dev) BAD(ctx, "null buffer");
    return dev_eval_ext2_locked(ctx, (const u64*)coeffs, col_stride, n_log, k, (const u64*)zeta, (u64*)out_dev);
}

extern "C" int b200zkp_batch_eval_ext2(b200zkp_batch* b, const uint64_t zeta[2], uint64_t* out) {
    if (!b || !zeta || !out) return B200ZKP_ERR_BAD_ARG;
    b200zkp_ctx* ctx = b->ctx;
    Guard g(ctx);
    DevBuf d_out;
    TRY(d_out.alloc(ctx, (size_t)b->k * 16));
    TRY(dev_eval_ext2_locked(ctx, b->coeffs.get(), (u64)1 << b->n_log, b->n_log, b->k, (const u64*)zeta, d_out.get()));
    return d2h(ctx, out, d_out.get(), d_out.bytes());
}

// an opening instance as b200zkp_fri_begin and b200zkp_batch_openings take it: every check before anything is launched
static int check_instance(b200zkp_ctx* ctx, b200zkp_batch* const* oracles, uint32_t n_oracles, uint32_t n_points, const uint64_t* points,
                          const uint32_t* point_n_polys, const uint32_t* poly_oracle, const uint32_t* poly_index, u32* total_out,
                          u32* max_k_out) {
    if (!oracles || !n_oracles || !n_points || !points || !point_n_polys || !poly_oracle || !poly_index)
        BAD(ctx, "null or empty argument");
    u32 n_log = oracles[0] ? oracles[0]->n_log : 0, rate_bits = oracles[0] ? oracles[0]->rate_bits : 0;
    for (u32 i = 0; i < n_oracles; i++) {
        if (!oracles[i] || oracles[i]->ctx != ctx) BAD(ctx, "oracle belongs to another context");
        if (oracles[i]->n_log != n_log || oracles[i]->rate_bits != rate_bits) BAD(ctx, "oracles differ in degree or rate");
    }
    u64 total = 0;
    u32 max_k = 0;
    for (u32 b = 0; b < n_points; b++) { total += point_n_polys[b]; max_k = std::max(max_k, point_n_polys[b]); }
    if (total > UINT32_MAX) BAD(ctx, "too many polynomials");
    for (u64 i = 0; i < total; i++) {
        if (poly_oracle[i] >= n_oracles) BAD(ctx, "oracle index out of range");
        if (poly_index[i] >= oracles[poly_oracle[i]]->k) BAD(ctx, "polynomial index out of range");
    }
    if (!max_k) BAD(ctx, "no polynomial to open");
    *total_out = (u32)total;
    *max_k_out = max_k;
    return 0;
}

extern "C" int b200zkp_batch_openings(b200zkp_ctx* ctx, b200zkp_batch* const* oracles, uint32_t n_oracles, uint32_t n_points,
                                      const uint64_t* points, const uint32_t* point_n_polys, const uint32_t* poly_oracle,
                                      const uint32_t* poly_index, uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!out) BAD(ctx, "null out");
    u32 m = 0, max_k = 0;
    TRY(check_instance(ctx, oracles, n_oracles, n_points, points, point_n_polys, poly_oracle, poly_index, &m, &max_k));
    const u32 n_log = oracles[0]->n_log;
    const u64 n = (u64)1 << n_log;
    // one table: the m entries, then the points
    std::vector<evalk::EvalEntry> tab(m + n_points);
    u32 e = 0;
    for (u32 b = 0; b < n_points; b++)
        for (u32 j = 0; j < point_n_polys[b]; j++, e++) {
            tab[e].col = oracles[poly_oracle[e]]->coeffs.get() + (u64)poly_index[e] * n;
            tab[e].point = b;
        }
    evalk::Ext2* pts = (evalk::Ext2*)(tab.data() + m);
    for (u32 b = 0; b < n_points; b++) { pts[b].a = gl_host_canon(points[2 * b]); pts[b].b = gl_host_canon(points[2 * b + 1]); }
    static_assert(sizeof(evalk::EvalEntry) == sizeof(evalk::Ext2), "points share the entry table");
    DevBuf d_tab, d_out;
    TRY(d_tab.alloc(ctx, tab.size() * sizeof(evalk::EvalEntry)));
    TRY(d_out.alloc(ctx, (size_t)m * sizeof(evalk::Ext2)));
    TRY(h2d(ctx, d_tab.get(), tab.data(), d_tab.bytes()));
    evalk::EvalList L{};
    L.entries = (const evalk::EvalEntry*)d_tab.get();
    L.points = (const evalk::Ext2*)(L.entries + m);
    TRY(eval_list_locked(ctx, L, m, n_log, (evalk::Ext2*)d_out.get()));
    return d2h(ctx, out, d_out.get(), d_out.bytes());
}

// ------------------------------------------------------------------------------------------------ opening proof (N2 + N3)
struct HostExt { u64 a, b; };
static inline u64 host_add(u64 x, u64 y) { u64 s = x + y; return (s < x || s >= hostgl::P) ? s - hostgl::P : s; }
static inline HostExt host_ext_mul(HostExt x, HostExt y) {
    HostExt r;
    r.a = host_add(hostgl::mul(x.a, y.a), hostgl::mul(7, hostgl::mul(x.b, y.b)));
    r.b = host_add(hostgl::mul(x.a, y.b), hostgl::mul(x.b, y.a));
    return r;
}
static inline HostExt host_ext_pow(HostExt x, u64 e) {
    HostExt r{1, 0};
    while (e) { if (e & 1) r = host_ext_mul(r, x); x = host_ext_mul(x, x); e >>= 1; }
    return r;
}
static inline evalk::Ext2 to_dev(HostExt x) { evalk::Ext2 r; r.a = x.a; r.b = x.b; return r; }

struct FriLayer {
    DevBuf rows, digests, cap;
    u32 arity_bits = 0, cap_height = 0;
    u64 n_leaves = 0;
};

struct b200zkp_fri {
    b200zkp_ctx* ctx = nullptr;
    u32 n_log = 0, rate_bits = 0;
    u32 cur_log = 0;          // log2 of the current (folded) LDE size
    u64 shift = 7;            // coset shift of the current values
    DevBuf coef[2];           // ping-pong coefficient planes; coef[i] = [2][cap_i], plane stride cap_i
    u64 coef_stride[2] = {};
    int cur = 0;
    DevBuf values;            // [2][N] planes, bit-reversed values of the current layer
    u64 N = 0;
    bool values_ready = false;
    int pending_arity_bits = -1;
    std::vector<FriLayer> layers;
};

static int fri_alloc_state(b200zkp_ctx* ctx, u32 n_log, u32 rate_bits, std::unique_ptr<b200zkp_fri>* out) {
    if (rate_bits > 8 || n_log + rate_bits > 32) BAD(ctx, "n_log + rate_bits exceeds two-adicity");
    std::unique_ptr<b200zkp_fri> f(new (std::nothrow) b200zkp_fri());
    if (!f) return B200ZKP_ERR_OOM;
    f->ctx = ctx; f->n_log = n_log; f->rate_bits = rate_bits; f->cur_log = n_log + rate_bits;
    f->N = (u64)1 << f->cur_log;
    f->coef_stride[0] = f->N; f->coef_stride[1] = std::max<u64>(f->N / 2, 1);
    for (int i = 0; i < 2; i++) TRY(f->coef[i].alloc(ctx, (size_t)2 * f->coef_stride[i] * 8));
    TRY(f->values.alloc(ctx, (size_t)2 * f->N * 8));
    CUDA_TRY(ctx, cudaMemsetAsync(f->coef[0].get(), 0, f->coef[0].bytes(), ctx->stream));
    *out = std::move(f);
    return 0;
}

// values = bit-reversed coset_fft(shift) of the current coefficients
static int fri_compute_values(b200zkp_fri* f) {
    b200zkp_ctx* ctx = f->ctx;
    u64 M = (u64)1 << f->cur_log;
    const u64* scale = nullptr;
    TRY(get_power_scale(ctx, f->shift, f->cur_log, &scale));
    TRY(run_transform(ctx, f->coef[f->cur].get(), f->coef_stride[f->cur], f->values.get(), M, nullptr, f->cur_log, 2, /*dir=*/0,
                      /*bitrev_out=*/true, scale, 0, /*inverse_scale=*/false, /*canon_in=*/false));
    f->values_ready = true;
    return 0;
}

extern "C" int b200zkp_fri_begin(b200zkp_ctx* ctx, b200zkp_batch* const* oracles, uint32_t n_oracles, uint32_t n_points,
                                 const uint64_t* points, const uint32_t* point_n_polys, const uint32_t* poly_oracle,
                                 const uint32_t* poly_index, const uint64_t alpha_in[2], uint32_t flags, b200zkp_fri** out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!out) BAD(ctx, "null out");
    *out = nullptr;
    if (!alpha_in) BAD(ctx, "null or empty argument");
    u32 total = 0, max_k = 0;
    TRY(check_instance(ctx, oracles, n_oracles, n_points, points, point_n_polys, poly_oracle, poly_index, &total, &max_k));
    const u32 n_log = oracles[0]->n_log, rate_bits = oracles[0]->rate_bits;
    u64 n = (u64)1 << n_log;
    std::unique_ptr<b200zkp_fri> f;
    TRY(fri_alloc_state(ctx, n_log, rate_bits, &f));
    HostExt alpha{gl_host_canon(alpha_in[0]), gl_host_canon(alpha_in[1])};
    u32 n_seg = (u32)((n + frik::SCAN_SEG - 1) / frik::SCAN_SEG);
    DevBuf d_ptrs, d_pw, d_comp, d_tot, d_carry;
    TRY(d_ptrs.alloc(ctx, (size_t)max_k * 8));
    TRY(d_pw.alloc(ctx, (size_t)max_k * 16));
    TRY(d_comp.alloc(ctx, (size_t)2 * n * 8));
    TRY(d_tot.alloc(ctx, (size_t)n_seg * 16));
    TRY(d_carry.alloc(ctx, (size_t)n_seg * 16));
    u64* fin_a = f->coef[0].get();
    u64* fin_b = f->coef[0].get() + f->coef_stride[0];
    u64* comp_a = d_comp.get();
    u64* comp_im = d_comp.get() + n;
    evalk::Ext2* pw = (evalk::Ext2*)d_pw.get();
    evalk::Ext2* tot = (evalk::Ext2*)d_tot.get();
    evalk::Ext2* carry = (evalk::Ext2*)d_carry.get();
    std::vector<const u64*> ptrs(max_k);
    u32 off = 0;
    for (u32 b = 0; b < n_points; b++) {
        u32 k = point_n_polys[b];
        if (!k) continue;       // an empty batch contributes the zero polynomial and alpha^0
        for (u32 i = 0; i < k; i++) ptrs[i] = oracles[poly_oracle[off + i]]->coeffs.get() + (u64)poly_index[off + i] * n;
        off += k;
        TRY(h2d(ctx, d_ptrs.get(), ptrs.data(), (size_t)k * 8));
        frik::ext_powers_kernel<<<(k + 127) / 128, 128, 0, ctx->stream>>>(to_dev(alpha), k, pw);
        LAUNCH_CHECK(ctx);
        frik::reduce_polys_base_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(
            (const u64* const*)d_ptrs.get(), k, n, pw, comp_a, comp_im);
        LAUNCH_CHECK(ctx);
        HostExt z{gl_host_canon(points[2 * b]), gl_host_canon(points[2 * b + 1])};
        frik::scan_totals_kernel<<<n_seg, frik::SCAN_THREADS, 0, ctx->stream>>>(comp_a, comp_im, n, to_dev(z), tot);
        LAUNCH_CHECK(ctx);
        frik::scan_carries_kernel<<<1, frik::SCAN_THREADS, 0, ctx->stream>>>(tot, n_seg, to_dev(z), carry);
        LAUNCH_CHECK(ctx);
        // alpha.shift_poly(&mut final_poly): final_poly *= alpha^count, count = polynomials of this batch
        frik::divide_by_linear_kernel<<<n_seg, frik::SCAN_THREADS, 0, ctx->stream>>>(
            comp_a, comp_im, n, to_dev(z), carry, to_dev(host_ext_pow(alpha, k)),
            (flags & B200ZKP_FRI_MUL_BY_X) ? 1u : 0u, fin_a, fin_b);
        LAUNCH_CHECK(ctx);
        // the pointer table is reused by the next batch: the copy above is stream-ordered after these kernels
    }
    TRY(fri_compute_values(f.get()));
    *out = f.release();
    return 0;
}

extern "C" int b200zkp_fri_begin_from_coeffs(b200zkp_ctx* ctx, const uint64_t* coeffs, uint32_t n_log, uint32_t rate_bits,
                                             b200zkp_fri** out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!out) BAD(ctx, "null out");
    *out = nullptr;
    if (!coeffs) BAD(ctx, "null buffer");
    std::unique_ptr<b200zkp_fri> f;
    TRY(fri_alloc_state(ctx, n_log, rate_bits, &f));
    u64 n = (u64)1 << n_log;
    // stage the interleaved input in the (still unused) values buffer
    TRY(h2d(ctx, f->values.get(), coeffs, (size_t)n * 16));
    frik::deinterleave_kernel<<<(unsigned)((2 * n + 255) / 256), 256, 0, ctx->stream>>>(f->values.get(), n, f->coef[0].get(), f->coef[0].get() + f->coef_stride[0]);
    LAUNCH_CHECK(ctx);
    TRY(fri_compute_values(f.get()));
    *out = f.release();
    return 0;
}

extern "C" void b200zkp_fri_free(b200zkp_fri* f) {
    if (!f) return;
    Guard g(f->ctx);
    cudaStreamSynchronize(f->ctx->stream);
    delete f;
}

extern "C" int b200zkp_fri_shape(const b200zkp_fri* f, uint32_t shape[4]) {
    if (!f || !shape) return B200ZKP_ERR_BAD_ARG;
    shape[0] = f->n_log; shape[1] = f->rate_bits; shape[2] = f->cur_log; shape[3] = (uint32_t)f->layers.size();
    return 0;
}

static int fri_copy_coeffs(b200zkp_fri* f, u64 len, u64* out) {
    b200zkp_ctx* ctx = f->ctx;
    if (!len) return 0;
    DevBuf d;
    TRY(d.alloc(ctx, (size_t)len * 16));
    const u64* pa = f->coef[f->cur].get();
    frik::interleave_kernel<<<(unsigned)((2 * len + 255) / 256), 256, 0, ctx->stream>>>(pa, pa + f->coef_stride[f->cur], len, d.get());
    LAUNCH_CHECK(ctx);
    return d2h(ctx, out, d.get(), d.bytes());
}

extern "C" int b200zkp_fri_coeffs(b200zkp_fri* f, uint64_t* out) {
    if (!f || !out) return B200ZKP_ERR_BAD_ARG;
    Guard g(f->ctx);
    return fri_copy_coeffs(f, (u64)1 << f->cur_log, (u64*)out);
}

extern "C" int b200zkp_fri_final_poly(b200zkp_fri* f, uint64_t* out) {
    if (!f || !out) return B200ZKP_ERR_BAD_ARG;
    Guard g(f->ctx);
    if (f->pending_arity_bits >= 0) BAD(f->ctx, "a committed layer is waiting for its beta (b200zkp_fri_fold)");
    return fri_copy_coeffs(f, ((u64)1 << f->cur_log) >> f->rate_bits, (u64*)out);
}

extern "C" int b200zkp_fri_commit_layer(b200zkp_fri* f, uint32_t arity_bits, uint32_t cap_height, uint64_t* cap_out) {
    if (!f) return B200ZKP_ERR_BAD_ARG;
    b200zkp_ctx* ctx = f->ctx;
    Guard g(ctx);
    if (!cap_out) BAD(ctx, "null cap_out");
    if (f->pending_arity_bits >= 0) BAD(ctx, "previous layer not folded yet");
    if (arity_bits == 0 || arity_bits > f->cur_log) BAD(ctx, "arity_bits out of range");
    if (cap_height > f->cur_log - arity_bits) BAD(ctx, "cap_height exceeds log2(number of leaves)");
    u64 M = (u64)1 << f->cur_log;
    FriLayer L;
    L.arity_bits = arity_bits; L.cap_height = cap_height; L.n_leaves = M >> arity_bits;
    TRY(L.rows.alloc(ctx, (size_t)M * 16));
    TRY(L.digests.alloc(ctx, (size_t)2 * (L.n_leaves - ((u64)1 << cap_height)) * 32));
    TRY(L.cap.alloc(ctx, ((size_t)32) << cap_height));
    frik::interleave_kernel<<<(unsigned)((2 * M + 255) / 256), 256, 0, ctx->stream>>>(f->values.get(), f->values.get() + M, M, L.rows.get());
    LAUNCH_CHECK(ctx);
    u32 leaf_len = 2u << arity_bits;
    TRY(dev_merkle_locked(ctx, L.rows.get(), leaf_len, 1, leaf_len, L.n_leaves, cap_height, L.digests.get(), L.cap.get()));
    TRY(d2h(ctx, cap_out, L.cap.get(), L.cap.bytes()));
    f->layers.push_back(std::move(L));
    f->pending_arity_bits = (int)arity_bits;
    return 0;
}

extern "C" int b200zkp_fri_fold(b200zkp_fri* f, const uint64_t beta_in[2]) {
    if (!f) return B200ZKP_ERR_BAD_ARG;
    b200zkp_ctx* ctx = f->ctx;
    Guard g(ctx);
    if (!beta_in) BAD(ctx, "null beta");
    if (f->pending_arity_bits < 0) BAD(ctx, "no committed layer to fold");
    u32 ab = (u32)f->pending_arity_bits;
    u64 out_len = ((u64)1 << f->cur_log) >> ab;
    int nxt = f->cur ^ 1;
    HostExt beta{gl_host_canon(beta_in[0]), gl_host_canon(beta_in[1])};
    const u64* ia = f->coef[f->cur].get();
    u64* oa = f->coef[nxt].get();
    frik::fold_kernel<<<(unsigned)((out_len + 127) / 128), 128, 0, ctx->stream>>>(
        ia, ia + f->coef_stride[f->cur], out_len, 1u << ab, to_dev(beta), oa, oa + f->coef_stride[nxt]);
    LAUNCH_CHECK(ctx);
    f->cur = nxt;
    f->cur_log -= ab;
    for (u32 i = 0; i < ab; i++) f->shift = hostgl::mul(f->shift, f->shift);   // shift = shift^arity
    f->pending_arity_bits = -1;
    f->values_ready = false;
    return fri_compute_values(f);
}

extern "C" int b200zkp_fri_query(b200zkp_fri* f, uint32_t layer, const uint64_t* idx, uint64_t n_idx, uint64_t* evals,
                                 uint64_t* siblings) {
    if (!f || (!idx && n_idx)) return B200ZKP_ERR_BAD_ARG;
    b200zkp_ctx* ctx = f->ctx;
    Guard g(ctx);
    if (layer >= f->layers.size()) BAD(ctx, "layer out of range");
    const FriLayer& L = f->layers[layer];
    if (!n_idx) return 0;
    for (u64 i = 0; i < n_idx; i++) if (idx[i] >= L.n_leaves) BAD(ctx, "leaf index out of range");
    u32 lg = 0;
    log2_exact(L.n_leaves, &lg);
    u32 depth = lg - L.cap_height, row_len = 2u << L.arity_bits;
    DevBuf d_idx, d_rows, d_sib;
    TRY(d_idx.alloc(ctx, n_idx * 8));
    TRY(d_rows.alloc(ctx, evals ? n_idx * row_len * 8 : 0));
    TRY(d_sib.alloc(ctx, siblings ? n_idx * depth * 32 : 0));
    TRY(h2d(ctx, d_idx.get(), idx, d_idx.bytes()));
    if (d_rows.bytes()) {
        u64 cnt = n_idx * row_len;
        frik::gather_rows_rm_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, ctx->stream>>>(L.rows.get(), row_len, d_idx.get(), n_idx, d_rows.get());
        LAUNCH_CHECK(ctx);
    }
    // the layer's leaves are row-major: only the siblings come from the shared gather
    TRY(dev_gather_locked(ctx, nullptr, 0, 0, L.digests.get(), L.n_leaves, depth, d_idx.get(), n_idx, nullptr, d_sib.get()));
    if (d_rows.bytes()) CUDA_TRY(ctx, cudaMemcpyAsync(evals, d_rows.get(), d_rows.bytes(), cudaMemcpyDeviceToHost, ctx->stream));
    if (d_sib.bytes()) CUDA_TRY(ctx, cudaMemcpyAsync(siblings, d_sib.get(), d_sib.bytes(), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int b200zkp_pow_grind(b200zkp_ctx* ctx, const uint64_t state[12], uint32_t witness_pos, uint32_t response_pos,
                                 uint32_t min_leading_zeros, uint64_t max_candidates, uint64_t* witness) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!state || !witness) BAD(ctx, "null buffer");
    if (witness_pos >= 12 || response_pos >= 12 || min_leading_zeros > 64) BAD(ctx, "bad argument");
    if (max_candidates == 0 || max_candidates > hostgl::P) max_candidates = hostgl::P;
    DevBuf d;
    TRY(d.alloc(ctx, 13 * 8));      // 12 state words + the running minimum
    u64 h[13];
    for (int i = 0; i < 12; i++) h[i] = gl_host_canon(state[i]);
    h[12] = ~(u64)0;
    TRY(h2d(ctx, d.get(), h, d.bytes()));
    u64 start = 0, window = (u64)1 << 18, best = ~(u64)0;
    while (start < max_candidates) {
        u64 count = std::min(window, max_candidates - start);
        frik::pow_grind_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(
            d.get(), witness_pos, response_pos, min_leading_zeros, start, count, (unsigned long long*)d.get() + 12);
        LAUNCH_CHECK(ctx);
        TRY(d2h(ctx, &best, d.get() + 12, 8));
        if (best != ~(u64)0) break;
        start += count;
        if (window < ((u64)1 << 24)) window <<= 2;
    }
    if (best == ~(u64)0) { ctx->err = "proof of work: no witness below the bound"; return B200ZKP_ERR_UNSUPPORTED; }
    *witness = best;
    return 0;
}

// ------------------------------------------------------------------------------------------------ MerkleTree
extern "C" int b200zkp_merkle_new(b200zkp_ctx* ctx, const uint64_t* leaves, uint64_t n_leaves, uint32_t leaf_len,
                                  uint32_t cap_height, b200zkp_tree** out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!out) BAD(ctx, "null out");
    *out = nullptr;
    u32 lg = 0;
    if (!log2_exact(n_leaves, &lg)) BAD(ctx, "number of leaves must be a power of two");
    if (cap_height > lg) BAD(ctx, "cap_height exceeds log2(number of leaves)");
    if (!leaves && leaf_len) BAD(ctx, "null leaves");
    std::unique_ptr<b200zkp_tree> t(new (std::nothrow) b200zkp_tree());
    if (!t) return B200ZKP_ERR_OOM;
    t->ctx = ctx; t->n_leaves = n_leaves; t->leaf_len = leaf_len; t->cap_height = cap_height;
    DevBuf d_leaves;
    TRY(t->digests.alloc(ctx, (size_t)2 * (n_leaves - ((u64)1 << cap_height)) * 32));
    TRY(t->cap.alloc(ctx, ((size_t)32) << cap_height));
    TRY(d_leaves.alloc(ctx, std::max<size_t>((size_t)n_leaves * leaf_len * 8, 8)));
    TRY(h2d(ctx, d_leaves.get(), leaves, (size_t)n_leaves * leaf_len * 8));
    TRY(dev_merkle_locked(ctx, d_leaves.get(), leaf_len, 1, leaf_len, n_leaves, cap_height, t->digests.get(), t->cap.get()));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *out = t.release();
    return 0;
}
extern "C" void b200zkp_tree_free(b200zkp_tree* t) {
    if (!t) return;
    Guard g(t->ctx);
    cudaStreamSynchronize(t->ctx->stream);
    delete t;
}
extern "C" int b200zkp_tree_cap(b200zkp_tree* t, uint64_t* out) {
    if (!t || !out) return B200ZKP_ERR_BAD_ARG;
    Guard g(t->ctx);
    return d2h(t->ctx, out, t->cap.get(), t->cap.bytes());
}
extern "C" int b200zkp_tree_digests(b200zkp_tree* t, uint64_t* out) {
    if (!t) return B200ZKP_ERR_BAD_ARG;
    Guard g(t->ctx);
    if (t->digests.bytes() && !out) BAD(t->ctx, "null out");
    return d2h(t->ctx, out, t->digests.get(), t->digests.bytes());
}
extern "C" int b200zkp_tree_prove(b200zkp_tree* t, const uint64_t* idx, uint64_t n_idx, uint64_t* siblings) {
    if (!t || (!idx && n_idx)) return B200ZKP_ERR_BAD_ARG;
    Guard g(t->ctx);
    u32 lg = 0;
    log2_exact(t->n_leaves, &lg);
    const u32 depth = lg - t->cap_height;     // 0: empty proofs, only the indices are checked
    if (!siblings && n_idx && depth) BAD(t->ctx, "null out");
    return gather_locked(t->ctx, nullptr, t->n_leaves, 0, t->digests.get(), depth, (const u64*)idx, n_idx, nullptr, (u64*)siblings);
}

// ------------------------------------------------------------------------------------------------ permutation argument (N1a)
static int dev_partial_products_locked(b200zkp_ctx* ctx, const u64* wires, u64 wires_stride, const u64* sigmas, u64 sigmas_stride,
                                       u32 n_log, u32 R, u32 degree, const u64* k_is, const u64* betas, const u64* gammas, u32 C,
                                       u64* out, u64 out_stride) {
    if (n_log > 32) BAD(ctx, "n_log out of range");
    if (!R || !degree || !C) BAD(ctx, "num_routed, degree and num_challenges must be positive");
    const u32 chunks = (R + degree - 1) / degree;
    if (chunks > (u32)perm::MAX_CHUNKS) BAD(ctx, "more than 32 chunks of routed wires");
    const u64 n = (u64)1 << n_log;
    if (wires_stride < n || sigmas_stride < n || out_stride < n) BAD(ctx, "column stride smaller than n");
    // small host vectors -> device (canonical)
    std::vector<u64> small((size_t)R + 2 * C);
    for (u32 j = 0; j < R; j++) small[j] = k_is[j] % hostgl::P;
    for (u32 c = 0; c < C; c++) { small[R + c] = betas[c] % hostgl::P; small[R + C + c] = gammas[c] % hostgl::P; }
    const u32 per = 4;
    const u32 n_blocks = (u32)((n + (u64)perm::SCAN_THREADS * per - 1) / ((u64)perm::SCAN_THREADS * per));
    DevBuf d_small, d_run, d_tot;
    TRY(d_small.alloc(ctx, small.size() * 8));
    TRY(d_run.alloc(ctx, (size_t)C * chunks * n * 8));
    TRY(d_tot.alloc(ctx, (size_t)C * n_blocks * 8));
    TRY(h2d(ctx, d_small.get(), small.data(), d_small.bytes()));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));    // `small` is a pageable host vector
    perm::Params p;
    p.wires = wires; p.wires_stride = wires_stride; p.sigmas = sigmas; p.sigmas_stride = sigmas_stride;
    p.k_is = d_small.get(); p.betas = d_small.get() + R; p.gammas = d_small.get() + R + C;
    p.omega = hostgl::root(n_log); p.n = n; p.R = R; p.degree = degree; p.chunks = chunks; p.C = C;
    perm::chunk_products_kernel<<<dim3((unsigned)((n + 127) / 128), C), 128, 0, ctx->stream>>>(p, d_run.get());
    LAUNCH_CHECK(ctx);
    perm::block_totals_kernel<<<dim3(n_blocks, C), perm::SCAN_THREADS, 0, ctx->stream>>>(d_run.get(), n, chunks, per, d_tot.get());
    LAUNCH_CHECK(ctx);
    perm::scan_totals_kernel<<<C, perm::SCAN_THREADS, 0, ctx->stream>>>(d_tot.get(), n_blocks);
    LAUNCH_CHECK(ctx);
    perm::finish_kernel<<<dim3(n_blocks, C), perm::SCAN_THREADS, 0, ctx->stream>>>(d_run.get(), d_tot.get(), n, chunks, per, C, out, out_stride);
    LAUNCH_CHECK(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int b200zkp_dev_partial_products_and_zs(b200zkp_ctx* ctx, const uint64_t* wires_dev, uint64_t wires_col_stride,
                                                   const uint64_t* sigmas_dev, uint64_t sigmas_col_stride, uint32_t n_log,
                                                   uint32_t num_routed, uint32_t degree, const uint64_t* k_is,
                                                   const uint64_t* betas, const uint64_t* gammas, uint32_t num_challenges,
                                                   uint64_t* out_dev, uint64_t out_col_stride) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!wires_dev || !sigmas_dev || !k_is || !betas || !gammas || !out_dev) BAD(ctx, "null buffer");
    return dev_partial_products_locked(ctx, (const u64*)wires_dev, wires_col_stride, (const u64*)sigmas_dev, sigmas_col_stride, n_log,
                                       num_routed, degree, (const u64*)k_is, (const u64*)betas, (const u64*)gammas, num_challenges,
                                       (u64*)out_dev, out_col_stride);
}

extern "C" int b200zkp_partial_products_and_zs(b200zkp_ctx* ctx, const uint64_t* wires, const uint64_t* sigmas, uint32_t n_log,
                                               uint32_t num_routed, uint32_t degree, const uint64_t* k_is, const uint64_t* betas,
                                               const uint64_t* gammas, uint32_t num_challenges, uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!wires || !sigmas || !k_is || !betas || !gammas || !out) BAD(ctx, "null buffer");
    if (n_log > 32 || !num_routed || !degree || !num_challenges) BAD(ctx, "bad shape");
    const u64 n = (u64)1 << n_log;
    const u32 chunks = (num_routed + degree - 1) / degree;
    const size_t in_b = (size_t)num_routed * n * 8, out_b = (size_t)num_challenges * chunks * n * 8;
    DevBuf d_w, d_s, d_o;
    TRY(d_w.alloc(ctx, in_b));
    TRY(d_s.alloc(ctx, in_b));
    TRY(d_o.alloc(ctx, out_b));
    TRY(h2d(ctx, d_w.get(), wires, in_b));
    TRY(h2d(ctx, d_s.get(), sigmas, in_b));
    TRY(dev_partial_products_locked(ctx, d_w.get(), n, d_s.get(), n, n_log, num_routed, degree, (const u64*)k_is,
                                    (const u64*)betas, (const u64*)gammas, num_challenges, d_o.get(), n));
    return d2h(ctx, out, d_o.get(), out_b);
}

// ------------------------------------------------------------------------------------------------ Hasher / field helpers
static constexpr size_t MAILBOX_BYTES = 64 << 10;
static bool mailbox_ready(b200zkp_ctx* ctx) {
    if (ctx->mailbox) return true;
    if (cudaHostAlloc(&ctx->mailbox, MAILBOX_BYTES, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(&ctx->mailbox_dev, ctx->mailbox, 0) != cudaSuccess) {
        (void)cudaGetLastError();
        if (ctx->mailbox) cudaFreeHost(ctx->mailbox);
        ctx->mailbox = ctx->mailbox_dev = nullptr;
        return false;
    }
    return true;
}

template <typename F>
static int with_io(b200zkp_ctx* ctx, const void* in, size_t in_b, void* out, size_t out_b, F body) {
    const size_t in_pad = (in_b + 255) & ~(size_t)255;
    if (in_pad + out_b <= MAILBOX_BYTES && mailbox_ready(ctx)) {
        // latency path: the kernel reads its input from and writes its result to mapped host memory
        if (in_b) memcpy(ctx->mailbox, in, in_b);
        int rc = body((u64*)ctx->mailbox_dev, (u64*)((char*)ctx->mailbox_dev + in_pad));
        if (rc) return rc;
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        if (out_b) memcpy(out, (char*)ctx->mailbox + in_pad, out_b);
        return 0;
    }
    DevBuf d_in, d_out;
    TRY(d_in.alloc(ctx, std::max<size_t>(in_b, 8)));
    TRY(d_out.alloc(ctx, std::max<size_t>(out_b, 8)));
    TRY(h2d(ctx, d_in.get(), in, in_b));
    TRY(body(d_in.get(), d_out.get()));
    return d2h(ctx, out, d_out.get(), out_b);
}

extern "C" int b200zkp_poseidon_permute(b200zkp_ctx* ctx, const uint64_t* in, uint64_t count, uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!count) return 0;
    if (!in || !out) BAD(ctx, "null buffer");
    return with_io(ctx, in, count * 96, out, count * 96, [&](u64* di, u64* dout) -> int {
        if (count <= COOP_MAX_NODES)
            merkle::permute_coop_kernel<<<(unsigned)((count * 16 + 127) / 128), 128, 0, ctx->stream>>>(di, nullptr, dout, count, 0u, ctx->round_add);
        else
            merkle::permute_kernel<<<(unsigned)((count + 127) / 128), 128, 0, ctx->stream>>>(di, dout, count);
        LAUNCH_CHECK(ctx);
        return 0;
    });
}

// iop/challenger.rs `duplexing`, chained: io = state[12] || inputs[n_inputs] in, state[12] || squeezed[8 * n_squeeze] out
extern "C" int b200zkp_duplex_chain(b200zkp_ctx* ctx, uint64_t state[12], const uint64_t* inputs, uint64_t n_inputs,
                                    uint32_t n_squeeze, uint64_t* squeezed) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!state || (n_inputs && !inputs) || (n_squeeze && !squeezed)) BAD(ctx, "null buffer");
    if (n_inputs > 4096 || n_squeeze > 512) BAD(ctx, "transcript step too large");
    std::vector<u64> in(12 + n_inputs), out(12 + (size_t)8 * n_squeeze);
    memcpy(in.data(), state, 96);
    if (n_inputs) memcpy(in.data() + 12, inputs, n_inputs * 8);
    TRY(with_io(ctx, in.data(), in.size() * 8, out.data(), out.size() * 8, [&](u64* di, u64* dout) -> int {
        merkle::duplex_chain_kernel<<<1, 32, 0, ctx->stream>>>(di, n_inputs, n_squeeze, dout, ctx->round_add);
        LAUNCH_CHECK(ctx);
        return 0;
    }));
    memcpy(state, out.data(), 96);
    if (n_squeeze) memcpy(squeezed, out.data() + 12, (size_t)n_squeeze * 64);
    return 0;
}

static int hash_rows(b200zkp_ctx* ctx, const u64* in, u64 count, u32 len, u64* out, bool noop_short) {
    if (!count) return 0;
    if ((!in && len) || !out) BAD(ctx, "null buffer");
    return with_io(ctx, in, count * len * 8, out, count * 32, [&](u64* di, u64* dout) -> int {
        merkle::TreeShape shape; shape.sub_log = 0; shape.sub_digests = 0;
        if (count <= COOP_MAX_NODES)
            merkle::leaf_hash_coop_kernel<<<(unsigned)((count * 16 + 127) / 128), 128, 0, ctx->stream>>>(di, len, 1, len, 0, count, shape, nullptr, dout, noop_short ? 1u : 0u, ctx->round_add);
        else
            merkle::leaf_hash_kernel<<<(unsigned)((count + B200ZKP_HASH_THREADS - 1) / B200ZKP_HASH_THREADS), B200ZKP_HASH_THREADS, 0, ctx->stream>>>(di, len, 1, len, 0, count, shape, nullptr, dout, noop_short ? 1u : 0u);
        LAUNCH_CHECK(ctx);
        return 0;
    });
}
extern "C" int b200zkp_hash_no_pad(b200zkp_ctx* ctx, const uint64_t* in, uint64_t count, uint32_t len, uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return hash_rows(ctx, (const u64*)in, count, len, (u64*)out, false);
}
extern "C" int b200zkp_hash_or_noop(b200zkp_ctx* ctx, const uint64_t* in, uint64_t count, uint32_t len, uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return hash_rows(ctx, (const u64*)in, count, len, (u64*)out, true);
}

extern "C" int b200zkp_two_to_one(b200zkp_ctx* ctx, const uint64_t* left, const uint64_t* right, uint64_t count,
                                  uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!count) return 0;
    if (!left || !right || !out) BAD(ctx, "null buffer");
    DevBuf d_r;
    TRY(d_r.alloc(ctx, count * 32));
    TRY(h2d(ctx, d_r.get(), right, count * 32));
    return with_io(ctx, left, count * 32, out, count * 32, [&](u64* dl, u64* dout) -> int {
        if (count <= COOP_MAX_NODES)
            merkle::permute_coop_kernel<<<(unsigned)((count * 16 + 127) / 128), 128, 0, ctx->stream>>>(dl, d_r.get(), dout, count, 1u, ctx->round_add);
        else
            merkle::two_to_one_kernel<<<(unsigned)((count + 127) / 128), 128, 0, ctx->stream>>>(dl, d_r.get(), dout, count);
        LAUNCH_CHECK(ctx);
        return 0;
    });
}

static int transform_host(b200zkp_ctx* ctx, u64* data, u32 n_log, u32 k, int dir) {
    if (!k) return 0;
    if (!data) BAD(ctx, "null buffer");
    if (n_log > 32) BAD(ctx, "n_log exceeds two-adicity");
    size_t bytes = ((size_t)k << n_log) * 8;
    DevBuf d, scratch, dout;
    TRY(d.alloc(ctx, bytes));
    TRY(scratch.alloc(ctx, bytes));
    TRY(dout.alloc(ctx, bytes));
    TRY(h2d(ctx, d.get(), data, bytes));
    u64 n = (u64)1 << n_log;
    if (dir) TRY(dev_intt_locked(ctx, d.get(), n, dout.get(), n, scratch.get(), n_log, k));
    else TRY(run_transform(ctx, d.get(), n, dout.get(), n, scratch.get(), n_log, k, 0, false, nullptr, 0, false, true));
    return d2h(ctx, data, dout.get(), bytes);
}
extern "C" int b200zkp_ntt(b200zkp_ctx* ctx, uint64_t* data, uint32_t n_log, uint32_t k) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return transform_host(ctx, (u64*)data, n_log, k, 0);
}
extern "C" int b200zkp_intt(b200zkp_ctx* ctx, uint64_t* data, uint32_t n_log, uint32_t k) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    return transform_host(ctx, (u64*)data, n_log, k, 1);
}

// PolynomialValues::coset_ifft(shift) (plonky2_field polynomial/mod.rs): values on shift * <w_n>, natural order ->
// coefficients: inverse transform, then coefficient j times shift^-j.  prove() runs it on the quotient values
// (compute_quotient_polys: quotient_values.coset_ifft(F::coset_shift()), row N1c).
static int dev_coset_intt_locked(b200zkp_ctx* ctx, const u64* values, u64 in_stride, u64* coeffs, u64 out_stride, u64* scratch,
                                 u32 n_log, u32 k, u64 shift) {
    if (n_log > 32) BAD(ctx, "n_log exceeds two-adicity");
    shift %= hostgl::P;
    if (!shift) BAD(ctx, "coset shift must be non-zero");
    if (!k) return 0;
    TRY(dev_intt_locked(ctx, values, in_stride, coeffs, out_stride, scratch, n_log, k));
    if (shift == 1 || n_log == 0) return 0;
    const u64* pw = nullptr;
    TRY(get_power_scale(ctx, hostgl::inv(shift), n_log, &pw));
    u64 n = (u64)1 << n_log;
    ntt::scale_columns_kernel<<<dim3((unsigned)((n + 255) / 256), k), 256, 0, ctx->stream>>>(coeffs, out_stride, n, pw);
    LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int b200zkp_dev_coset_intt(b200zkp_ctx* ctx, const uint64_t* values, uint64_t in_stride, uint64_t* coeffs,
                                      uint64_t out_stride, uint64_t* scratch, uint32_t n_log, uint32_t k, uint64_t shift) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!values || !coeffs) BAD(ctx, "null buffer");
    if (n_log > 10 && !scratch) BAD(ctx, "scratch required for n_log > 10");
    return dev_coset_intt_locked(ctx, (const u64*)values, in_stride, (u64*)coeffs, out_stride, (u64*)scratch, n_log, k, shift);
}

extern "C" int b200zkp_coset_intt(b200zkp_ctx* ctx, uint64_t* data, uint32_t n_log, uint32_t k, uint64_t shift) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!k) return 0;
    if (!data) BAD(ctx, "null buffer");
    if (n_log > 32) BAD(ctx, "n_log exceeds two-adicity");
    size_t bytes = ((size_t)k << n_log) * 8;
    DevBuf d, scratch, dout;
    TRY(d.alloc(ctx, bytes));
    TRY(scratch.alloc(ctx, bytes));
    TRY(dout.alloc(ctx, bytes));
    TRY(h2d(ctx, d.get(), data, bytes));
    u64 n = (u64)1 << n_log;
    TRY(dev_coset_intt_locked(ctx, d.get(), n, dout.get(), n, scratch.get(), n_log, k, shift));
    return d2h(ctx, data, dout.get(), bytes);
}

// natural-order coset LDE (an independent route from the leaf-order dev_lde: zero-pad, scale by 7^i,
// one size-N natural transform) — plonky2's own formulation of A4.
extern "C" int b200zkp_coset_lde(b200zkp_ctx* ctx, const uint64_t* coeffs, uint32_t n_log, uint32_t k,
                                 uint32_t rate_bits, uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!k) return 0;
    if (!coeffs || !out) BAD(ctx, "null buffer");
    u32 N_log = n_log + rate_bits;
    if (N_log > 32 || rate_bits > 8) BAD(ctx, "n_log + rate_bits exceeds two-adicity");
    u64 n = (u64)1 << n_log, N = (u64)1 << N_log;
    const u64* scale = nullptr;
    TRY(get_power_scale(ctx, 7, N_log, &scale));
    size_t big = (size_t)k * N * 8;
    DevBuf d_pad, d_scr, d_out;
    TRY(d_pad.alloc(ctx, big));
    TRY(d_scr.alloc(ctx, big));
    TRY(d_out.alloc(ctx, big));
    CUDA_TRY(ctx, cudaMemsetAsync(d_pad.get(), 0, big, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpy2DAsync(d_pad.get(), N * 8, coeffs, n * 8, n * 8, k, cudaMemcpyHostToDevice, ctx->stream));
    TRY(run_transform(ctx, d_pad.get(), N, d_out.get(), N, d_scr.get(), N_log, k, 0, false, scale, 0, false, true));
    return d2h(ctx, out, d_out.get(), big);
}

// ------------------------------------------------------------------------------------------------ field primitive probe
// Exposes the device field primitives one by one so tests can hit the rare carry / borrow paths directly.
__global__ void field_op_kernel(int op, const u64* __restrict__ a, const u64* __restrict__ b, u64* __restrict__ out, u64 count) {
    u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= count) return;
    u64 x = a[g], y = b[g], r = 0;
    switch (op) {
        case 0: r = gl::mul(x, y); break;                          // any x any -> canonical
        case 1: r = gl::add(gl::canon(x), gl::canon(y)); break;    // canonical + canonical
        case 2: r = gl::sub(gl::canon(x), gl::canon(y)); break;
        case 3: r = gl::canon(gl::reduce128(x, y)); break;         // (hi = y : lo = x) mod p
        case 4: r = gl::canon(gl::add_nc(x, gl::canon(y))); break; // arbitrary + canonical
        case 5: r = gl::canon(poseidon::combine3((u32)x & 0x7FFFFFFFu, (u32)(x >> 32) & 0x7FFFFFFFu, (u32)y & 0x7FFFFFFFu, gl::canon(y >> 1))); break;
        case 6: r = gl::canon(poseidon::sbox(x)); break;
        case 7: r = gl::canon(poseidon::mul_add_nc(x, y, x ^ y)); break;   // (x ^ y) + x * y
        default: break;
    }
    out[g] = r;
}

extern "C" int b200zkp_field_op(b200zkp_ctx* ctx, int op, const uint64_t* a, const uint64_t* b, uint64_t count, uint64_t* out) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!count) return 0;
    if (!a || !b || !out || op < 0 || op > 7) BAD(ctx, "bad argument");
    DevBuf d_b;
    TRY(d_b.alloc(ctx, count * 8));
    TRY(h2d(ctx, d_b.get(), b, count * 8));
    return with_io(ctx, a, count * 8, out, count * 8, [&](u64* da, u64* dout) -> int {
        field_op_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(op, da, d_b.get(), dout, count);
        LAUNCH_CHECK(ctx);
        return 0;
    });
}

// ------------------------------------------------------------------------------------------------ integer-pipe roof
// Every instruction consumes a value produced inside the loop, so ptxas cannot hoist or strength-reduce it
// (a multiply by loop-invariant operands is hoisted and the "IMAD.WIDE" chain degenerates into 64-bit adds).
template <int KIND>
__global__ void __launch_bounds__(256) int_pipe_kernel(u32 iters, u32* sink) {
    u32 a = threadIdx.x * 2654435761u + 12345u, b = blockIdx.x * 40503u + 77u;
    u64 w[8];
    u32 x[8];
    double d[8];
    const double dc = 1.0 + 1e-9 * (double)(b & 7);
    const u32 uz = poseidon::OPAQUE_ZERO;
#pragma unroll
    for (int i = 0; i < 8; i++) { w[i] = ((u64)(a + i) << 32) | (b * (i + 3)); x[i] = a * (2 * i + 1) + b; d[i] = 1.0 + 1e-6 * (double)(a & 1023) * (i + 1); }
    for (u32 it = 0; it < iters; it++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int j = (i + 1) & 7;
                if (KIND == 0) {          // IMAD.WIDE.U32 with a 64-bit accumulator, multiplicand from another chain
                    asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mad.wide.u32 %0, lo, %2, %0; }" : "+l"(w[i]) : "l"(w[j]), "r"(b));
                } else if (KIND == 1) {   // IADD3
                    asm volatile("add.u32 %0, %0, %1;" : "+r"(x[i]) : "r"(x[j]));
                } else if (KIND == 2) {   // IMAD (32-bit)
                    asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                } else if (KIND == 3) {   // alternating IMAD.WIDE / LOP3 (fma pipe + alu pipe)
                    if (i & 1) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                    else asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mad.wide.u32 %0, lo, %2, %0; }" : "+l"(w[i]) : "l"(w[(i + 2) & 7]), "r"(b));
                } else if (KIND == 4) {   // LOP3
                    asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                } else if (KIND == 5) {   // IMAD.HI.U32
                    asm volatile("mul.hi.u32 %0, %0, %1;" : "+r"(x[i]) : "r"(x[j]));
                } else if (KIND == 6) {   // alternating IMAD (32-bit) / LOP3
                    if (i & 1) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                    else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(x[(i + 2) & 7]), "r"(b));
                } else if (KIND == 7) {   // add with carry chain (IADD3 + IADD3.X)
                    asm volatile("{ add.cc.u32 %0, %0, %1; addc.u32 %0, %0, %2; }" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                } else if (KIND == 8) {   // IMAD.WIDE.U32 without an accumulator (32x32 -> 64, addend RZ)
                    asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mul.wide.u32 %0, lo, hi; }" : "=l"(w[i]) : "l"(w[j]));
                } else if (KIND == 9) {   // DFMA (FP64 pipe)
                    asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(d[i]) : "d"(dc), "d"(d[j]));
                } else if (KIND == 10) {  // alternating DFMA / IMAD.WIDE.U32: do the FP64 and multiplier pipes overlap?
                    if (i & 1) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(d[i]) : "d"(dc), "d"(d[(i + 2) & 7]));
                    else asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mad.wide.u32 %0, lo, %2, %0; }" : "+l"(w[i]) : "l"(w[(i + 2) & 7]), "r"(b));
                } else if (KIND == 11) {  // alternating DFMA / IMAD (32-bit)
                    if (i & 1) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(d[i]) : "d"(dc), "d"(d[(i + 2) & 7]));
                    else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(x[(i + 2) & 7]), "r"(b));
                } else if (KIND == 12) {  // alternating DFMA / LOP3
                    if (i & 1) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(d[i]) : "d"(dc), "d"(d[(i + 2) & 7]));
                    else asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[(i + 2) & 7]), "r"(b));
                } else if (KIND == 13) {  // alternating IMAD.WIDE.U32 (accumulating) / IMAD: both on the multiplier pipe
                    if (i & 1) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(x[(i + 2) & 7]), "r"(b));
                    else asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mad.wide.u32 %0, lo, %2, %0; }" : "+l"(w[i]) : "l"(w[(i + 2) & 7]), "r"(b));
                } else if (KIND == 14) {  // alternating IMAD.WIDE.U32 without accumulator / LOP3
                    if (i & 1) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[(i + 2) & 7]), "r"(b));
                    else asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mul.wide.u32 %0, lo, hi; }" : "=l"(w[i]) : "l"(w[(i + 2) & 7]));
                } else if (KIND == 15) {  // IMAD.WIDE.U32 (accumulating) : LOP3 = 1 : 3
                    if (i & 3) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                    else asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mad.wide.u32 %0, lo, %2, %0; }" : "+l"(w[i]) : "l"(w[(i + 4) & 7]), "r"(b));
                } else if (KIND == 16) {  // three-input IADD3 with a uniform-register operand (the pinned adds of the MDS layer)
                    x[i] = x[i] + x[j] + uz;
                } else if (KIND == 17) {  // alternating three-input IADD3 / IMAD
                    if (i & 1) x[i] = x[i] + x[(i + 2) & 7] + uz;
                    else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(x[(i + 2) & 7]), "r"(b));
                } else if (KIND == 18) {  // IMAD.WIDE (accumulating) : IMAD : LOP3 : IADD3 = 1 : 2 : 2 : 3, roughly the permutation's mix
                    if (i == 0) asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mad.wide.u32 %0, lo, %2, %0; }" : "+l"(w[0]) : "l"(w[r & 7]), "r"(b));
                    else if (i == 1 || i == 4) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                    else if (i == 2 || i == 5) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                    else x[i] = x[i] + x[j] + uz;
                } else {                  // KIND 19: IMAD.WIDE.U32 (accumulating) : LOP3 : IMAD = 1 : 2 : 1
                    if (i == 0 || i == 4) asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %1; mad.wide.u32 %0, lo, %2, %0; }" : "+l"(w[i]) : "l"(w[(i + 4) & 7]), "r"(b));
                    else if (i & 1) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                    else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(x[j]), "r"(b));
                }
            }
        }
    }
    u64 ww = 0; u32 xx = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { ww ^= w[i]; xx ^= x[i]; ww ^= (u64)__double_as_longlong(d[i]); }
    xx ^= (u32)ww ^ (u32)(ww >> 32);
    if (xx == 0xdeadbeefu && iters == 0xffffffffu) *sink = xx;   // keep the chains alive
}

extern "C" int b200zkp_int_pipe_bench(b200zkp_ctx* ctx, int kind, uint32_t iters, double* out_gips) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!out_gips || kind < 0 || kind > 19) BAD(ctx, "bad argument");
    int sms = 0;
    CUDA_TRY(ctx, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
    DevBuf sink_buf;
    TRY(sink_buf.alloc(ctx, 8));
    u32* sink = (u32*)sink_buf.get();
    unsigned blocks = (unsigned)sms * 8;
    struct Events {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        ~Events() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); }
    } ev;
    CUDA_TRY(ctx, cudaEventCreate(&ev.e0));
    CUDA_TRY(ctx, cudaEventCreate(&ev.e1));
    auto launch = [&](u32 n) {
        switch (kind) {
            case 0: int_pipe_kernel<0><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 1: int_pipe_kernel<1><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 2: int_pipe_kernel<2><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 3: int_pipe_kernel<3><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 4: int_pipe_kernel<4><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 5: int_pipe_kernel<5><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 6: int_pipe_kernel<6><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 7: int_pipe_kernel<7><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 8: int_pipe_kernel<8><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 9: int_pipe_kernel<9><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 10: int_pipe_kernel<10><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 11: int_pipe_kernel<11><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 12: int_pipe_kernel<12><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 13: int_pipe_kernel<13><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 14: int_pipe_kernel<14><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 15: int_pipe_kernel<15><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 16: int_pipe_kernel<16><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 17: int_pipe_kernel<17><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            case 18: int_pipe_kernel<18><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
            default: int_pipe_kernel<19><<<blocks, 256, 0, ctx->stream>>>(n, sink); break;
        }
        ctx->launches++;
    };
    launch(iters / 8 + 1);  // warm-up
    CUDA_TRY(ctx, cudaEventRecord(ev.e0, ctx->stream));
    launch(iters);
    CUDA_TRY(ctx, cudaEventRecord(ev.e1, ctx->stream));
    CUDA_TRY(ctx, cudaEventSynchronize(ev.e1));
    float ms = 0;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ev.e0, ev.e1));
    double instr = (double)blocks * 256.0 * (double)iters * 64.0 * (kind == 7 ? 2.0 : 1.0);   // 8 rounds x 8 instructions (x2 for the carry pair)
    *out_gips = instr / (ms * 1e-3) / 1e9;
    return 0;
}

// ------------------------------------------------------------------------------------------------ row N1b
extern "C" int b200zkp_dev_quotient_values(b200zkp_ctx* ctx, const b200zkp_vanishing_desc* d, const uint64_t* cs, uint64_t cs_stride,
                                           const uint64_t* wires, uint64_t wires_stride, const uint64_t* zpp, uint64_t zpp_stride,
                                           uint64_t* out_dev, uint64_t out_stride) {
    if (!ctx) return B200ZKP_ERR_BAD_ARG;
    Guard g(ctx);
    if (!d || !cs || !wires || !zpp || !out_dev) BAD(ctx, "null argument");
    if (!d->k_is || !d->betas || !d->gammas || !d->alphas) BAD(ctx, "null challenge / shift list");
    const u32 Cn = d->num_challenges, R = d->num_routed_wires, deg = d->quotient_degree_factor;
    if (Cn == 0 || Cn > vanish::MAX_CHALLENGES) BAD(ctx, "num_challenges must be 1..4");
    if (R == 0 || R > 128 || (R & 3) || deg == 0) BAD(ctx, "bad routed wire count / chunk size");
    if (d->n_gates == 0 || d->n_gates > vanish::MAX_GATES || d->num_selectors == 0) BAD(ctx, "bad gate list");
    const u32 Q_log = d->degree_bits + d->quotient_degree_bits;
    if (Q_log > 32 || d->quotient_degree_bits > 8) BAD(ctx, "quotient domain exceeds the field's two-adicity");
    const u64 Q = (u64)1 << Q_log, n = (u64)1 << d->degree_bits;
    if (cs_stride < Q || wires_stride < Q || zpp_stride < Q || out_stride < Q) BAD(ctx, "stride shorter than the quotient domain");
    vanish::Params p{};
    u32 max_constraints = 0;
    for (u32 i = 0; i < d->n_gates; i++) {
        const u32 kind = d->gate_kind[i];
        if (!vanish::gate_supported(kind)) { ctx->err = "gate kind not supported by the device evaluator"; return B200ZKP_ERR_UNSUPPORTED; }
        const u32 p0 = d->gate_params[i][0], p1 = d->gate_params[i][1], p2 = d->gate_params[i][2];
        if ((kind == vanish::GATE_BASE_SUM && (p0 < 2 || p0 > 64 || p1 == 0)) ||
            (kind == vanish::GATE_INTERPOLATION_HIGH_DEGREE && (p0 == 0 || p0 > 5)) ||
            (kind == vanish::GATE_INTERPOLATION_LOW_DEGREE && (p0 == 0 || p0 > 4)) ||
            ((kind == vanish::GATE_REDUCING || kind == vanish::GATE_REDUCING_EXTENSION || kind == vanish::GATE_EXPONENTIATION) && (p0 == 0 || p0 > 128)) ||
            (kind == vanish::GATE_RANDOM_ACCESS && (p0 == 0 || p0 > 6 || p1 == 0 || p1 > 64 || p2 > 2)) ||
            vanish::gate_num_wires(kind, R, p0, p1, p2) > 135)
            BAD(ctx, "gate parameters out of range for 135 wires");
        if (d->gate_selector_index[i] >= d->num_selectors || d->gate_group_begin[i] > i || d->gate_group_end[i] <= i ||
            d->gate_group_end[i] > d->n_gates)
            BAD(ctx, "gate outside its selector group");
        p.gates[i] = vanish::GateDesc{kind, d->gate_selector_index[i], d->gate_group_begin[i], d->gate_group_end[i], p0, p1, p2};
        max_constraints = std::max(max_constraints, vanish::gate_num_constraints(kind, R, 2, p0, p1, p2));
    }
    const u32 chunks = (R + deg - 1) / deg;
    p.n_terms = Cn + Cn * chunks + max_constraints;
    // small tables, one upload: k_is | alpha powers [C][n_terms] | Z_H on the coset | its inverse
    const u32 qn = 1u << d->quotient_degree_bits;
    std::vector<u64> pack(R + (size_t)Cn * p.n_terms + 2 * qn);
    for (u32 j = 0; j < R; j++) pack[j] = gl_host_canon(d->k_is[j]);
    for (u32 c = 0; c < Cn; c++) {
        u64 a = gl_host_canon(d->alphas[c]), x = 1;
        for (u32 t = 0; t < p.n_terms; t++) { pack[R + (size_t)c * p.n_terms + t] = x; x = hostgl::mul(x, a); }
        p.betas[c] = gl_host_canon(d->betas[c]);
        p.gammas[c] = gl_host_canon(d->gammas[c]);
    }
    const u64 shift_n = hostgl::pw(7, n), wq = d->quotient_degree_bits ? hostgl::root(d->quotient_degree_bits) : 1;
    u64 wpow = 1;
    for (u32 i = 0; i < qn; i++) {
        const u64 xn = hostgl::mul(shift_n, wpow);                  // x^n = 7^n w_(2^q)^i
        const u64 zh = xn ? xn - 1 : hostgl::P - 1;
        if (zh == 0) BAD(ctx, "Z_H vanishes on the coset");
        pack[R + (size_t)Cn * p.n_terms + i] = zh;
        pack[R + (size_t)Cn * p.n_terms + qn + i] = hostgl::inv(zh);
        wpow = hostgl::mul(wpow, wq);
    }
    for (int i = 0; i < 4; i++) p.pi_hash[i] = gl_host_canon(d->public_inputs_hash[i]);
    TwoLevel tw{};
    TRY(get_tw(ctx, 0, Q_log, &tw));
    DevBuf d_pack;
    TRY(d_pack.alloc(ctx, pack.size() * 8));
    TRY(h2d(ctx, d_pack.get(), pack.data(), pack.size() * 8));    // (the pageable source is staged by the runtime before cudaMemcpyAsync returns)
    p.cs = (const u64*)cs; p.wires = (const u64*)wires; p.zpp = (const u64*)zpp;
    p.cs_stride = cs_stride; p.wires_stride = wires_stride; p.zpp_stride = zpp_stride;
    p.n_log = d->degree_bits; p.q_bits = d->quotient_degree_bits;
    p.num_selectors = d->num_selectors; p.num_gate_consts = 2; p.num_routed = R; p.num_challenges = Cn;
    p.num_prods = chunks - 1; p.degree = deg; p.n_gates = d->n_gates;
    p.k_is = d_pack.get();
    p.alpha_pows = p.k_is + R;
    p.zh = p.alpha_pows + (size_t)Cn * p.n_terms;
    p.zh_inv = p.zh + qn;
    p.tw_lo = tw.lo; p.tw_hi = tw.hi; p.tw_lo_bits = tw.lo_bits;
    p.n_inv = hostgl::inv(n % hostgl::P);
    p.out = (u64*)out_dev; p.out_stride = out_stride;
    vanish::quotient_values_kernel<<<(unsigned)((Q + 127) / 128), 128, 0, ctx->stream>>>(p);
    LAUNCH_CHECK(ctx);
    return 0;
}

// ------------------------------------------------------------------------------------------------ multi-GPU (NCCL)
#include "sharded.inl"
