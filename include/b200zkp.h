/* b200zkp — C ABI of the B200-native polynomial-commitment path.
 *
 * Drop-in boundary for the one hot path of intmax-zkp-core's prover: plonky2's
 *   PolynomialBatch::from_values / from_coeffs   (plonky2/src/fri/oracle.rs)
 *   MerkleTree::new / prove                      (plonky2/src/hash/merkle_tree.rs)
 *   PoseidonHash::{hash_no_pad, two_to_one}, PoseidonPermutation::permute   (plonky2/src/hash/*.rs)
 *   fft / ifft / coset LDE                       (plonky2_field: field/src/fft.rs, polynomial/mod.rs)
 * at InternetMaximalism/plonky2 @ f99ed9c — the git dependency pinned by
 * /root/reference/Cargo.toml:12 and Cargo.lock:333-335 (its source is not vendored in the reference).
 * The reference reaches these through CircuitBuilder::build and CircuitData::prove, e.g.
 * /root/reference/src/transaction/circuits/mod.rs:158,453, src/zkdsa/circuits/mod.rs:37,326,
 * src/rollup/circuits/mod.rs:605,1247.  The Rust binding a maintainer adds is in INTEGRATION.md.
 *
 * Conventions
 *   - every field element is a uint64_t (GoldilocksField is #[repr(transparent)] over u64), host
 *     little-endian; inputs may be non-canonical (>= p), every output is canonical.
 *   - polynomial batches are column-major: k columns of n = 2^n_log elements, column c at c*n.
 *   - leaves are rows of the LDE in bit-reversed order: leaf j = LDE row bitrev(j, n_log+rate_bits);
 *     exported row-major, N = n << rate_bits rows of (k + salt) elements.
 *   - digests use plonky2's MerkleTree.digests layout (2*(N - 2^cap_height) entries of 4 elements);
 *     the cap has 2^cap_height entries of 4 elements.
 *   - all functions return 0 on success, a negative b200zkp_status otherwise; nothing throws or
 *     aborts across this boundary.  b200zkp_last_error(ctx) describes the last failure on ctx.
 *   - a ctx owns one device, one stream and its twiddle caches; calls on one ctx are serialised by an
 *     internal mutex, distinct ctxs are independent.  There is NO CPU fallback: without a CUDA
 *     device every compute entry point fails with B200ZKP_ERR_CUDA.
 *   - "_dev" entry points take device pointers (caller-owned, e.g. torch tensors) and enqueue on the
 *     ctx stream without synchronising; the others take host pointers and return when the result is
 *     in the caller's buffer.
 */
#ifndef B200ZKP_H
#define B200ZKP_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    B200ZKP_OK = 0,
    B200ZKP_ERR_BAD_ARG = -1, /* plonky2's asserts: power-of-two sizes, cap_height <= log2(N), ... */
    B200ZKP_ERR_OOM = -2,
    B200ZKP_ERR_CUDA = -3,
    B200ZKP_ERR_UNSUPPORTED = -4,
    B200ZKP_ERR_NCCL = -5
} b200zkp_status;

typedef struct b200zkp_ctx b200zkp_ctx;
typedef struct b200zkp_batch b200zkp_batch; /* plonky2 PolynomialBatch */
typedef struct b200zkp_tree b200zkp_tree;   /* plonky2 MerkleTree */

#define B200ZKP_SALT_SIZE 4 /* plonky2 fri/oracle.rs SALT_SIZE */

/* ---- library / context ------------------------------------------------------------------- */
const char* b200zkp_version(void);
/* number of CUDA devices visible, or a negative status */
int b200zkp_device_count(void);
/* stream == NULL: the ctx creates its own non-blocking stream; otherwise a cudaStream_t to share */
int b200zkp_ctx_create(int device, void* stream, b200zkp_ctx** out);
void b200zkp_ctx_destroy(b200zkp_ctx* ctx);
const char* b200zkp_last_error(const b200zkp_ctx* ctx);
int b200zkp_ctx_synchronize(b200zkp_ctx* ctx);
/* freed device buffers are cached per ctx for reuse by the next request of the same size (a prover commits the same
 * shapes over and over).  The cache holds at most `bytes` (default: 1/8 of the device memory, 22 GB on a B200 — one
 * 2^20 x 135 batch); buffers that do not fit go straight back to the driver.  b200zkp_ctx_trim synchronises the stream
 * and returns every cached buffer to the driver. */
int b200zkp_ctx_set_pool_limit(b200zkp_ctx* ctx, uint64_t bytes);
int b200zkp_ctx_trim(b200zkp_ctx* ctx);
/* number of kernels this ctx has launched since creation (bench.py's gpu_launches) */
uint64_t b200zkp_ctx_launch_count(const b200zkp_ctx* ctx);
/* per-stage device timing (CUDA events on the ctx stream around each stage; off by default).
 * b200zkp_ctx_stage_ms synchronises, returns the summed milliseconds and span counts per stage since the
 * last call, and resets them.  Labels follow plonky2's TimingTree scopes ("IFFT", "FFT + blinding",
 * "build Merkle tree" split into leaf hashing and the level reduction). */
enum { B200ZKP_STAGE_INTT = 0, B200ZKP_STAGE_LDE = 1, B200ZKP_STAGE_LEAF_HASH = 2, B200ZKP_STAGE_TREE = 3,
       B200ZKP_N_STAGES = 4 };
int b200zkp_ctx_set_timing(b200zkp_ctx* ctx, int enabled);
int b200zkp_ctx_stage_ms(b200zkp_ctx* ctx, double ms[B200ZKP_N_STAGES], uint32_t counts[B200ZKP_N_STAGES]);
/* pinned host memory for callers that want full-speed H2D/D2H */
int b200zkp_host_alloc(size_t bytes, void** out);
void b200zkp_host_free(void* p);

/* ---- PolynomialBatch::from_values / from_coeffs (host buffers) ---------------------------- */
/* values: k*n column-major evaluations on the size-n subgroup.  salt: NULL (blinding = false, every
 * config the reference uses) or 4*N column-major elements in natural LDE order (the F::rand_vec
 * columns plonky2 appends when blinding).  The batch keeps coefficients, LDE, digests and cap on the
 * device; nothing but the cap is copied back until an accessor asks. */
int b200zkp_commit_from_values(b200zkp_ctx* ctx, const uint64_t* values, uint32_t n_log, uint32_t k,
                               uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt,
                               b200zkp_batch** out);
int b200zkp_commit_from_coeffs(b200zkp_ctx* ctx, const uint64_t* coeffs, uint32_t n_log, uint32_t k,
                               uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt,
                               b200zkp_batch** out);
/* Strict drop-in ("copy-back") commit in one call: what plonky2's struct fields need, written to host buffers while the
 * device is still hashing (coefficients and row-major leaves stream out on a copy stream during the leaf hash).
 * Any of coeffs_out (k*n), leaves_out (N*(k+salt)), digests_out (4*2*(N-2^h)), cap_out (4*2^h) may be NULL;
 * out may be NULL (nothing is kept on the device) or receives the batch handle as in b200zkp_commit_from_values.
 * Use pinned host buffers (b200zkp_host_alloc) for full PCIe speed. */
int b200zkp_commit_copy_back(b200zkp_ctx* ctx, const uint64_t* in, int is_coeffs, uint32_t n_log, uint32_t k,
                             uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, uint64_t* coeffs_out,
                             uint64_t* leaves_out, uint64_t* digests_out, uint64_t* cap_out, b200zkp_batch** out);
/* the same commitment of a k x n matrix already in HBM (in_dev, column-major as for b200zkp_dev_commit; salt_dev NULL or
 * 4*N device words as for b200zkp_commit_from_values): an owned handle like the one b200zkp_commit_from_values returns,
 * which every b200zkp_batch_* call and b200zkp_fri_begin accept.  Asynchronous on the ctx stream; the inputs are only read
 * and must stay valid until the stream has run the commit.  Argument errors as for b200zkp_dev_commit; on any error *out
 * stays NULL. */
int b200zkp_batch_from_device(b200zkp_ctx* ctx, const uint64_t* in_dev, int is_coeffs, uint32_t n_log, uint32_t k,
                              uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt_dev, b200zkp_batch** out);
void b200zkp_batch_free(b200zkp_batch* b);
/* shape: n_log, k, rate_bits, cap_height, salt_size */
int b200zkp_batch_shape(const b200zkp_batch* b, uint32_t shape[5]);
int b200zkp_batch_cap(b200zkp_batch* b, uint64_t* out /* 4 * 2^cap_height */);
int b200zkp_batch_coeffs(b200zkp_batch* b, uint64_t* out /* k * n column-major */);
int b200zkp_batch_leaves(b200zkp_batch* b, uint64_t* out /* N * (k+salt) row-major */);
int b200zkp_batch_digests(b200zkp_batch* b, uint64_t* out /* 4 * 2*(N - 2^cap_height) */);
/* MerkleTree::get + MerkleTree::prove for a list of leaf indices:
 * rows: n_idx * (k+salt); siblings: n_idx * (log2 N - cap_height) * 4 (bottom-up); either may be NULL */
int b200zkp_batch_rows(b200zkp_batch* b, const uint64_t* idx, uint64_t n_idx, uint64_t* rows,
                       uint64_t* siblings);
/* PolynomialBatch::get_lde_values(index, step): leaf bitrev(index*step) without the salt, k elements */
int b200zkp_batch_lde_values(b200zkp_batch* b, uint64_t index, uint64_t step, uint64_t* out);
/* device views of a batch, valid until b200zkp_batch_free: coefficients [k][n], LDE
 * [(k+salt)][N] column-major in leaf (bit-reversed) row order, digests, cap */
int b200zkp_batch_device_ptrs(b200zkp_batch* b, const uint64_t** coeffs, const uint64_t** lde,
                              const uint64_t** digests, const uint64_t** cap);

/* ---- openings (row N3): OpeningSet::new's evaluation loop ----------------------------------- */
/* out[c] = p_c(zeta) for the k polynomials of the batch, zeta and the results in the quadratic extension
 * F_p[X]/(X^2 - 7) as (real, imaginary) pairs: zeta[2] -> out[k*2].  Runs on the coefficients already in HBM. */
int b200zkp_batch_eval_ext2(b200zkp_batch* b, const uint64_t zeta[2], uint64_t* out);
/* same on caller-owned device buffers (coeffs [k][col_stride], out_dev k*2 on the device; async on the ctx stream) */
int b200zkp_dev_eval_ext2(b200zkp_ctx* ctx, const uint64_t* coeffs, uint64_t col_stride, uint32_t n_log, uint32_t k,
                          const uint64_t zeta[2], uint64_t* out_dev);

/* OpeningSet::new in its FRI form (to_fri_openings): every polynomial of an opening instance evaluated at its point, the
 * instance described as for b200zkp_fri_begin (oracles, points, polynomials per point as (oracle, index) pairs).
 * out: 2 words per listed polynomial, batch after batch — the order the challenger observes them.  One launch pair for the
 * whole instance, one copy back.  Errors (before anything is launched): bad arg for null or empty arguments, an oracle of
 * another ctx, oracles of differing n_log or rate_bits, an oracle or polynomial index out of range. */
int b200zkp_batch_openings(b200zkp_ctx* ctx, b200zkp_batch* const* oracles, uint32_t n_oracles, uint32_t n_points,
                           const uint64_t* points, const uint32_t* point_n_polys, const uint32_t* poly_oracle,
                           const uint32_t* poly_index, uint64_t* out);

/* ---- opening proof (rows N2 + N3): PolynomialBatch::prove_openings / fri_proof ---------------- */
/* Replaces the data-parallel steps of plonky2 @ f99ed9c  fri/oracle.rs `prove_openings`, fri/prover.rs
 * `fri_committed_trees`, `fri_proof_of_work`, `fri_prover_query_round`; the Fiat-Shamir challenger stays with the caller,
 * who feeds each challenge back in (alpha, the betas) exactly where plonky2 draws it.  All big data stays in HBM.
 *
 * b200zkp_fri_begin: final_poly = sum over opening points b of  alpha^(..) * (F_b(X) - F_b(z_b)) / (X - z_b),
 * F_b = sum_j alpha^j f_bj (ReducingFactor::reduce_polys_base, divide_by_linear, shift_poly), multiplied by X when
 * B200ZKP_FRI_MUL_BY_X is set (the 2022 plonky2 does, see DESIGN.md), then its LDE on the coset 7<w_N> in bit-reversed
 * order.  oracles: batches of equal n_log and rate_bits on this ctx; point b opens polynomials
 * (poly_oracle[i], poly_index[i]) for the next point_n_polys[b] entries i of the concatenated lists;
 * points: n_points * 2 words. */
typedef struct b200zkp_fri b200zkp_fri;
enum { B200ZKP_FRI_MUL_BY_X = 1 };
int b200zkp_fri_begin(b200zkp_ctx* ctx, b200zkp_batch* const* oracles, uint32_t n_oracles, uint32_t n_points,
                      const uint64_t* points, const uint32_t* point_n_polys, const uint32_t* poly_oracle,
                      const uint32_t* poly_index, const uint64_t alpha[2], uint32_t flags, b200zkp_fri** out);
/* same state from extension coefficients given by the caller: coeffs n * 2 words, (real, imaginary) interleaved */
int b200zkp_fri_begin_from_coeffs(b200zkp_ctx* ctx, const uint64_t* coeffs, uint32_t n_log, uint32_t rate_bits,
                                  b200zkp_fri** out);
void b200zkp_fri_free(b200zkp_fri* f);
/* shape: degree log n_log, rate_bits, log2 of the current (folded) LDE size, committed layers */
int b200zkp_fri_shape(const b200zkp_fri* f, uint32_t shape[4]);
/* current coefficients, zero-padded to the current LDE size: 2^shape[2] * 2 words interleaved */
int b200zkp_fri_coeffs(b200zkp_fri* f, uint64_t* out);
/* one reduction layer of fri_committed_trees: MerkleTree::new over the bit-reversed values chunked by 2^arity_bits
 * (leaf = 2 * arity words); cap_out 4 * 2^cap_height.  Follow with b200zkp_fri_fold(beta): coefficients are folded
 * (reduce_with_powers over chunks of arity), the coset shift is raised to the arity, values = coset_fft. */
int b200zkp_fri_commit_layer(b200zkp_fri* f, uint32_t arity_bits, uint32_t cap_height, uint64_t* cap_out);
int b200zkp_fri_fold(b200zkp_fri* f, const uint64_t beta[2]);
/* final_poly: the current coefficients truncated to len >> rate_bits: (2^shape[2] >> rate_bits) * 2 words */
int b200zkp_fri_final_poly(b200zkp_fri* f, uint64_t* out);
/* FriQueryStep for leaves idx of committed layer `layer`: evals n_idx * 2 * arity words (tree.get),
 * siblings n_idx * (log2 leaves - cap_height) * 4 (tree.prove); either may be NULL */
int b200zkp_fri_query(b200zkp_fri* f, uint32_t layer, const uint64_t* idx, uint64_t n_idx, uint64_t* evals,
                      uint64_t* siblings);
/* fri_proof_of_work: the SMALLEST w < max_candidates (0: the whole field) for which
 * permute(state with state[witness_pos] = w)[response_pos] has >= min_leading_zeros leading zero bits as a canonical
 * u64 (plonky2 grinds with rayon find_any, so any witness verifies; the smallest makes proofs reproducible).
 * hash_no_pad(current_hash || w).elements[0]: state = (h0..h3, 0 x 8), witness_pos 4, response_pos 0.
 * Returns B200ZKP_ERR_UNSUPPORTED when no candidate below the bound qualifies. */
int b200zkp_pow_grind(b200zkp_ctx* ctx, const uint64_t state[12], uint32_t witness_pos, uint32_t response_pos,
                      uint32_t min_leading_zeros, uint64_t max_candidates, uint64_t* witness);

/* ---- MerkleTree::new (host buffers) -------------------------------------------------------- */
/* leaves: n_leaves rows of leaf_len elements, row-major.  hash_or_noop: leaf_len <= 4 is not hashed. */
int b200zkp_merkle_new(b200zkp_ctx* ctx, const uint64_t* leaves, uint64_t n_leaves, uint32_t leaf_len,
                       uint32_t cap_height, b200zkp_tree** out);
void b200zkp_tree_free(b200zkp_tree* t);
int b200zkp_tree_cap(b200zkp_tree* t, uint64_t* out);
int b200zkp_tree_digests(b200zkp_tree* t, uint64_t* out);
int b200zkp_tree_prove(b200zkp_tree* t, const uint64_t* idx, uint64_t n_idx, uint64_t* siblings);

/* ---- Hasher / field helpers (host buffers, batched) --------------------------------------- */
int b200zkp_poseidon_permute(b200zkp_ctx* ctx, const uint64_t* in, uint64_t count, uint64_t* out); /* 12 each */
int b200zkp_hash_no_pad(b200zkp_ctx* ctx, const uint64_t* in, uint64_t count, uint32_t len, uint64_t* out);
int b200zkp_hash_or_noop(b200zkp_ctx* ctx, const uint64_t* in, uint64_t count, uint32_t len, uint64_t* out);
int b200zkp_two_to_one(b200zkp_ctx* ctx, const uint64_t* left, const uint64_t* right, uint64_t count,
                       uint64_t* out);
/* The Fiat-Shamir transcript (plonky2 iop/challenger.rs `Challenger::duplexing`), any number of steps in ONE launch:
 * every chunk of up to 8 of the n_inputs pending observations overwrites the head of state[12] (overwrite-mode sponge) and is
 * followed by a permutation; then n_squeeze further permutations run, each appending its 8 rate words to `squeezed`
 * (8 * n_squeeze words).  state is updated in place.  A transcript that defers its observations until the next challenge is
 * drawn makes one call where it made one b200zkp_poseidon_permute per 8 elements (host mirror: fri.py Challenger). */
int b200zkp_duplex_chain(b200zkp_ctx* ctx, uint64_t state[12], const uint64_t* inputs, uint64_t n_inputs,
                         uint32_t n_squeeze, uint64_t* squeezed);
/* in-place transforms of k columns of 2^n_log elements (natural order in and out) */
int b200zkp_ntt(b200zkp_ctx* ctx, uint64_t* data, uint32_t n_log, uint32_t k);
int b200zkp_intt(b200zkp_ctx* ctx, uint64_t* data, uint32_t n_log, uint32_t k);
/* PolynomialValues::coset_ifft(shift) (plonky2_field polynomial/mod.rs): k columns of values on shift * <w_n>, natural
 * order, in place -> coefficients.  prove() runs it on the quotient values (compute_quotient_polys, shift = 7) before
 * cutting them into degree-n chunks for PolynomialBatch::from_coeffs (row N1c).  Error: bad arg for shift = 0 mod p. */
int b200zkp_coset_intt(b200zkp_ctx* ctx, uint64_t* data, uint32_t n_log, uint32_t k, uint64_t shift);
/* coset LDE: coeffs k*n -> out k*N, out[c][i] = p_c(7 * w_N^i), natural order (A4) */
int b200zkp_coset_lde(b200zkp_ctx* ctx, const uint64_t* coeffs, uint32_t n_log, uint32_t k,
                      uint32_t rate_bits, uint64_t* out);

/* ---- device-resident stages (caller-owned device buffers; async on the ctx stream) --------- */
/* values [k][in_stride] -> coeffs [k][out_stride], natural order.  scratch: k*n elements, may alias
 * nothing; needed when n_log > 10 (may be NULL otherwise). */
int b200zkp_dev_intt(b200zkp_ctx* ctx, const uint64_t* values, uint64_t in_stride, uint64_t* coeffs,
                     uint64_t out_stride, uint64_t* scratch, uint32_t n_log, uint32_t k);
/* device form of b200zkp_coset_intt: values [k][in_stride] -> coeffs [k][out_stride]; scratch as for b200zkp_dev_intt */
int b200zkp_dev_coset_intt(b200zkp_ctx* ctx, const uint64_t* values, uint64_t in_stride, uint64_t* coeffs,
                           uint64_t out_stride, uint64_t* scratch, uint32_t n_log, uint32_t k, uint64_t shift);
/* coeffs [k][coeff_stride] -> lde [k][lde_stride] in leaf order, only leaf blocks
 * [block_begin, block_end) of the 2^rate_bits coset blocks (block b = leaves [b*n, (b+1)*n), i.e. the
 * coset 7*w_N^bitrev(b)); block b is written at column offset (b - block_begin)*n. */
int b200zkp_dev_lde(b200zkp_ctx* ctx, const uint64_t* coeffs, uint64_t coeff_stride, uint64_t* lde,
                    uint64_t lde_stride, uint32_t n_log, uint32_t k, uint32_t rate_bits,
                    uint32_t block_begin, uint32_t block_end);
/* salt [4][N] natural order -> rows of lde columns in leaf order for blocks [block_begin, block_end) */
int b200zkp_dev_salt(b200zkp_ctx* ctx, const uint64_t* salt, uint64_t* lde_salt_cols, uint64_t lde_stride,
                     uint32_t n_log, uint32_t rate_bits, uint32_t block_begin, uint32_t block_end);
/* F::rand_vec on the device: out_dev[e] = element (first + e) of the stream (key, nonce), e < count; async on the ctx stream.
 * The stream: ChaCha20 of RFC 8439 (20 rounds, key and nonce read as little-endian words, 32-bit block counter from 0).
 * Element j is keystream bytes [16 j, 16 j + 16) read as little-endian u64 lo, hi: (lo + 2^64 hi) mod p, canonical (within
 * 2^-64 of uniform; plonky2's own draw is exactly uniform).  key and nonce are host pointers, read before the call returns.
 * The salts of a blinded commitment: 4N elements, element c*N + i = salt column c at natural LDE row i, the salt_dev layout
 * of b200zkp_batch_from_device.  The key must be secret and fresh for every proof (drawn from the OS); a nonce per oracle.
 * count == 0 launches nothing.  B200ZKP_ERR_BAD_ARG: a null key, nonce or out_dev with count > 0, or a range that needs a
 * block counter of 2^32 or more (first + count > 2^34). */
int b200zkp_dev_random_field(b200zkp_ctx* ctx, const uint8_t key[32], const uint8_t nonce[12], uint64_t first,
                             uint64_t count, uint64_t* out_dev);
/* Merkle forest over n_leaves leaves, element (row, c) at leaves[row*row_stride + c*col_stride]:
 * digests 4*2*(n_leaves - 2^cap_height), cap 4*2^cap_height (both device). */
int b200zkp_dev_merkle(b200zkp_ctx* ctx, const uint64_t* leaves, uint64_t row_stride, uint64_t col_stride,
                       uint32_t leaf_len, uint64_t n_leaves, uint32_t cap_height, uint64_t* digests,
                       uint64_t* cap);
/* b200zkp_dev_lde + b200zkp_dev_merkle over the same leaf blocks (leaves (block_end - block_begin) * n, cap_height counted
 * within that range), software-pipelined: the transforms of block b+1 run on a second stream while block b is hashed. */
int b200zkp_dev_lde_merkle(b200zkp_ctx* ctx, const uint64_t* coeffs, uint64_t coeff_stride, uint64_t* lde,
                           uint64_t lde_stride, uint32_t n_log, uint32_t k, uint32_t rate_bits, uint32_t block_begin,
                           uint32_t block_end, uint32_t cap_height, uint64_t* digests, uint64_t* cap);
/* whole commitment on caller-owned device buffers (what bench.py times with inputs resident in HBM):
 * in [k][n] -> coeffs [k][n], lde [(k+salt)][N], digests, cap.  is_coeffs selects from_coeffs. */
int b200zkp_dev_commit(b200zkp_ctx* ctx, const uint64_t* in, int is_coeffs, uint32_t n_log, uint32_t k,
                       uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, uint64_t* coeffs,
                       uint64_t* lde, uint64_t* digests, uint64_t* cap);
/* MerkleTree::get + MerkleTree::prove on caller-owned device buffers (e.g. one rank's leaf shard): element (row, c) at
 * lde[c*col_stride + row]; idx_dev n_idx leaf indices on the device; rows_dev n_idx*row_len, siblings_dev
 * n_idx*(log2 n_leaves - cap_height)*4, either may be NULL.  The indices live on the device and cannot be validated by
 * the host: each is reduced modulo n_leaves (never an out-of-range read) */
int b200zkp_dev_gather(b200zkp_ctx* ctx, const uint64_t* lde, uint64_t col_stride, uint32_t row_len,
                       const uint64_t* digests, uint64_t n_leaves, uint32_t cap_height, const uint64_t* idx_dev,
                       uint64_t n_idx, uint64_t* rows_dev, uint64_t* siblings_dev);
/* column-major [cols][col_stride] rows [row0,row0+n_rows) -> row-major [n_rows][cols] (device) */
int b200zkp_dev_transpose_to_rows(b200zkp_ctx* ctx, const uint64_t* cm, uint64_t col_stride, uint32_t cols,
                                  uint64_t row0, uint64_t n_rows, uint64_t* rm);
/* Row N1a — permutation argument: the Z and partial-product polynomials prove() commits after the wires.
 * Replaces plonky2 @ f99ed9c plonky2/src/plonk/prover.rs `all_wires_permutation_partial_products` /
 * `wires_permutation_partial_products_and_zs` (with `quotient_chunk_products`, `partial_products_and_z_gx`), reached from
 * the reference through every prove() (/root/reference/src/transaction/circuits/mod.rs:453, src/zkdsa/circuits/mod.rs:326,
 * src/rollup/circuits/mod.rs:1247).
 * wires, sigmas: num_routed columns of n = 2^n_log values, column-major (the routed wires are the first columns of the
 * witness matrix handed to commit_from_values; sigmas = ProverOnlyCircuitData::sigmas transposed); k_is[num_routed]
 * (CommonCircuitData::k_is, 7^j), betas / gammas[num_challenges]; degree = quotient_degree_factor (chunk size).
 * out: num_challenges * ceil(num_routed / degree) columns of n canonical values in the order of the committed batch:
 * Z of every challenge, then the num_partial_products = ceil(num_routed / degree) - 1 partial products challenge by
 * challenge.  The _dev_ form takes device pointers with column strides (so `out` can feed b200zkp_dev_commit directly);
 * k_is / betas / gammas are always host arrays.  Errors: bad arg for zero sizes, more than 32 chunks, strides < n. */
int b200zkp_partial_products_and_zs(b200zkp_ctx* ctx, const uint64_t* wires, const uint64_t* sigmas, uint32_t n_log,
                                    uint32_t num_routed, uint32_t degree, const uint64_t* k_is, const uint64_t* betas,
                                    const uint64_t* gammas, uint32_t num_challenges, uint64_t* out);
int b200zkp_dev_partial_products_and_zs(b200zkp_ctx* ctx, const uint64_t* wires_dev, uint64_t wires_col_stride,
                                        const uint64_t* sigmas_dev, uint64_t sigmas_col_stride, uint32_t n_log,
                                        uint32_t num_routed, uint32_t degree, const uint64_t* k_is, const uint64_t* betas,
                                        const uint64_t* gammas, uint32_t num_challenges, uint64_t* out_dev,
                                        uint64_t out_col_stride);

/* ---- row N1b: compute_quotient_polys — the vanishing polynomial on the quotient coset, divided by Z_H -----------------
 * Replaces plonky2 @ f99ed9c plonk/prover.rs `compute_quotient_polys` up to its coset_ifft (b200zkp_dev_coset_intt does
 * that, b200zkp_dev_commit(is_coeffs) commits the chunks), with plonk/vanishing_poly.rs `eval_vanishing_poly_base_batch`
 * and the eval_unfiltered of the gate types below; reached from every prove() of the reference
 * (/root/reference/src/rollup/circuits/mod.rs:1247, src/transaction/circuits/mod.rs:453).  It reads the three LDEs where
 * the commitments left them (device, column-major, leaf order), so no LDE crosses PCIe any more.
 * The circuit description is what CommonCircuitData holds: the gate list in CircuitBuilder's order (sorted by degree) with
 * each gate's selector polynomial and selector group (gates/selectors.rs), num_constants = num_selectors + 2 gate constants,
 * standard_recursion_config's 135 wires / 80 routed wires.  Gate types evaluated: NoopGate, ConstantGate (2 constants),
 * PublicInputGate, ArithmeticGate (20 ops), PoseidonGate, PoseidonMdsGate, BaseSumGate<B>, ArithmeticExtensionGate,
 * MulExtensionGate, ReducingGate, ReducingExtensionGate, RandomAccessGate, ExponentiationGate,
 * HighDegreeInterpolationGate, LowDegreeInterpolationGate; any other kind (the u32 / comparison gates, id 13) is
 * B200ZKP_ERR_UNSUPPORTED (not silently skipped).  The wire layouts are restated from memory of plonky2 @ f99ed9c
 * (parity unpinned, as for every gate here; DESIGN.md section 4d). */
enum { B200ZKP_GATE_NOOP = 0, B200ZKP_GATE_CONSTANT = 1, B200ZKP_GATE_PUBLIC_INPUT = 2, B200ZKP_GATE_ARITHMETIC = 3,
       B200ZKP_GATE_POSEIDON = 4,
       /* gates with parameters take them from gate_params[i] = { p0, p1, p2 } (Gate::new_from_config values in brackets) */
       B200ZKP_GATE_ARITHMETIC_EXTENSION = 5, /* ArithmeticExtensionGate, 10 ops */
       B200ZKP_GATE_MUL_EXTENSION = 6,        /* MulExtensionGate, 13 ops */
       B200ZKP_GATE_BASE_SUM = 7,             /* BaseSumGate<B>: { B, num_limbs } [2, 63] */
       B200ZKP_GATE_REDUCING = 8,             /* ReducingGate: { num_coeffs } [43] */
       B200ZKP_GATE_REDUCING_EXTENSION = 9,   /* ReducingExtensionGate: { num_coeffs } [32] */
       B200ZKP_GATE_RANDOM_ACCESS = 10,       /* RandomAccessGate: { bits, num_copies, num_extra_constants } [e.g. 4, 4, 2] */
       B200ZKP_GATE_EXPONENTIATION = 11,      /* ExponentiationGate: { num_power_bits } [66] */
       B200ZKP_GATE_POSEIDON_MDS = 12,        /* PoseidonMdsGate */
       /* 13 is not assigned.  The interpolation gates (gates/interpolation.rs, low_degree_interpolation.rs) take
        * { subgroup_bits }: m = 2^subgroup_bits points of the coset shift * <g>, g = the primitive 2^subgroup_bits-th root of
        * unity (the NTT's); D = 2, ext(j) = wires j, j + 1 as one element of F[X]/(X^2 - 7).  Shared layout: wire 0 the
        * shift; value(i) = ext(1 + D i), i < m; evaluation point ext(1 + D m); evaluation value ext(3 + D m); coeff(i) =
        * ext(5 + D m + D i), i < m; end_coeffs = 5 + 4m; the first 5 + 2m wires are routed. */
       B200ZKP_GATE_INTERPOLATION_HIGH_DEGREE = 14, /* HighDegreeInterpolationGate { subgroup_bits 1..5 }: constraints
        * value(i) - interpolant(shift g^i) for i < m, then eval_value - interpolant(eval_point), D components each:
        * D (m + 1) constraints, 5 + 4m wires, degree m (a FRI arity <= 8) */
       B200ZKP_GATE_INTERPOLATION_LOW_DEGREE = 15 };  /* LowDegreeInterpolationGate { subgroup_bits 1..4 }: also
        * shift_pow(i) = wire end_coeffs + i - 2 and eval_pow(i) = ext(end_coeffs + m - 2 + D (i - 2)) for 2 <= i < m
        * (shift_pow(1) = shift, eval_pow(1) = eval_point).  Constraints: shift_pow(i-1) shift - shift_pow(i), 2 <= i < m;
        * value(i) - sum_j c_j shift_pow(j) g^(ij), i < m (shift_pow(0) = 1); eval_pow(i-1) eval_point - eval_pow(i),
        * 2 <= i < m; eval_value - (c_0 + sum_(i>=1) c_i eval_pow(i)): 5m - 4 constraints, 7m - 1 wires, degree 2 (what
        * standard_recursion_config's arity-16 FRI verifier instantiates, subgroup_bits 4) */
#define B200ZKP_MAX_GATES 16
typedef struct {
    uint32_t degree_bits;               /* n = 2^degree_bits rows */
    uint32_t quotient_degree_bits;      /* the quotient is evaluated on n << quotient_degree_bits points (<= rate_bits of the LDEs) */
    uint32_t quotient_degree_factor;    /* chunk size of the permutation argument (max_degree of check_partial_products) */
    uint32_t num_routed_wires;          /* 80 */
    uint32_t num_challenges;            /* <= 4 */
    uint32_t num_selectors;
    uint32_t n_gates;
    uint32_t gate_kind[B200ZKP_MAX_GATES], gate_selector_index[B200ZKP_MAX_GATES];
    uint32_t gate_group_begin[B200ZKP_MAX_GATES], gate_group_end[B200ZKP_MAX_GATES];
    uint32_t gate_params[B200ZKP_MAX_GATES][3];
    const uint64_t* k_is;               /* num_routed_wires coset shifts (host) */
    const uint64_t *betas, *gammas, *alphas;   /* num_challenges each (host) */
    uint64_t public_inputs_hash[4];
} b200zkp_vanishing_desc;
/* constants_sigmas [num_selectors + 2 + num_routed_wires][cs_stride], wires [135][wires_stride], zs_partial_products
 * [num_challenges * ceil(num_routed / factor)][zpp_stride]: device LDEs in leaf order (what b200zkp_dev_commit wrote), every
 * stride >= n << quotient_degree_bits.  out_dev: [num_challenges][out_stride] quotient values in natural order on 7 <w>. */
int b200zkp_dev_quotient_values(b200zkp_ctx* ctx, const b200zkp_vanishing_desc* desc, const uint64_t* constants_sigmas,
                                uint64_t cs_stride, const uint64_t* wires, uint64_t wires_stride,
                                const uint64_t* zs_partial_products, uint64_t zpp_stride, uint64_t* out_dev, uint64_t out_stride);

/* ---- one commitment partitioned over several GPUs (SURVEY.md 8e; NVLink / NVSwitch peer memory + NCCL) --------------
 * north_star's partition: rank g of G (a power of two, G <= 2^rate_bits and G <= 2^cap_height) inverse-transforms its columns
 * into its "exchange window"; every rank then extends ALL k columns on its 2^rate_bits/G coset blocks = leaves
 * [g*N/G, (g+1)*N/G), hashes them and builds its 2^cap_height/G cap subtrees without further communication; one ncclAllGather
 * of 32 * 2^cap_height bytes hands every rank the cap.
 * Columns are dealt to the ranks in groups of L = max(8, G): rank g owns the w = L/G columns [j*L + g*w, j*L + (g+1)*w) of every
 * group j (b200zkp_sharded_columns lists them).  A group is a whole number of sponge chunks, so with host inputs the leaves are
 * hashed group by group while later groups are still being uploaded.
 * The all-gather of the coefficients has two forms:
 *   peer exchange (default when every rank can map every other rank's memory: peer access inside one process, CUDA IPC
 *     between processes, at most 8 ranks): the first pass of the coset transforms reads its coefficient tiles straight from
 *     the owners' windows over NVLink and files them in the local coefficient matrix on the way (one fused kernel, no NCCL
 *     call, no staging); ordering by epoch-stamped flags in peer memory (CUDA events inside one process).  Host inputs form a
 *     pipeline of column chunks: upload / inverse transform / gather + coset transforms / sponge absorption.
 *   NCCL exchange (fallback, or b200zkp_comm_set_peer_exchange(comm, 0)): point-to-point groups into
 *     a local gather buffer after the inverse transforms; the same kernels then read the shards from there.
 *
 * Two ways to form the communicator, matching how the caller is deployed:
 *   b200zkp_comm_init_all   ONE process drives n GPUs (what a single rayon `prove()` process needs; plonky2 is one process,
 *                           /root/reference/Cargo.toml:19-21): ctxs[i] is rank i (distinct devices).  Each entry point below
 *                           then serves all n ranks, internally on one host thread per rank.
 *   b200zkp_comm_init_rank  one process per GPU (torchrun / MPI style): rank 0 makes an id with b200zkp_comm_unique_id,
 *                           hands it to the others out of band, every process calls init_rank with its ctx.
 * libnccl.so.2 is loaded on first use (dlopen; a copy already loaded by the host process, e.g. torch's, is reused): the
 * single-GPU entry points do not need NCCL.  Errors: B200ZKP_ERR_NCCL, text in b200zkp_comm_last_error. */
typedef struct b200zkp_comm b200zkp_comm;
typedef struct b200zkp_sharded b200zkp_sharded; /* a PolynomialBatch whose leaves are partitioned over the ranks */
#define B200ZKP_COMM_ID_BYTES 128
int b200zkp_comm_unique_id(uint8_t id[B200ZKP_COMM_ID_BYTES]);
int b200zkp_comm_init_rank(b200zkp_ctx* ctx, const uint8_t id[B200ZKP_COMM_ID_BYTES], int rank, int world,
                           b200zkp_comm** out);
int b200zkp_comm_init_all(b200zkp_ctx* const* ctxs, int n, b200zkp_comm** out);
void b200zkp_comm_destroy(b200zkp_comm* comm);
const char* b200zkp_comm_last_error(const b200zkp_comm* comm);
/* shape: world size, ranks driven by this process (1 after init_rank, world after init_all), global rank of local rank 0 */
int b200zkp_comm_shape(const b200zkp_comm* comm, int32_t shape[3]);
/* NCCL exchange: peers per group (default 2; 0 = the whole exchange in one group, i.e. no overlap with the transforms) */
int b200zkp_comm_set_exchange_group(b200zkp_comm* comm, uint32_t peers_per_group);
/* choose between the two forms of the exchange (collective: the same value on every process, between commits);
 * b200zkp_comm_peer_exchange: 1 when the peer form is the one in use (it was set up successfully and is switched on) */
int b200zkp_comm_set_peer_exchange(b200zkp_comm* comm, int enabled);
int b200zkp_comm_peer_exchange(const b200zkp_comm* comm);

/* buffers of one partitioned commitment on every local rank (coefficients of all k columns, the rank's leaf range of the
 * LDE, its digests, the full cap); reusable for any number of commits of that shape */
int b200zkp_sharded_create(b200zkp_comm* comm, uint32_t n_log, uint32_t k, uint32_t rate_bits, uint32_t cap_height,
                           b200zkp_sharded** out);
void b200zkp_sharded_free(b200zkp_sharded* sh);
/* partition of local rank `local`: lay = { n_cols, L, w, block_begin, block_end, N_local, cap_begin, cap_end }: the rank owns
 * n_cols columns, w of every group of L (see above); coset blocks / leaves / cap entries as ranges */
int b200zkp_sharded_layout(const b200zkp_sharded* sh, int local, uint64_t lay[8]);
/* the columns of local rank `local` in increasing order (cols may be NULL to ask for the count only) */
int b200zkp_sharded_columns(const b200zkp_sharded* sh, int local, uint32_t* cols, uint32_t capacity, uint32_t* n_cols);
/* PolynomialBatch::from_values / from_coeffs, partitioned.  inputs[i]: the columns of local rank i (b200zkp_sharded_columns)
 * packed in increasing order, column-major n_cols * n words, host memory (pinned for full PCIe speed; the upload is chunked and
 * overlaps the transforms and the hashing) or, with inputs_on_device, memory of that rank's device (read on the ctx stream); the same
 * kind of input on every rank.
 * cap_out: NULL -> the call only enqueues (results are complete after b200zkp_sharded_synchronize); else 4 * 2^cap_height
 * words of host memory, written before the call returns.  Collective: every process of the communicator calls it. */
int b200zkp_sharded_commit(b200zkp_sharded* sh, const uint64_t* const* inputs, int inputs_on_device, int is_coeffs,
                           uint64_t* cap_out);
/* convenience for the one-process deployment and for tests: `values` is the FULL k*n column-major host matrix (every
 * process passes the same one); creates the buffers, commits, returns the cap */
int b200zkp_sharded_commit_from_values(b200zkp_comm* comm, const uint64_t* values, uint32_t n_log, uint32_t k,
                                       uint32_t rate_bits, uint32_t cap_height, uint64_t* cap_out, b200zkp_sharded** out);
int b200zkp_sharded_synchronize(b200zkp_sharded* sh);
/* device views on local rank `local`: coefficients [ceil(k/L)*L][n] (all columns, natural column order, zero columns past k),
 * LDE [k][N_local] (the rank's leaves, column-major), digests of its cap subtrees (plonky2 layout), the full cap */
int b200zkp_sharded_device_ptrs(b200zkp_sharded* sh, int local, const uint64_t** coeffs, const uint64_t** lde,
                                const uint64_t** digests, const uint64_t** cap);
/* MerkleTree::get + MerkleTree::prove for GLOBAL leaf indices (what the FRI query rounds open): the owning rank gathers row
 * and sibling path; rows n_idx * k, siblings n_idx * (log2 N - cap_height) * 4 (host; either may be NULL).  Collective. */
int b200zkp_sharded_rows(b200zkp_sharded* sh, const uint64_t* idx, uint64_t n_idx, uint64_t* rows, uint64_t* siblings);

#ifdef __cplusplus
}
#endif
#endif /* B200ZKP_H */
