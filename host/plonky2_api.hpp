// C++ host-side mirror of the plonky2 API surface of the commitment path, above the C ABI (include/b200zkp.h).
//
// The reference is compiled code (Rust) whose toolchain is absent in this image, so the host layer that a
// patched plonky2 would provide is written in C++ here with the same names, argument meaning and error
// behaviour as plonky2 @ f99ed9c (pinned by /root/reference/Cargo.toml:12):
//     PolynomialBatch::from_values / from_coeffs / get_lde_values        plonky2/src/fri/oracle.rs
//     MerkleTree::new / prove, MerkleCap, MerkleProof                    plonky2/src/hash/merkle_tree.rs
//     PoseidonHash::{hash_no_pad, hash_or_noop, two_to_one}              plonky2/src/hash/poseidon.rs
// plonky2's assert!/panic! become std::invalid_argument / std::runtime_error.  Header-only; link libb200zkp.so.
#pragma once
#include <array>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../include/b200zkp.h"

namespace plonky2 {

using F = uint64_t;  // GoldilocksField is #[repr(transparent)] over u64
constexpr uint64_t GOLDILOCKS_ORDER = 0xFFFFFFFF00000001ull;
constexpr size_t SALT_SIZE = B200ZKP_SALT_SIZE;

struct HashOut {
    std::array<F, 4> elements{};
    bool operator==(const HashOut& o) const { return elements == o.elements; }
    bool operator!=(const HashOut& o) const { return !(*this == o); }
};
using MerkleCap = std::vector<HashOut>;
struct MerkleProof { std::vector<HashOut> siblings; };

inline size_t log2_strict(uint64_t n) {
    if (n == 0 || (n & (n - 1))) throw std::invalid_argument("Not a power of two: " + std::to_string(n));
    size_t l = 0;
    while ((uint64_t(1) << l) < n) l++;
    return l;
}

class Context {
  public:
    explicit Context(int device = 0, void* cuda_stream = nullptr) {
        int rc = b200zkp_ctx_create(device, cuda_stream, &ctx_);
        if (rc != 0) throw std::runtime_error("b200zkp_ctx_create failed (no CUDA device? there is no CPU fallback)");
    }
    ~Context() { b200zkp_ctx_destroy(ctx_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    b200zkp_ctx* raw() const { return ctx_; }
    void check(int rc) const {
        if (rc == B200ZKP_ERR_BAD_ARG) throw std::invalid_argument(b200zkp_last_error(ctx_));
        if (rc != 0) throw std::runtime_error(b200zkp_last_error(ctx_));
    }
  private:
    b200zkp_ctx* ctx_ = nullptr;
};

struct PoseidonHash {
    static constexpr size_t HASH_SIZE = 32;
    static HashOut hash_no_pad(const Context& c, const std::vector<F>& in) {
        HashOut h;
        c.check(b200zkp_hash_no_pad(c.raw(), in.data(), 1, (uint32_t)in.size(), h.elements.data()));
        return h;
    }
    static HashOut hash_or_noop(const Context& c, const std::vector<F>& in) {
        HashOut h;
        c.check(b200zkp_hash_or_noop(c.raw(), in.data(), 1, (uint32_t)in.size(), h.elements.data()));
        return h;
    }
    static HashOut two_to_one(const Context& c, const HashOut& l, const HashOut& r) {
        HashOut h;
        c.check(b200zkp_two_to_one(c.raw(), l.elements.data(), r.elements.data(), 1, h.elements.data()));
        return h;
    }
};

// merkle_proofs.rs verify_merkle_proof_to_cap: throws std::runtime_error("Invalid Merkle proof.")
inline void verify_merkle_proof_to_cap(const Context& c, const std::vector<F>& leaf_data, uint64_t leaf_index,
                                       const MerkleCap& cap, const MerkleProof& proof) {
    HashOut cur = PoseidonHash::hash_or_noop(c, leaf_data);
    uint64_t index = leaf_index;
    for (const HashOut& sib : proof.siblings) {
        cur = (index & 1) ? PoseidonHash::two_to_one(c, sib, cur) : PoseidonHash::two_to_one(c, cur, sib);
        index >>= 1;
    }
    if (index >= cap.size() || cur != cap[index]) throw std::runtime_error("Invalid Merkle proof.");
}

class MerkleTree {
  public:
    // leaves: one Vec<F> per leaf, all of one length (plonky2 Vec<Vec<F>>)
    static MerkleTree new_(const Context& c, const std::vector<std::vector<F>>& leaves, size_t cap_height) {
        size_t n = leaves.size();
        size_t lg = log2_strict(n);
        if (cap_height > lg)
            throw std::invalid_argument("cap_height=" + std::to_string(cap_height) +
                                        " should be at most log2(leaves.len())=" + std::to_string(lg));
        size_t len = leaves[0].size();
        std::vector<F> flat(n * len);
        for (size_t i = 0; i < n; i++) {
            if (leaves[i].size() != len) throw std::invalid_argument("leaves must have equal length");
            std::copy(leaves[i].begin(), leaves[i].end(), flat.begin() + i * len);
        }
        MerkleTree t;
        t.ctx_ = &c;
        t.n_leaves_ = n;
        t.cap_height_ = cap_height;
        b200zkp_tree* h = nullptr;
        c.check(b200zkp_merkle_new(c.raw(), flat.data(), n, (uint32_t)len, (uint32_t)cap_height, &h));
        t.h_.reset(h, b200zkp_tree_free);
        t.cap.resize(size_t(1) << cap_height);
        c.check(b200zkp_tree_cap(h, t.cap[0].elements.data()));
        return t;
    }
    MerkleProof prove(uint64_t leaf_index) const {
        MerkleProof p;
        p.siblings.resize(log2_strict(n_leaves_) - cap_height_);
        ctx_->check(b200zkp_tree_prove(h_.get(), &leaf_index, 1, p.siblings.empty() ? nullptr : p.siblings[0].elements.data()));
        return p;
    }
    std::vector<HashOut> digests() const {
        std::vector<HashOut> d(2 * (n_leaves_ - (size_t(1) << cap_height_)));
        ctx_->check(b200zkp_tree_digests(h_.get(), d.empty() ? nullptr : d[0].elements.data()));
        return d;
    }
    MerkleCap cap;
  private:
    const Context* ctx_ = nullptr;
    std::shared_ptr<b200zkp_tree> h_;
    size_t n_leaves_ = 0, cap_height_ = 0;
};

class PolynomialBatch {
  public:
    // values / polynomials: k vectors of n elements (plonky2 Vec<PolynomialValues<F>> / Vec<PolynomialCoeffs<F>>).
    // salt: empty unless blinding; then SALT_SIZE vectors of N = n << rate_bits elements (plonky2 draws them from
    // the thread RNG; pass them explicitly for reproducible commitments).
    static PolynomialBatch from_values(const Context& c, const std::vector<std::vector<F>>& values, size_t rate_bits,
                                       bool blinding, size_t cap_height, const std::vector<std::vector<F>>& salt = {}) {
        return commit(c, values, false, rate_bits, blinding, cap_height, salt);
    }
    static PolynomialBatch from_coeffs(const Context& c, const std::vector<std::vector<F>>& polynomials, size_t rate_bits,
                                       bool blinding, size_t cap_height, const std::vector<std::vector<F>>& salt = {}) {
        return commit(c, polynomials, true, rate_bits, blinding, cap_height, salt);
    }
    // from_values / from_coeffs of a k x n column-major matrix already in device memory (b200zkp_batch_from_device); the
    // commit is enqueued on the ctx stream, `in_dev` must stay valid until it has run (the cap read below waits for it)
    static PolynomialBatch from_device(const Context& c, const uint64_t* in_dev, bool is_coeffs, size_t n_log, size_t k,
                                       size_t rate_bits, size_t cap_height) {
        PolynomialBatch b;
        b.ctx_ = &c;
        b.degree_log = n_log; b.rate_bits = rate_bits; b.cap_height = cap_height; b.num_polys = k;
        b200zkp_batch* h = nullptr;
        c.check(b200zkp_batch_from_device(c.raw(), in_dev, is_coeffs ? 1 : 0, (uint32_t)n_log, (uint32_t)k, (uint32_t)rate_bits,
                                          (uint32_t)cap_height, nullptr, &h));
        b.h_.reset(h, b200zkp_batch_free);
        b.cap.resize(size_t(1) << cap_height);
        c.check(b200zkp_batch_cap(h, b.cap[0].elements.data()));
        return b;
    }
    // &leaves[reverse_bits(index * step, degree_log + rate_bits)][..len - salt]
    std::vector<F> get_lde_values(uint64_t index, uint64_t step = 1) const {
        std::vector<F> out(num_polys);
        ctx_->check(b200zkp_batch_lde_values(h_.get(), index, step, out.data()));
        return out;
    }
    std::vector<std::vector<F>> polynomials() const {
        size_t n = size_t(1) << degree_log;
        std::vector<F> flat(num_polys * n);
        ctx_->check(b200zkp_batch_coeffs(h_.get(), flat.data()));
        std::vector<std::vector<F>> out(num_polys);
        for (size_t i = 0; i < num_polys; i++) out[i].assign(flat.begin() + i * n, flat.begin() + (i + 1) * n);
        return out;
    }
    // leaf row + Merkle proof (MerkleTree::get + MerkleTree::prove), what a FRI query round opens
    std::pair<std::vector<F>, MerkleProof> open(uint64_t leaf_index) const {
        std::vector<F> row(num_polys + salt_size);
        MerkleProof p;
        p.siblings.resize(degree_log + rate_bits - cap_height);
        ctx_->check(b200zkp_batch_rows(h_.get(), &leaf_index, 1, row.data(), p.siblings.empty() ? nullptr : p.siblings[0].elements.data()));
        return {row, p};
    }
    // OpeningSet::new's `p.to_extension().eval(zeta)` for every polynomial: zeta and results as (real, imaginary) pairs
    std::vector<std::array<F, 2>> eval_ext2(const std::array<F, 2>& zeta) const {
        std::vector<std::array<F, 2>> out(num_polys);
        ctx_->check(b200zkp_batch_eval_ext2(h_.get(), zeta.data(), out[0].data()));
        return out;
    }
    b200zkp_batch* raw() const { return h_.get(); }
    const Context& context() const { return *ctx_; }
    MerkleCap cap;  // merkle_tree.cap
    size_t degree_log = 0, rate_bits = 0, cap_height = 0, num_polys = 0, salt_size = 0;
    bool blinding = false;

  private:
    static PolynomialBatch commit(const Context& c, const std::vector<std::vector<F>>& cols, bool is_coeffs, size_t rate_bits,
                                  bool blinding, size_t cap_height, const std::vector<std::vector<F>>& salt) {
        if (cols.empty()) throw std::invalid_argument("empty polynomial batch");
        size_t n = cols[0].size(), k = cols.size();
        size_t n_log = log2_strict(n);
        std::vector<F> flat(k * n);
        for (size_t i = 0; i < k; i++) {
            if (cols[i].size() != n) throw std::invalid_argument("polynomials must have equal length");
            std::copy(cols[i].begin(), cols[i].end(), flat.begin() + i * n);
        }
        std::vector<F> s;
        if (blinding) {
            size_t N = n << rate_bits;
            if (salt.size() != SALT_SIZE) throw std::invalid_argument("blinding needs SALT_SIZE salt columns");
            s.resize(SALT_SIZE * N);
            for (size_t i = 0; i < SALT_SIZE; i++) {
                if (salt[i].size() != N) throw std::invalid_argument("salt columns must have N elements");
                std::copy(salt[i].begin(), salt[i].end(), s.begin() + i * N);
            }
        }
        PolynomialBatch b;
        b.ctx_ = &c;
        b.degree_log = n_log; b.rate_bits = rate_bits; b.cap_height = cap_height; b.num_polys = k;
        b.blinding = blinding; b.salt_size = blinding ? SALT_SIZE : 0;
        b200zkp_batch* h = nullptr;
        auto fn = is_coeffs ? b200zkp_commit_from_coeffs : b200zkp_commit_from_values;
        c.check(fn(c.raw(), flat.data(), (uint32_t)n_log, (uint32_t)k, (uint32_t)rate_bits, (uint32_t)cap_height,
                   blinding ? s.data() : nullptr, &h));
        b.h_.reset(h, b200zkp_batch_free);
        b.cap.resize(size_t(1) << cap_height);
        c.check(b200zkp_batch_cap(h, b.cap[0].elements.data()));
        return b;
    }
    const Context* ctx_ = nullptr;
    std::shared_ptr<b200zkp_batch> h_;
};

// The same commitment partitioned over every GPU of the box, driven by ONE process (b200zkp_comm_init_all): what a
// single-process rayon prove() (/root/reference/Cargo.toml:19-21) binds when more than one device is visible.  The cap
// equals PolynomialBatch::from_values' bit for bit; leaves live where they are hashed (rank g owns leaves
// [g*N/G, (g+1)*N/G)) and are opened through open(), which asks the owning rank.
class ShardedPolynomialBatch {
  public:
    // contexts: one per device, contexts[i] = rank i; their number must be a power of two <= 2^rate_bits, 2^cap_height
    static ShardedPolynomialBatch from_values(const std::vector<const Context*>& contexts, const std::vector<std::vector<F>>& values,
                                              size_t rate_bits, size_t cap_height) {
        if (values.empty() || contexts.empty()) throw std::invalid_argument("empty polynomial batch");
        size_t n = values[0].size(), k = values.size(), n_log = log2_strict(n);
        std::vector<F> flat(k * n);
        for (size_t i = 0; i < k; i++) {
            if (values[i].size() != n) throw std::invalid_argument("polynomials must have equal length");
            std::copy(values[i].begin(), values[i].end(), flat.begin() + i * n);
        }
        std::vector<b200zkp_ctx*> raw;
        for (auto* c : contexts) raw.push_back(c->raw());
        ShardedPolynomialBatch b;
        b200zkp_comm* comm = nullptr;
        contexts[0]->check(b200zkp_comm_init_all(raw.data(), (int)raw.size(), &comm));
        b.comm_.reset(comm, b200zkp_comm_destroy);
        b.degree_log = n_log; b.rate_bits = rate_bits; b.cap_height = cap_height; b.num_polys = k;
        b.cap.resize(size_t(1) << cap_height);
        b200zkp_sharded* sh = nullptr;
        b.check(b200zkp_sharded_commit_from_values(comm, flat.data(), (uint32_t)n_log, (uint32_t)k, (uint32_t)rate_bits,
                                                   (uint32_t)cap_height, b.cap[0].elements.data(), &sh));
        b.h_.reset(sh, b200zkp_sharded_free);
        return b;
    }
    // leaf row + Merkle proof for a GLOBAL leaf index (MerkleTree::get + MerkleTree::prove on the owning rank)
    std::pair<std::vector<F>, MerkleProof> open(uint64_t leaf_index) const {
        std::vector<F> row(num_polys);
        MerkleProof p;
        p.siblings.resize(degree_log + rate_bits - cap_height);
        check(b200zkp_sharded_rows(h_.get(), &leaf_index, 1, row.data(), p.siblings.empty() ? nullptr : p.siblings[0].elements.data()));
        return {row, p};
    }
    MerkleCap cap;
    size_t degree_log = 0, rate_bits = 0, cap_height = 0, num_polys = 0;

  private:
    void check(int rc) const {
        if (rc == B200ZKP_ERR_BAD_ARG) throw std::invalid_argument(b200zkp_comm_last_error(comm_.get()));
        if (rc != 0) throw std::runtime_error(b200zkp_comm_last_error(comm_.get()));
    }
    std::shared_ptr<b200zkp_comm> comm_;      // (declared before h_: the buffers are released first)
    std::shared_ptr<b200zkp_sharded> h_;
};

// OpeningSet::new in its FRI form (b200zkp_batch_openings): for each point, the values of its (oracle, index) polynomials
inline std::vector<std::vector<std::array<F, 2>>> batch_openings(
        const Context& c, const std::vector<const PolynomialBatch*>& oracles, const std::vector<std::array<F, 2>>& points,
        const std::vector<std::vector<std::pair<uint32_t, uint32_t>>>& polys) {
    if (points.size() != polys.size()) throw std::invalid_argument("one polynomial list per point");
    std::vector<b200zkp_batch*> handles;
    for (auto* o : oracles) handles.push_back(o->raw());
    std::vector<uint32_t> counts, po, pi;
    for (auto& ps : polys) {
        counts.push_back((uint32_t)ps.size());
        for (auto& p : ps) { po.push_back(p.first); pi.push_back(p.second); }
    }
    std::vector<std::array<F, 2>> flat(std::max<size_t>(po.size(), 1));
    c.check(b200zkp_batch_openings(c.raw(), handles.data(), (uint32_t)handles.size(), (uint32_t)points.size(), points[0].data(),
                                   counts.data(), po.data(), pi.data(), flat[0].data()));
    std::vector<std::vector<std::array<F, 2>>> out;
    size_t off = 0;
    for (auto& ps : polys) {
        out.emplace_back(flat.begin() + off, flat.begin() + off + ps.size());
        off += ps.size();
    }
    return out;
}

}  // namespace plonky2
