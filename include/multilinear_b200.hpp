// C++ host-side mirror of the reference's public interface for the PCS hot path (header-only, over the C ABI).
// The reference is Rust and cannot be built here; this header keeps its type and method names so that tests read like
// the reference's own (tests/cpp/reference_tests.cpp).  Reference panics become std::runtime_error (ml::Panic),
// Option::None becomes std::optional.  All array work happens in libmultilinear_b200.so on the GPU.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "multilinear_b200.h"

namespace ml {

struct Panic : std::runtime_error {
    int code;
    Panic(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
inline void check(int st) {
    if (st != ML_OK) throw Panic(st, ml_last_error());
}

// Field128 (src/field.rs:31): 16 little-endian bytes, canonical
struct alignas(16) Field128 {
    unsigned __int128 v;
    static Field128 from(long long x) {  // From<i64> (src/field.rs:150-154): sign-extend, one conditional subtract
        const unsigned __int128 M = ((((unsigned __int128)0xFFFFFFFFFFFFFFFFULL) << 64) | 0xFFFFD30000000001ULL);
        unsigned __int128 u = (unsigned __int128)(__int128)x;
        return Field128{u >= M ? u - M : u};
    }
    bool operator==(const Field128& o) const { return v == o.v; }
    bool operator!=(const Field128& o) const { return v != o.v; }
    const uint8_t* bytes() const { return reinterpret_cast<const uint8_t*>(&v); }
    uint8_t* bytes() { return reinterpret_cast<uint8_t*>(&v); }
};
static_assert(sizeof(Field128) == 16, "Field128 must be 16 bytes");
using F = Field128;
using HashDigest = std::array<uint8_t, 32>;
constexpr size_t LOG_BLOWUP = ML_LOG_BLOWUP;
constexpr size_t NUM_QUERIES = ML_NUM_QUERIES;

inline const uint8_t* raw(const std::vector<F>& v) { return reinterpret_cast<const uint8_t*>(v.data()); }
inline uint8_t* raw(std::vector<F>& v) { return reinterpret_cast<uint8_t*>(v.data()); }

// NttField (src/ntt/mod.rs:10-59)
inline std::optional<F> pow_2_generator(uint64_t log_size) {
    F g;
    int st = ml_pow2_generator(log_size, g.bytes());
    if (st == ML_ERR_OUT_OF_RANGE) return std::nullopt;
    check(st);
    return g;
}
inline std::optional<std::vector<F>> pow_2_generator_powers(uint64_t log_size) {
    if (log_size > 40) return std::nullopt;
    std::vector<F> out((size_t)1 << log_size);
    check(ml_pow2_generator_powers(log_size, raw(out)));
    return out;
}

struct Polynomial;
struct LagrangePolynomial {
    F gen;
    std::vector<F> evals;
    Polynomial intt() const;  // src/ntt/mod.rs:132-173
};
struct Polynomial {
    std::vector<F> coeffs;
    LagrangePolynomial ntt(F gen) const {  // src/ntt/mod.rs:69-110
        LagrangePolynomial out{gen, std::vector<F>(coeffs.size())};
        check(ml_ntt(raw(coeffs), coeffs.size(), gen.bytes(), raw(out.evals)));
        return out;
    }
    bool operator==(const Polynomial& o) const { return coeffs == o.coeffs; }
};
inline Polynomial LagrangePolynomial::intt() const {
    Polynomial out{std::vector<F>(evals.size())};
    check(ml_intt(raw(evals), evals.size(), gen.bytes(), raw(out.coeffs)));
    return out;
}
inline void bit_reverse_permutation(std::vector<F>& values) { check(ml_bit_reverse_permutation(raw(values), values.size(), 16)); }
inline std::vector<F> reed_solomon(std::vector<F> coeffs, F gen) {  // src/fri/mod.rs:19-28
    std::vector<F> code(coeffs.size() << LOG_BLOWUP);
    check(ml_reed_solomon(raw(coeffs), coeffs.size(), gen.bytes(), raw(code)));
    return code;
}

// src/polynomials.rs:100-188
struct MultilinearPolynomialEvals;
struct MultilinearPolynomial {
    std::vector<F> coeffs;
    MultilinearPolynomialEvals to_evaluation() const;
    F evaluate(const std::vector<F>& args) const {
        F out;
        check(ml_mle_coeffs_evaluate(raw(coeffs), coeffs.size(), raw(args), args.size(), out.bytes()));
        return out;
    }
};
struct MultilinearPolynomialEvals {
    std::vector<F> evals;
    MultilinearPolynomial to_coefficient() const {
        MultilinearPolynomial out{std::vector<F>(evals.size())};
        check(ml_mle_to_coefficient(raw(evals), evals.size(), raw(out.coeffs)));
        return out;
    }
    F evaluate(const std::vector<F>& args) const {
        F out;
        check(ml_mle_evals_evaluate(raw(evals), evals.size(), raw(args), args.size(), out.bytes()));
        return out;
    }
    bool operator==(const MultilinearPolynomialEvals& o) const { return evals == o.evals; }
};
inline MultilinearPolynomialEvals MultilinearPolynomial::to_evaluation() const {
    MultilinearPolynomialEvals out{std::vector<F>(coeffs.size())};
    check(ml_mle_to_evaluation(raw(coeffs), coeffs.size(), raw(out.evals)));
    return out;
}

// src/transcript.rs
class Transcript {
  public:
    Transcript() { check(ml_transcript_new(&h_)); }
    Transcript(const Transcript& o) { check(ml_transcript_clone(o.h_, &h_)); }
    Transcript& operator=(const Transcript&) = delete;
    ~Transcript() { ml_transcript_free(h_); }
    void absorb(const uint8_t* values, size_t len) { check(ml_transcript_absorb(h_, values, len)); }
    std::array<uint8_t, 32> random() const {
        std::array<uint8_t, 32> out;
        check(ml_transcript_random(h_, out.data()));
        return out;
    }
    F next_challenge() {
        F out;
        check(ml_transcript_next_challenge(h_, out.bytes()));
        return out;
    }
    ml_transcript* handle() { return h_; }

  private:
    ml_transcript* h_ = nullptr;
};

// src/merkle_tree/mod.rs — items are fixed-size byte strings
enum class Direction : uint8_t { Left = 0, Right = 1 };
struct MerkleInclusionPath {
    std::vector<uint8_t> value;
    std::vector<std::pair<HashDigest, Direction>> path;
    // verify / batch_verify (:216-293): 0 = Ok, else an ML_V_* code
    int verify(const HashDigest& root, size_t index) const {
        std::vector<uint8_t> digs(32 * path.size() + 1), dirs(path.size() + 1);
        for (size_t i = 0; i < path.size(); i++) {
            memcpy(&digs[32 * i], path[i].first.data(), 32);
            dirs[i] = (uint8_t)path[i].second;
        }
        return ml_merkle_path_verify(value.data(), value.size(), digs.data(), dirs.data(), path.size(), root.data(), index);
    }
};
class Merkle {
  public:
    static Merkle commit(const std::vector<std::vector<uint8_t>>& data) {  // :65-85
        const size_t item = data.empty() ? 0 : data[0].size();
        std::vector<uint8_t> flat;
        for (auto& d : data) flat.insert(flat.end(), d.begin(), d.end());
        Merkle m;
        m.value_bytes_ = item;
        check(ml_merkle_commit(flat.data(), item, data.size(), &m.h_));
        return m;
    }
    static Merkle batch_commit(const std::vector<std::vector<std::vector<uint8_t>>>& data) {  // :92-131
        if (data.empty()) throw Panic(ML_ERR_SIZE, "Data must not be empty");
        const size_t n = data[0].size(), item = n ? data[0][0].size() : 0;
        std::vector<std::vector<uint8_t>> flats(data.size());
        std::vector<const uint8_t*> ptrs;
        for (size_t b = 0; b < data.size(); b++) {
            if (data[b].size() != n) throw Panic(ML_ERR_SIZE, "All batches must have the same length");
            for (auto& d : data[b]) flats[b].insert(flats[b].end(), d.begin(), d.end());
            ptrs.push_back(flats[b].data());
        }
        Merkle m;
        m.value_bytes_ = item * data.size();
        check(ml_merkle_batch_commit(ptrs.data(), data.size(), item, n, &m.h_));
        return m;
    }
    Merkle(Merkle&& o) noexcept : h_(o.h_), value_bytes_(o.value_bytes_) { o.h_ = nullptr; }
    Merkle(const Merkle&) = delete;
    ~Merkle() { if (h_) ml_merkle_free(h_); }
    HashDigest root() const {
        HashDigest r;
        check(ml_merkle_root(h_, r.data()));
        return r;
    }
    std::optional<MerkleInclusionPath> open(size_t index) const {  // :31-58, :134-175
        MerkleInclusionPath p;
        p.value.resize(value_bytes_ ? value_bytes_ : 1);
        std::vector<uint8_t> digs(64 * 32), dirs(64);
        size_t len = 0;
        int st = ml_merkle_open(h_, index, p.value.data(), digs.data(), dirs.data(), &len);
        if (st == ML_ERR_OUT_OF_RANGE) return std::nullopt;
        check(st);
        p.value.resize(value_bytes_);
        for (size_t i = 0; i < len; i++) {
            HashDigest d;
            memcpy(d.data(), &digs[32 * i], 32);
            p.path.emplace_back(d, (Direction)dirs[i]);
        }
        return p;
    }
    std::optional<MerkleInclusionPath> batch_open(size_t index) const { return open(index); }

  private:
    Merkle() = default;
    ml_merkle* h_ = nullptr;
    size_t value_bytes_ = 0;
};

// src/fri/mod.rs:239-341
class FriProof {
  public:
    static FriProof prove(const std::vector<F>& code, const std::vector<F>& gen_pows, Transcript& t) {  // :261-285
        FriProof p;
        check(ml_fri_prove(raw(code), code.size(), raw(gen_pows), gen_pows.size(), t.handle(), &p.h_));
        return p;
    }
    FriProof(FriProof&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~FriProof() { if (h_) ml_fri_proof_free(h_); }
    int verify() const { return ml_fri_verify(h_); }  // :287-309; 0 = Ok(())
    std::vector<HashDigest> commitments() const {
        std::vector<HashDigest> out(ml_fri_proof_num_commitments(h_));
        if (!out.empty()) check(ml_fri_proof_commitments(h_, out[0].data()));
        return out;
    }
    std::vector<uint8_t> serialize() const {  // bincode, :367-391
        std::vector<uint8_t> out(ml_fri_proof_serialized_len(h_));
        check(ml_fri_proof_serialize(h_, out.data()));
        return out;
    }

  private:
    friend class ShardedFriProver;
    FriProof() = default;
    ml_fri_proof* h_ = nullptr;
};

// src/constraint_system/sumcheck.rs:10-15 — SumcheckTables of arbitrary trace width (System::build_tables :22-38).
// The composition the reference passes as a closure (:176) is a list of terms: comp(x) = sum_t coef_t * prod_k x[cols_t[k]].
struct CompositionTerm {
    F coef;
    std::vector<uint32_t> cols;
};
struct SumcheckPolynomial {
    std::vector<F> nonzero_coeffs;  // :17-19
};
class SumcheckTables {
  public:
    static SumcheckTables build(const std::vector<F>& row_point, const std::vector<F>& matrix, size_t width) {
        SumcheckTables t;
        check(ml_wsumcheck_build(raw(row_point), row_point.size(), raw(matrix), width, matrix.size() / width, &t.h_));
        return t;
    }
    SumcheckTables(SumcheckTables&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~SumcheckTables() { if (h_) ml_wsumcheck_free(h_); }
    void set_composition(const std::vector<CompositionTerm>& terms) {
        std::vector<F> coefs;
        std::vector<uint32_t> lens, cols;
        for (auto& t : terms) {
            coefs.push_back(t.coef);
            lens.push_back((uint32_t)t.cols.size());
            cols.insert(cols.end(), t.cols.begin(), t.cols.end());
        }
        if (cols.empty()) cols.push_back(0);
        check(ml_wsumcheck_set_composition(h_, terms.size(), raw(coefs), lens.data(), cols.data()));
    }
    size_t height() const { return ml_wsumcheck_height(h_); }
    F partial_sum(F r) {  // :204-232
        F out;
        check(ml_wsumcheck_partial_sum(h_, r.bytes(), out.bytes()));
        return out;
    }
    void fold(F r) { check(ml_wsumcheck_fold(h_, r.bytes())); }  // :234-247
    // :147-172 — returns (polynomials, randoms)
    std::pair<std::vector<SumcheckPolynomial>, std::vector<F>> compute_sumcheck_polynomials(size_t composition_degree, Transcript& t, F sum) {
        size_t rounds = 0;
        for (size_t h = height(); h > 1; h >>= 1) rounds++;
        const size_t td = composition_degree + 1;
        std::vector<F> coeffs(rounds * td + 1), randoms(rounds + 1);
        check(ml_wsumcheck_compute_polynomials(h_, composition_degree, t.handle(), sum.bytes(), raw(coeffs), raw(randoms)));
        std::vector<SumcheckPolynomial> pols(rounds);
        for (size_t k = 0; k < rounds; k++) pols[k].nonzero_coeffs.assign(coeffs.begin() + k * td, coeffs.begin() + (k + 1) * td);
        randoms.resize(rounds);
        return {std::move(pols), std::move(randoms)};
    }

  private:
    SumcheckTables() = default;
    ml_wsumcheck* h_ = nullptr;
};
// the width-w sumcheck over several GPUs from one process (ml_wsumcheck_shard_*, csrc/wsumcheck_shard.cu); `devices` may repeat
// (virtual ranks).  The result equals SumcheckTables::build + set_composition + compute_sumcheck_polynomials exactly.
class ShardedWideSumcheckTables {
  public:
    ShardedWideSumcheckTables(const std::vector<int>& devices, size_t width, size_t n_vars) : width_(width) {
        std::vector<int> ranks(devices.size());
        for (size_t i = 0; i < ranks.size(); i++) ranks[i] = (int)i;
        check(ml_wsumcheck_shard_create((int)devices.size(), (int)devices.size(), ranks.data(), devices.data(), width, n_vars, &h_));
    }
    ShardedWideSumcheckTables(const ShardedWideSumcheckTables&) = delete;
    ~ShardedWideSumcheckTables() { if (h_) ml_wsumcheck_shard_free(h_); }
    void set_composition(const std::vector<CompositionTerm>& terms) {
        std::vector<F> coefs;
        std::vector<uint32_t> lens, cols;
        for (auto& t : terms) {
            coefs.push_back(t.coef);
            lens.push_back((uint32_t)t.cols.size());
            cols.insert(cols.end(), t.cols.begin(), t.cols.end());
        }
        if (cols.empty()) cols.push_back(0);
        check(ml_wsumcheck_shard_set_composition(h_, terms.size(), raw(coefs), lens.data(), cols.data()));
    }
    // :147-172 of the trace `matrix` (row-major [2^n_vars][width]) at `row_point` — returns (polynomials, randoms)
    std::pair<std::vector<SumcheckPolynomial>, std::vector<F>> compute_sumcheck_polynomials(const std::vector<F>& row_point, const std::vector<F>& matrix,
                                                                                          size_t composition_degree, Transcript& t, F sum) {
        const size_t rounds = row_point.size(), td = composition_degree + 1;
        std::vector<F> coeffs(rounds * td + 1), randoms(rounds + 1);
        check(ml_wsumcheck_shard_compute_polynomials(h_, raw(row_point), rounds, raw(matrix), width_, matrix.size() / width_, composition_degree, t.handle(),
                                                     sum.bytes(), raw(coeffs), raw(randoms)));
        std::vector<SumcheckPolynomial> pols(rounds);
        for (size_t k = 0; k < rounds; k++) pols[k].nonzero_coeffs.assign(coeffs.begin() + k * td, coeffs.begin() + (k + 1) * td);
        randoms.resize(rounds);
        return {std::move(pols), std::move(randoms)};
    }

  private:
    ml_wsumcheck_shard* h_ = nullptr;
    size_t width_;
};

// src/fri/multilinear_pcs.rs:79-191
class PCSProof {
  public:
    static PCSProof prove(const std::vector<F>& inputs, F output, const MultilinearPolynomialEvals& poly, Transcript& t) {  // :90-136
        PCSProof p;
        check(ml_pcs_prove(raw(inputs), inputs.size(), output.bytes(), raw(poly.evals), poly.evals.size(), t.handle(), &p.h_));
        return p;
    }
    PCSProof(PCSProof&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~PCSProof() { if (h_) ml_pcs_proof_free(h_); }
    int verify(Transcript& t) const { return ml_pcs_verify(h_, t.handle()); }  // :138-190
    std::vector<std::array<F, 2>> sumcheck_polynomials() const {
        std::vector<std::array<F, 2>> out(ml_pcs_proof_num_rounds(h_));
        if (!out.empty()) check(ml_pcs_proof_sumcheck_coeffs(h_, reinterpret_cast<uint8_t*>(out.data())));
        return out;
    }

  private:
    friend class ShardedPCSProver;
    PCSProof() = default;
    ml_pcs_proof* h_ = nullptr;
};
// PCSProof::prove of one polynomial over several GPUs from one process (ml_pcs_shard_*, csrc/pcs_shard.cu); `devices` may repeat
// (virtual ranks).  The proof bytes equal PCSProof::prove's.
class ShardedPCSProver {
  public:
    ShardedPCSProver(const std::vector<int>& devices, size_t n_vars) {
        std::vector<int> ranks(devices.size());
        for (size_t i = 0; i < ranks.size(); i++) ranks[i] = (int)i;
        check(ml_pcs_shard_create((int)devices.size(), (int)devices.size(), ranks.data(), devices.data(), n_vars, &h_));
    }
    ShardedPCSProver(const ShardedPCSProver&) = delete;
    ~ShardedPCSProver() { if (h_) ml_pcs_shard_free(h_); }
    PCSProof prove(const std::vector<F>& inputs, F output, const MultilinearPolynomialEvals& poly, Transcript& t) {
        PCSProof p;
        check(ml_pcs_shard_prove(h_, raw(inputs), inputs.size(), output.bytes(), raw(poly.evals), poly.evals.size(), t.handle(), &p.h_));
        return p;
    }

  private:
    ml_pcs_shard* h_ = nullptr;
};
// FriProof::prove of one polynomial over several GPUs from one process (ml_fri_shard_*, csrc/fri_shard.cu), from its code or from
// its 2^log_n coefficients (reed_solomon + prove); `devices` may repeat (virtual ranks).  The proof bytes equal FriProof::prove's.
class ShardedFriProver {
  public:
    ShardedFriProver(const std::vector<int>& devices, size_t log_n) {
        std::vector<int> ranks(devices.size());
        for (size_t i = 0; i < ranks.size(); i++) ranks[i] = (int)i;
        check(ml_fri_shard_create((int)devices.size(), (int)devices.size(), ranks.data(), devices.data(), log_n, &h_));
    }
    ShardedFriProver(const ShardedFriProver&) = delete;
    ~ShardedFriProver() { if (h_) ml_fri_shard_free(h_); }
    FriProof prove(const std::vector<F>& code, const std::vector<F>& gen_pows, Transcript& t) {  // fri/mod.rs:261-285
        FriProof p;
        check(ml_fri_shard_prove(h_, raw(code), code.size(), raw(gen_pows), gen_pows.size(), t.handle(), &p.h_));
        return p;
    }
    FriProof rs_prove(const std::vector<F>& coeffs, Transcript& t) {  // reed_solomon (fri/mod.rs:19-28) + prove
        FriProof p;
        check(ml_fri_shard_rs_prove(h_, raw(coeffs), coeffs.size(), t.handle(), &p.h_));
        return p;
    }

  private:
    ml_fri_shard* h_ = nullptr;
};
// src/fri/batched_fri.rs:284-398
class BatchedFriProof {
  public:
    static BatchedFriProof prove(const std::vector<std::vector<F>>& codes, const std::vector<F>& gen_pows, Transcript& t) {  // :286-318
        std::vector<const uint8_t*> ptrs;
        for (auto& c : codes) ptrs.push_back(raw(c));
        BatchedFriProof p;
        check(ml_batched_fri_prove(ptrs.data(), codes.size(), codes.empty() ? 0 : codes[0].size(), raw(gen_pows), gen_pows.size(), t.handle(), &p.h_));
        return p;
    }
    BatchedFriProof(BatchedFriProof&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~BatchedFriProof() { if (h_) ml_bfri_proof_free(h_); }
    int verify() const { return ml_batched_fri_verify(h_); }  // :320-354; 0 = Ok(())
    std::vector<uint8_t> serialize() const {  // bincode
        std::vector<uint8_t> out(ml_bfri_proof_serialized_len(h_));
        check(ml_bfri_proof_serialize(h_, out.data()));
        return out;
    }

  private:
    friend class ShardedBatchedFriProver;
    BatchedFriProof() = default;
    ml_bfri_proof* h_ = nullptr;
};
// BatchedFriProof::prove of B codes over several GPUs from one process, every code split by block (ml_bfri_shard_*,
// csrc/bfri_shard.cu), from the codes or from the polynomials' 2^log_n coefficients (reed_solomon of each + prove); `devices` may
// repeat (virtual ranks).  The proof bytes equal BatchedFriProof::prove's.
class ShardedBatchedFriProver {
  public:
    ShardedBatchedFriProver(const std::vector<int>& devices, size_t n_codes, size_t log_n) {
        std::vector<int> ranks(devices.size());
        for (size_t i = 0; i < ranks.size(); i++) ranks[i] = (int)i;
        check(ml_bfri_shard_create((int)devices.size(), (int)devices.size(), ranks.data(), devices.data(), n_codes, log_n, &h_));
    }
    ShardedBatchedFriProver(const ShardedBatchedFriProver&) = delete;
    ~ShardedBatchedFriProver() { if (h_) ml_bfri_shard_free(h_); }
    BatchedFriProof prove(const std::vector<std::vector<F>>& codes, const std::vector<F>& gen_pows, Transcript& t) {  // batched_fri.rs:286-318
        std::vector<const uint8_t*> ptrs;
        for (auto& c : codes) ptrs.push_back(raw(c));
        BatchedFriProof p;
        check(ml_bfri_shard_prove(h_, ptrs.data(), codes.size(), codes.empty() ? 0 : codes[0].size(), raw(gen_pows), gen_pows.size(), t.handle(), &p.h_));
        return p;
    }
    BatchedFriProof rs_prove(const std::vector<std::vector<F>>& coeffs, Transcript& t) {  // reed_solomon of each + prove
        std::vector<const uint8_t*> ptrs;
        for (auto& c : coeffs) ptrs.push_back(raw(c));
        BatchedFriProof p;
        check(ml_bfri_shard_rs_prove(h_, ptrs.data(), coeffs.size(), coeffs.empty() ? 0 : coeffs[0].size(), t.handle(), &p.h_));
        return p;
    }

  private:
    ml_bfri_shard* h_ = nullptr;
};

// src/fri/batched_pcs.rs:22-254
struct BatchedPCSClaim {
    std::vector<F> inputs, outputs;
};
class BatchedPCSProof {
  public:
    static BatchedPCSProof prove(const BatchedPCSClaim& claim, const std::vector<MultilinearPolynomialEvals>& polys, Transcript& t) {  // :130-180
        std::vector<const uint8_t*> ptrs;
        for (auto& p : polys) ptrs.push_back(raw(p.evals));
        BatchedPCSProof p;
        check(ml_batched_pcs_prove(raw(claim.inputs), claim.inputs.size(), raw(claim.outputs), polys.size(), ptrs.data(),
                                   polys.empty() ? 0 : polys[0].evals.size(), t.handle(), &p.h_));
        return p;
    }
    BatchedPCSProof(BatchedPCSProof&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~BatchedPCSProof() { if (h_) ml_bpcs_proof_free(h_); }
    int verify(Transcript& t) const { return ml_batched_pcs_verify(h_, t.handle()); }  // :182-253
    std::vector<uint8_t> fri_proof_bytes() const {  // bincode layout of the BatchedFriProof (see ml_bfri_proof_serialize)
        const ml_bfri_proof* f = ml_bpcs_proof_fri(h_);
        std::vector<uint8_t> out(ml_bfri_proof_serialized_len(f));
        check(ml_bfri_proof_serialize(f, out.data()));
        return out;
    }

  private:
    friend class ShardedBatchedProver;
    friend class ShardedBatchedBlockProver;
    BatchedPCSProof() = default;
    ml_bpcs_proof* h_ = nullptr;
};
// BatchedPCSProof::prove over several GPUs from one process (ml_shard_*, csrc/shard.cu); `devices` may repeat (virtual ranks)
class ShardedBatchedProver {
  public:
    ShardedBatchedProver(const std::vector<int>& devices, size_t n_polys, size_t n_vars) {
        std::vector<int> ranks(devices.size());
        for (size_t i = 0; i < ranks.size(); i++) ranks[i] = (int)i;
        check(ml_shard_create((int)devices.size(), (int)devices.size(), ranks.data(), devices.data(), n_polys, n_vars, &h_));
    }
    ShardedBatchedProver(const ShardedBatchedProver&) = delete;
    ~ShardedBatchedProver() { if (h_) ml_shard_free(h_); }
    BatchedPCSProof prove(const BatchedPCSClaim& claim, const std::vector<MultilinearPolynomialEvals>& polys, Transcript& t) {
        std::vector<const uint8_t*> ptrs;
        for (auto& p : polys) ptrs.push_back(raw(p.evals));
        BatchedPCSProof p;
        check(ml_shard_batched_pcs_prove(h_, raw(claim.inputs), claim.inputs.size(), raw(claim.outputs), polys.size(), ptrs.data(), t.handle(), &p.h_));
        return p;
    }

  private:
    ml_shard* h_ = nullptr;
};
// BatchedPCSProof::prove over several GPUs from one process with every polynomial split by block (ml_bpcs_shard_*,
// csrc/bpcs_shard.cu): any n_polys >= 1 on any power-of-two number of ranks; `devices` may repeat (virtual ranks)
class ShardedBatchedBlockProver {
  public:
    ShardedBatchedBlockProver(const std::vector<int>& devices, size_t n_polys, size_t n_vars) {
        std::vector<int> ranks(devices.size());
        for (size_t i = 0; i < ranks.size(); i++) ranks[i] = (int)i;
        check(ml_bpcs_shard_create((int)devices.size(), (int)devices.size(), ranks.data(), devices.data(), n_polys, n_vars, &h_));
    }
    ShardedBatchedBlockProver(const ShardedBatchedBlockProver&) = delete;
    ~ShardedBatchedBlockProver() { if (h_) ml_bpcs_shard_free(h_); }
    BatchedPCSProof prove(const BatchedPCSClaim& claim, const std::vector<MultilinearPolynomialEvals>& polys, Transcript& t) {
        std::vector<const uint8_t*> ptrs;
        for (auto& p : polys) ptrs.push_back(raw(p.evals));
        BatchedPCSProof p;
        check(ml_bpcs_shard_prove(h_, raw(claim.inputs), claim.inputs.size(), raw(claim.outputs), polys.size(), ptrs.data(),
                                  polys.empty() ? 0 : polys[0].evals.size(), t.handle(), &p.h_));
        return p;
    }

  private:
    ml_bpcs_shard* h_ = nullptr;
};

// src/polynomials.rs:3-98 — univariate helpers over the domain 0..n-1 (named Univariate* here: `Polynomial` above is src/ntt's)
struct UnivariatePolynomialEvals;
struct UnivariatePolynomial {
    std::vector<F> coeffs;
    UnivariatePolynomialEvals evaluate_over_domain() const;  // :16-28
};
struct UnivariatePolynomialEvals {
    std::vector<F> evals;
    bool operator==(const UnivariatePolynomialEvals& o) const { return evals == o.evals; }
    UnivariatePolynomial interpolate() const {  // :51-86
        UnivariatePolynomial p{std::vector<F>(evals.size())};
        check(ml_poly_interpolate(raw(evals), evals.size(), raw(p.coeffs)));
        return p;
    }
};
inline UnivariatePolynomialEvals UnivariatePolynomial::evaluate_over_domain() const {
    UnivariatePolynomialEvals e{std::vector<F>(coeffs.size())};
    check(ml_poly_evaluate_over_domain(raw(coeffs), coeffs.size(), raw(e.evals)));
    return e;
}

}  // namespace ml
