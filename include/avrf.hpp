// avrf.hpp - C++ mirror of the reference's Rust interface for the Thin-VRF verification path,
// above the C ABI of avrf.h.  Same names and meaning as `ark_vrf::thin` (reference src/thin.rs):
//
//   thin::Proof<S>{r, s}                          src/thin.rs:42-48
//   thin::BatchItem<S>                            src/thin.rs:172-179
//   thin::BatchVerifier<S>::{new_, prepare, push_prepared, push, verify}   src/thin.rs:198-326
//   Public<S>::verify  (thin::Verifier)           src/thin.rs:95-109,131-165
//   thin::BatchServer<S>::{submit, submit_compressed, wait}   (new: worker pool over avrf_server_*, throughput mode)
//   thin::ShardedBatchVerifier<S>                 (new: one batch over several GPUs of this process, avrf_thin_sharded_*)
//   pedersen::Proof{pk_com, r, ok, s, sb}         src/pedersen.rs:43-50
//   pedersen::verify (pedersen::Verifier)         src/pedersen.rs:188-253
//   pedersen::BatchVerifier<S>::{reserve, push, push_compressed, verify, verify_each, find_invalid}   src/pedersen.rs:322-427
//   pedersen::prove_many (Prover::prove, n proofs) src/pedersen.rs:136-186
//   pedersen::BatchServer<S>::{submit, submit_compressed, wait}   (new: the same worker pool for Pedersen batches)
//   pedersen::ShardedBatchVerifier<S>             (new: one Pedersen batch over several GPUs of this process)
//   Error::{VerificationFailure, InvalidData}     src/lib.rs:136-147
//
// The host toolchain of the reference (Rust) is absent from the build image, so this header is the
// compiled-language mirror; ark_vrf_b200/rust/gpu.rs is the binding a maintainer adds upstream.
#pragma once
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "avrf.h"

namespace ark_vrf {

enum class Error { VerificationFailure = 1, InvalidData = 2 };

struct Result {                      // Result<(), Error>
  int status;                        // AVRF_OK / AVRF_VERIFICATION_FAILURE / AVRF_INVALID_DATA
  bool is_ok() const { return status == AVRF_OK; }
  bool is_err() const { return status != AVRF_OK; }
  Error unwrap_err() const { return static_cast<Error>(status); }
};

using AffinePoint = std::array<uint8_t, 64>;   // x || y, format chosen by the suite tag below
using ScalarField = std::array<uint8_t, 32>;
struct VrfIo { AffinePoint input, output; };    // src/lib.rs:615-619
static_assert(sizeof(VrfIo) == 128, "VrfIo must be 128 contiguous bytes");

struct BandersnatchSha512Ell2 { static constexpr uint32_t ID = AVRF_SUITE_BANDERSNATCH_SHA512_ELL2; };
struct Ed25519Sha512Tai { static constexpr uint32_t ID = AVRF_SUITE_ED25519_SHA512_TAI; };
struct BabyJubJubSha512Tai { static constexpr uint32_t ID = AVRF_SUITE_BABYJUBJUB_SHA512_TAI; };

inline void check(int rc) {
  if (rc != 0) throw std::runtime_error(std::string("libavrf_gpu: ") + avrf_last_error());
}

namespace thin {

struct Proof { AffinePoint r; ScalarField s; };

struct BatchItem {                   // un-hashed: transcripts run on the GPU at verify
  AffinePoint pk; std::vector<VrfIo> ios; std::vector<uint8_t> ad; Proof proof;
};

template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
class BatchVerifier {
 public:
  BatchVerifier() : h_(avrf_thin_batch_new(S::ID, FMT)) { if (!h_) throw std::runtime_error(avrf_last_error()); }
  ~BatchVerifier() { avrf_thin_batch_free(h_); }
  BatchVerifier(const BatchVerifier&) = delete;
  BatchVerifier& operator=(const BatchVerifier&) = delete;
  static BatchVerifier new_() { return BatchVerifier(); }
  // like Vec::with_capacity: device memory for n proofs up front, so that a loop of push() never reallocates
  void reserve(uint64_t n, uint64_t n_ios, uint64_t ad_bytes) { check(avrf_thin_batch_reserve(h_, n, n_ios, ad_bytes)); }
  int64_t len() const { return avrf_thin_batch_len(h_); }
  void clear() { check(avrf_thin_batch_clear(h_)); }

  static BatchItem prepare(const AffinePoint& pk, const std::vector<VrfIo>& ios, const std::vector<uint8_t>& ad,
                           const Proof& proof) { return BatchItem{pk, ios, ad, proof}; }
  void push_prepared(const BatchItem& e) { push(e.pk, e.ios, e.ad, e.proof); }
  void push(const AffinePoint& pk, const std::vector<VrfIo>& ios, const std::vector<uint8_t>& ad, const Proof& proof) {
    check(avrf_thin_batch_push(h_, pk.data(), ios.empty() ? nullptr : ios[0].input.data(), (uint32_t)ios.size(),
                               ad.empty() ? nullptr : ad.data(), (uint32_t)ad.size(), proof.r.data(), proof.s.data()));
  }
  // Proofs still in wire format (what Proof::deserialize_compressed and the Public / Input / Output deserialisers
  // take): decoded and validated on the device.  Returns the number of proofs that do not decode; when it is not
  // zero nothing was pushed and ok[j] == 0 names them.
  uint64_t push_compressed(uint64_t n, const uint8_t* pk32, const uint8_t* ios32, const uint32_t* io_offsets,
                           const uint8_t* ad_blob, const uint32_t* ad_offsets, const uint8_t* r32, const uint8_t* s,
                           std::vector<uint8_t>* ok = nullptr) {
    uint64_t bad = 0;
    if (ok) ok->assign(n, 0);
    check(avrf_thin_batch_push_compressed(h_, n, pk32, ios32, io_offsets, ad_blob, ad_offsets, r32, s,
                                          ok && n ? ok->data() : nullptr, &bad));
    return bad;
  }
  Result verify() const {
    int32_t st = -1;
    check(avrf_thin_batch_verify(h_, &st));
    return Result{st};
  }
  avrf_batch* handle() const { return h_; }

 private:
  avrf_batch* h_;
};

// One batch over every GPU initialised with init_multi(), inside this process (include/avrf.h, "Multi-GPU batches").
inline int init_multi(int n_dev = 0) {
  check(avrf_init_multi(n_dev, nullptr));
  return avrf_device_count();
}

struct Batch;

template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
class ShardedBatchVerifier {
 public:
  ShardedBatchVerifier() : h_(avrf_thin_sharded_new(S::ID, FMT)) { if (!h_) throw std::runtime_error(avrf_last_error()); }
  ~ShardedBatchVerifier() { avrf_thin_sharded_free(h_); }
  ShardedBatchVerifier(const ShardedBatchVerifier&) = delete;
  ShardedBatchVerifier& operator=(const ShardedBatchVerifier&) = delete;
  inline void push_many(const Batch& b);
  Result verify() const {
    int32_t st = -1;
    check(avrf_thin_sharded_verify(h_, &st));
    return Result{st};
  }
  void clear() { check(avrf_thin_sharded_clear(h_)); }
  int devices() const { return avrf_thin_sharded_devices(h_); }
  int64_t len() const { return avrf_thin_sharded_len(h_); }
  avrf_sharded* handle() const { return h_; }

 private:
  avrf_sharded* h_;
};

// Throughput mode (no counterpart in the reference, whose verifier is a plain value that callers spread
// over threads themselves): a native pool of worker threads, one BatchVerifier handle each.  A `Batch` is the
// flattened argument list of a whole verification; it is borrowed until `wait` returns for its ticket.
struct Batch {
  std::vector<AffinePoint> pk, r;
  std::vector<ScalarField> s;
  std::vector<VrfIo> ios;
  std::vector<uint32_t> io_offsets{0}, ad_offsets{0};
  std::vector<uint8_t> ad;
  void push(const AffinePoint& pk_, const std::vector<VrfIo>& ios_, const std::vector<uint8_t>& ad_, const Proof& proof) {
    pk.push_back(pk_); r.push_back(proof.r); s.push_back(proof.s);
    ios.insert(ios.end(), ios_.begin(), ios_.end());
    ad.insert(ad.end(), ad_.begin(), ad_.end());
    io_offsets.push_back((uint32_t)ios.size());
    ad_offsets.push_back((uint32_t)ad.size());
  }
  size_t len() const { return pk.size(); }
};

template <class S, uint32_t FMT>
inline void ShardedBatchVerifier<S, FMT>::push_many(const Batch& b) {
  check(avrf_thin_sharded_push_many(h_, b.len(), b.len() ? b.pk[0].data() : nullptr,
                                    b.ios.empty() ? nullptr : b.ios[0].input.data(), b.io_offsets.data(),
                                    b.ad.empty() ? nullptr : b.ad.data(), b.ad_offsets.data(),
                                    b.len() ? b.r[0].data() : nullptr, b.len() ? b.s[0].data() : nullptr));
}

template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
class BatchServer {
 public:
  // hashers > 0: shared multi-buffer SHA-512 threads (eight batches' hash chains each) instead of a core per worker
  explicit BatchServer(uint32_t workers, uint32_t hashers = 0) : h_(avrf_server_new_ex(S::ID, FMT, workers, hashers)) {
    if (!h_) throw std::runtime_error(avrf_last_error());
  }
  ~BatchServer() { avrf_server_free(h_); }
  BatchServer(const BatchServer&) = delete;
  BatchServer& operator=(const BatchServer&) = delete;
  int64_t submit(const Batch& b) {
    int64_t t = avrf_server_submit(h_, b.len(), b.len() ? b.pk[0].data() : nullptr,
                                   b.ios.empty() ? nullptr : b.ios[0].input.data(), b.io_offsets.data(),
                                   b.ad.empty() ? nullptr : b.ad.data(), b.ad_offsets.data(),
                                   b.len() ? b.r[0].data() : nullptr, b.len() ? b.s[0].data() : nullptr);
    if (t < 0) check((int)t);
    return t;
  }
  // A batch of proofs in wire format, arguments as BatchVerifier::push_compressed.  The arrays, `ok` (n bytes) and
  // `n_bad` (both optional) are borrowed until wait() returns for the ticket; a proof that does not decode makes the
  // verdict InvalidData with *n_bad > 0 and ok[j] == 0 naming it.
  int64_t submit_compressed(uint64_t n, const uint8_t* pk32, const uint8_t* ios32, const uint32_t* io_offsets,
                            const uint8_t* ad_blob, const uint32_t* ad_offsets, const uint8_t* r32, const uint8_t* s,
                            uint8_t* ok = nullptr, uint64_t* n_bad = nullptr) {
    int64_t t = avrf_server_submit_compressed(h_, n, pk32, ios32, io_offsets, ad_blob, ad_offsets, r32, s, ok, n_bad);
    if (t < 0) check((int)t);
    return t;
  }
  Result wait(int64_t ticket) {
    int32_t st = -1;
    check(avrf_server_wait(h_, ticket, &st));
    return Result{st};
  }

 private:
  avrf_server* h_;
};

}  // namespace thin

namespace pedersen {

struct Proof { AffinePoint pk_com, r, ok; ScalarField s, sb; };   // src/pedersen.rs:43-50
static_assert(sizeof(Proof) == 256, "pedersen::Proof must be five contiguous fields");

// pedersen::Verifier::verify (src/pedersen.rs:188-253) for one proof: exact, both equations (avrf_pedersen_verify_one).
template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
Result verify(const std::vector<VrfIo>& ios, const std::vector<uint8_t>& ad, const Proof& proof) {
  int32_t st = -1;
  check(avrf_pedersen_verify_one(S::ID, FMT, ios.empty() ? nullptr : ios[0].input.data(), (uint32_t)ios.size(),
                                 ad.empty() ? nullptr : ad.data(), (uint32_t)ad.size(), proof.pk_com.data(), proof.r.data(),
                                 proof.ok.data(), proof.s.data(), proof.sb.data(), &st));
  return Result{st};
}

// pedersen::BatchVerifier (src/pedersen.rs:322-427), plus per-proof verdicts after a failed batch.
template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
class BatchVerifier {
 public:
  BatchVerifier() : h_(avrf_pedersen_batch_new(S::ID, FMT)) { if (!h_) throw std::runtime_error(avrf_last_error()); }
  ~BatchVerifier() { avrf_thin_batch_free(h_); }
  BatchVerifier(const BatchVerifier&) = delete;
  BatchVerifier& operator=(const BatchVerifier&) = delete;
  // like Vec::with_capacity: device memory for n proofs up front, so that a loop of push() never reallocates
  void reserve(uint64_t n, uint64_t n_ios, uint64_t ad_bytes) { check(avrf_thin_batch_reserve(h_, n, n_ios, ad_bytes)); }
  int64_t len() const { return avrf_thin_batch_len(h_); }
  void clear() { check(avrf_thin_batch_clear(h_)); }
  // one proof, staged in pinned memory and shipped to the device in chunks (avrf_pedersen_batch_push)
  void push(const std::vector<VrfIo>& ios, const std::vector<uint8_t>& ad, const Proof& proof) {
    check(avrf_pedersen_batch_push(h_, ios.empty() ? nullptr : ios[0].input.data(), (uint32_t)ios.size(),
                                   ad.empty() ? nullptr : ad.data(), (uint32_t)ad.size(), proof.pk_com.data(),
                                   proof.r.data(), proof.ok.data(), proof.s.data(), proof.sb.data()));
  }
  // Proofs in wire format: n records of Proof::serialize_compressed (pk_com | r | ok | s | sb, 160 bytes) and 64 bytes
  // of compressed (input, output) per pair, decoded and validated on the device.  Returns the number of proofs that
  // do not decode; when it is not zero nothing was pushed and ok[j] == 0 names them.
  uint64_t push_compressed(uint64_t n, const uint8_t* ios32, const uint32_t* io_offsets, const uint8_t* ad_blob,
                           const uint32_t* ad_offsets, const uint8_t* proofs, std::vector<uint8_t>* ok = nullptr) {
    uint64_t bad = 0;
    if (ok) ok->assign(n, 0);
    check(avrf_pedersen_batch_push_compressed(h_, n, ios32, io_offsets, ad_blob, ad_offsets, proofs,
                                              ok && n ? ok->data() : nullptr, &bad));
    return bad;
  }
  Result verify() const {
    int32_t st = -1;
    check(avrf_pedersen_batch_verify(h_, &st));
    return Result{st};
  }
  // statuses[j] = pedersen::Verifier::verify of proof j (AVRF_OK / AVRF_VERIFICATION_FAILURE / AVRF_INVALID_DATA)
  std::vector<int32_t> verify_each() const {
    std::vector<int32_t> st((size_t)len(), -1);
    check(avrf_pedersen_batch_verify_each(h_, st.empty() ? nullptr : st.data()));
    return st;
  }
  std::vector<size_t> find_invalid() const {
    std::vector<size_t> bad;
    std::vector<int32_t> st = verify_each();
    for (size_t j = 0; j < st.size(); j++)
      if (st[j] != AVRF_OK) bad.push_back(j);
    return bad;
  }
  avrf_batch* handle() const { return h_; }

 private:
  avrf_batch* h_;
};

// The flattened argument list of a whole Pedersen verification, for BatchServer::submit (borrowed until wait).
struct Batch {
  std::vector<AffinePoint> pk_com, r, ok;
  std::vector<ScalarField> s, sb;
  std::vector<VrfIo> ios;
  std::vector<uint32_t> io_offsets{0}, ad_offsets{0};
  std::vector<uint8_t> ad;
  void push(const std::vector<VrfIo>& ios_, const std::vector<uint8_t>& ad_, const Proof& proof) {
    pk_com.push_back(proof.pk_com); r.push_back(proof.r); ok.push_back(proof.ok);
    s.push_back(proof.s); sb.push_back(proof.sb);
    ios.insert(ios.end(), ios_.begin(), ios_.end());
    ad.insert(ad.end(), ad_.begin(), ad_.end());
    io_offsets.push_back((uint32_t)ios.size());
    ad_offsets.push_back((uint32_t)ad.size());
  }
  size_t len() const { return pk_com.size(); }
};

using thin::init_multi;

// One Pedersen batch over every GPU initialised with init_multi(), inside this process (include/avrf.h, "Multi-GPU
// batches": avrf_pedersen_sharded_new / _push_many and the avrf_thin_sharded_* calls that serve both schemes).
template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
class ShardedBatchVerifier {
 public:
  ShardedBatchVerifier() : h_(avrf_pedersen_sharded_new(S::ID, FMT)) { if (!h_) throw std::runtime_error(avrf_last_error()); }
  ~ShardedBatchVerifier() { avrf_thin_sharded_free(h_); }
  ShardedBatchVerifier(const ShardedBatchVerifier&) = delete;
  ShardedBatchVerifier& operator=(const ShardedBatchVerifier&) = delete;
  void push_many(const Batch& b) {
    const bool any = b.len() != 0;
    check(avrf_pedersen_sharded_push_many(h_, b.len(), b.ios.empty() ? nullptr : b.ios[0].input.data(), b.io_offsets.data(),
                                          b.ad.empty() ? nullptr : b.ad.data(), b.ad_offsets.data(),
                                          any ? b.pk_com[0].data() : nullptr, any ? b.r[0].data() : nullptr,
                                          any ? b.ok[0].data() : nullptr, any ? b.s[0].data() : nullptr,
                                          any ? b.sb[0].data() : nullptr));
  }
  Result verify() const {
    int32_t st = -1;
    check(avrf_thin_sharded_verify(h_, &st));
    return Result{st};
  }
  void clear() { check(avrf_thin_sharded_clear(h_)); }
  int devices() const { return avrf_thin_sharded_devices(h_); }
  int64_t len() const { return avrf_thin_sharded_len(h_); }
  avrf_sharded* handle() const { return h_; }

 private:
  avrf_sharded* h_;
};

// Throughput mode for Pedersen batches: the worker pool of thin::BatchServer, one pedersen::BatchVerifier handle per
// worker (avrf_pedersen_server_new).
template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
class BatchServer {
 public:
  // hashers > 0: shared multi-buffer SHA-512 threads; own_hash_workers of the workers keep a core each (mixed pool)
  explicit BatchServer(uint32_t workers, uint32_t hashers = 0, uint32_t own_hash_workers = 0)
      : h_(avrf_pedersen_server_new(S::ID, FMT, workers, hashers, own_hash_workers)) {
    if (!h_) throw std::runtime_error(avrf_last_error());
  }
  ~BatchServer() { avrf_server_free(h_); }
  BatchServer(const BatchServer&) = delete;
  BatchServer& operator=(const BatchServer&) = delete;
  int64_t submit(const Batch& b) {
    const bool any = b.len() != 0;
    int64_t t = avrf_pedersen_server_submit(h_, b.len(), b.ios.empty() ? nullptr : b.ios[0].input.data(), b.io_offsets.data(),
                                            b.ad.empty() ? nullptr : b.ad.data(), b.ad_offsets.data(),
                                            any ? b.pk_com[0].data() : nullptr, any ? b.r[0].data() : nullptr,
                                            any ? b.ok[0].data() : nullptr, any ? b.s[0].data() : nullptr,
                                            any ? b.sb[0].data() : nullptr);
    if (t < 0) check((int)t);
    return t;
  }
  // A batch in wire format, arguments as BatchVerifier::push_compressed; `ok` / `n_bad` as thin::BatchServer's.
  int64_t submit_compressed(uint64_t n, const uint8_t* ios32, const uint32_t* io_offsets, const uint8_t* ad_blob,
                            const uint32_t* ad_offsets, const uint8_t* proofs, uint8_t* ok = nullptr,
                            uint64_t* n_bad = nullptr) {
    int64_t t = avrf_pedersen_server_submit_compressed(h_, n, ios32, io_offsets, ad_blob, ad_offsets, proofs, ok, n_bad);
    if (t < 0) check((int)t);
    return t;
  }
  Result wait(int64_t ticket) {
    int32_t st = -1;
    check(avrf_server_wait(h_, ticket, &st));
    return Result{st};
  }

 private:
  avrf_server* h_;
};

struct Proven { std::vector<Proof> proofs; std::vector<ScalarField> blinding; };

// pedersen::Prover::prove (src/pedersen.rs:136-186) for n = sk.size() proofs (avrf_pedersen_prove_many): proof j signs
// pairs ios[io_offsets[j] ..] and ad[ad_offsets[j] ..] with sk[j]; pk[j] = sk[j] * G.
template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
Proven prove_many(const std::vector<ScalarField>& sk, const std::vector<AffinePoint>& pk, const std::vector<VrfIo>& ios,
                  const std::vector<uint32_t>& io_offsets, const std::vector<uint8_t>& ad,
                  const std::vector<uint32_t>& ad_offsets) {
  const size_t n = sk.size();
  if (pk.size() != n || io_offsets.size() != n + 1 || ad_offsets.size() != n + 1)
    throw std::invalid_argument("prove_many: sk, pk and the offsets must describe the same proofs");
  std::vector<AffinePoint> pkc(n), r(n), ok(n);
  std::vector<ScalarField> s(n), sb(n);
  Proven out;
  out.blinding.resize(n);
  check(avrf_pedersen_prove_many(S::ID, FMT, n, n ? sk[0].data() : nullptr, n ? pk[0].data() : nullptr,
                                 ios.empty() ? nullptr : ios[0].input.data(), io_offsets.data(),
                                 ad.empty() ? nullptr : ad.data(), ad_offsets.data(), n ? pkc[0].data() : nullptr,
                                 n ? r[0].data() : nullptr, n ? ok[0].data() : nullptr, n ? s[0].data() : nullptr,
                                 n ? sb[0].data() : nullptr, n ? out.blinding[0].data() : nullptr));
  out.proofs.resize(n);
  for (size_t j = 0; j < n; j++) out.proofs[j] = Proof{pkc[j], r[j], ok[j], s[j], sb[j]};
  return out;
}

}  // namespace pedersen

template <class S, uint32_t FMT = AVRF_FMT_MONTGOMERY>
struct Public {                      // Public<S> with thin::Verifier::verify
  AffinePoint point;
  Result verify(const std::vector<VrfIo>& ios, const std::vector<uint8_t>& ad, const thin::Proof& proof) const {
    int32_t st = -1;
    check(avrf_thin_verify_one(S::ID, FMT, point.data(), ios.empty() ? nullptr : ios[0].input.data(), (uint32_t)ios.size(),
                               ad.empty() ? nullptr : ad.data(), (uint32_t)ad.size(), proof.r.data(), proof.s.data(), &st));
    return Result{st};
  }
};

}  // namespace ark_vrf
