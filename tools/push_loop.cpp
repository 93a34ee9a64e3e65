// Drop-in path benchmark: the reference's own bench shape (benches/thin.rs:76-88) through the C++ mirror of its
// API (include/avrf.hpp) - `BatchVerifier::push` once per proof from ordinary heap memory, then `verify`.
// Built by __graft_entry__.build() into tools/libavrf_pushloop.so and called from bench.py (`drop_in` block, Thin)
// and tools/bench_pedersen.py (`drop_in` leg, Pedersen); the items are materialised as ordinary C++ values first
// (untimed, as the reference bench builds its proofs before the measured loop).
#include <chrono>
#include <cstring>
#include <memory>
#include <vector>

#include "avrf.hpp"

using namespace ark_vrf;

struct Item { AffinePoint pk; std::vector<VrfIo> ios; std::vector<uint8_t> ad; thin::Proof proof; };

struct PushLoop {
  std::vector<Item> items;
  std::unique_ptr<thin::BatchVerifier<BandersnatchSha512Ell2, AVRF_FMT_MONTGOMERY>> bv;
};

extern "C" {

// Arrays as for avrf_thin_batch_push_many (Bandersnatch, Montgomery format).
void* avrf_pushloop_new(uint64_t n, const uint8_t* pk, const uint8_t* ios, const uint32_t* io_off, const uint8_t* ad,
                        const uint32_t* ad_off, const uint8_t* r, const uint8_t* s) {
  try {
    auto* pl = new PushLoop();
    pl->items.resize(n);
    for (uint64_t j = 0; j < n; j++) {
      Item& it = pl->items[j];
      memcpy(it.pk.data(), pk + 64 * j, 64);
      it.ios.resize(io_off[j + 1] - io_off[j]);
      if (!it.ios.empty()) memcpy(it.ios.data(), ios + 128 * (size_t)io_off[j], 128 * it.ios.size());
      it.ad.assign(ad + ad_off[j], ad + ad_off[j + 1]);
      memcpy(it.proof.r.data(), r + 64 * j, 64);
      memcpy(it.proof.s.data(), s + 32 * j, 32);
    }
    pl->bv.reset(new thin::BatchVerifier<BandersnatchSha512Ell2, AVRF_FMT_MONTGOMERY>());
    return pl;
  } catch (...) {
    return nullptr;
  }
}

void* avrf_pushloop_stream(void* h) { return avrf_thin_batch_stream(static_cast<PushLoop*>(h)->bv->handle()); }

// One step: a fresh batch, push every item, verify.  Returns the verdict (or a negative error code);
// *push_ms / *verify_ms: host wall time of the two halves.
int avrf_pushloop_step(void* h, int reserve, double* push_ms, double* verify_ms) {
  PushLoop* pl = static_cast<PushLoop*>(h);
  try {
    auto t0 = std::chrono::steady_clock::now();
    pl->bv->clear();
    if (reserve) {
      uint64_t nio = 0, nad = 0;
      for (const Item& it : pl->items) { nio += it.ios.size(); nad += it.ad.size(); }
      pl->bv->reserve(pl->items.size(), nio, nad);
    }
    for (const Item& it : pl->items) pl->bv->push(it.pk, it.ios, it.ad, it.proof);
    auto t1 = std::chrono::steady_clock::now();
    Result res = pl->bv->verify();
    auto t2 = std::chrono::steady_clock::now();
    if (push_ms) *push_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    if (verify_ms) *verify_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
    return res.status;
  } catch (...) {
    return -1;
  }
}

void avrf_pushloop_free(void* h) { delete static_cast<PushLoop*>(h); }

// ---- Pedersen: pedersen::BatchVerifier::push once per proof ----------------------------------------------------------
struct PedItem { std::vector<VrfIo> ios; std::vector<uint8_t> ad; pedersen::Proof proof; };

struct PedPushLoop {
  std::vector<PedItem> items;
  std::unique_ptr<pedersen::BatchVerifier<BandersnatchSha512Ell2, AVRF_FMT_MONTGOMERY>> bv;
};

// Arrays as for avrf_pedersen_batch_push_many (Bandersnatch, Montgomery format).
void* avrf_pushloop_ped_new(uint64_t n, const uint8_t* ios, const uint32_t* io_off, const uint8_t* ad,
                            const uint32_t* ad_off, const uint8_t* pk_com, const uint8_t* r, const uint8_t* ok,
                            const uint8_t* s, const uint8_t* sb) {
  try {
    auto* pl = new PedPushLoop();
    pl->items.resize(n);
    for (uint64_t j = 0; j < n; j++) {
      PedItem& it = pl->items[j];
      it.ios.resize(io_off[j + 1] - io_off[j]);
      if (!it.ios.empty()) memcpy(it.ios.data(), ios + 128 * (size_t)io_off[j], 128 * it.ios.size());
      it.ad.assign(ad + ad_off[j], ad + ad_off[j + 1]);
      memcpy(it.proof.pk_com.data(), pk_com + 64 * j, 64);
      memcpy(it.proof.r.data(), r + 64 * j, 64);
      memcpy(it.proof.ok.data(), ok + 64 * j, 64);
      memcpy(it.proof.s.data(), s + 32 * j, 32);
      memcpy(it.proof.sb.data(), sb + 32 * j, 32);
    }
    pl->bv.reset(new pedersen::BatchVerifier<BandersnatchSha512Ell2, AVRF_FMT_MONTGOMERY>());
    return pl;
  } catch (...) {
    return nullptr;
  }
}

// One step over the first n_items items (0: all): a fresh batch, push every item, verify.  one_by_one_many != 0 pushes
// each item as a one-proof avrf_pedersen_batch_push_many instead of pedersen::BatchVerifier::push (what that push
// did before single pushes were staged), for comparison.  Returns the verdict (or a negative error code); *push_ms /
// *verify_ms: host wall time of the two halves.
int avrf_pushloop_ped_step(void* h, uint64_t n_items, int one_by_one_many, double* push_ms, double* verify_ms) {
  PedPushLoop* pl = static_cast<PedPushLoop*>(h);
  const size_t n = n_items && n_items < pl->items.size() ? (size_t)n_items : pl->items.size();
  try {
    auto t0 = std::chrono::steady_clock::now();
    pl->bv->clear();
    uint64_t nio = 0, nad = 0;
    for (size_t j = 0; j < n; j++) { nio += pl->items[j].ios.size(); nad += pl->items[j].ad.size(); }
    pl->bv->reserve(n, nio, nad);
    for (size_t j = 0; j < n; j++) {
      const PedItem& it = pl->items[j];
      if (!one_by_one_many) {
        pl->bv->push(it.ios, it.ad, it.proof);
        continue;
      }
      uint32_t io_off[2] = {0, (uint32_t)it.ios.size()}, ad_off[2] = {0, (uint32_t)it.ad.size()};
      check(avrf_pedersen_batch_push_many(pl->bv->handle(), 1, it.ios.empty() ? nullptr : it.ios[0].input.data(), io_off,
                                          it.ad.empty() ? nullptr : it.ad.data(), ad_off, it.proof.pk_com.data(),
                                          it.proof.r.data(), it.proof.ok.data(), it.proof.s.data(), it.proof.sb.data()));
    }
    auto t1 = std::chrono::steady_clock::now();
    Result res = pl->bv->verify();
    auto t2 = std::chrono::steady_clock::now();
    if (push_ms) *push_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    if (verify_ms) *verify_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
    return res.status;
  } catch (...) {
    return -1;
  }
}

void avrf_pushloop_ped_free(void* h) { delete static_cast<PedPushLoop*>(h); }

}  // extern "C"
