// GPU test driver for ark_vrf::pedersen::BatchVerifier::push (include/avrf.hpp): pushes Pedersen proofs one by one from
// ordinary heap values, as a caller of the reference's API does, and checks the verdict and batch seed against one
// push_many of the same arrays, then a tampered proof.
//
// blob (written by tests/test_gpu_pedersen_push.py, canonical): u32 n, pk_com[64n] r[64n] ok[64n] s[32n] sb[32n],
//       io_offsets[n+1] ad_offsets[n+1] (u32), ios[128 * io_offsets[n]], ad[ad_offsets[n]]
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>
#include <vector>

#include "avrf.hpp"

using namespace ark_vrf;
using Suite = BandersnatchSha512Ell2;
constexpr uint32_t FMT = AVRF_FMT_CANONICAL;

struct Item { std::vector<VrfIo> ios; std::vector<uint8_t> ad; pedersen::Proof proof; };

static std::vector<uint8_t> seed_of(avrf_batch* h) {
  std::vector<uint8_t> seed(64);
  check(avrf_thin_batch_tap(h, AVRF_TAP_SEED, seed.data(), seed.size()));
  return seed;
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  std::ifstream f(argv[1], std::ios::binary);
  std::vector<uint8_t> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  uint32_t n;
  memcpy(&n, buf.data(), 4);
  const uint8_t* pk_com = buf.data() + 4;
  const uint8_t *r = pk_com + 64 * (size_t)n, *ok = r + 64 * (size_t)n, *s = ok + 64 * (size_t)n, *sb = s + 32 * (size_t)n;
  std::vector<uint32_t> io_off(n + 1), ad_off(n + 1);
  memcpy(io_off.data(), sb + 32 * (size_t)n, 4 * (n + 1));
  memcpy(ad_off.data(), sb + 32 * (size_t)n + 4 * (n + 1), 4 * (n + 1));
  const uint8_t* ios = sb + 32 * (size_t)n + 8 * (n + 1);
  const uint8_t* ad = ios + 128 * (size_t)io_off[n];
  std::vector<Item> items(n);
  for (uint32_t j = 0; j < n; j++) {
    Item& it = items[j];
    it.ios.resize(io_off[j + 1] - io_off[j]);
    if (!it.ios.empty()) memcpy(it.ios.data(), ios + 128 * (size_t)io_off[j], 128 * it.ios.size());
    it.ad.assign(ad + ad_off[j], ad + ad_off[j + 1]);
    memcpy(it.proof.pk_com.data(), pk_com + 64 * (size_t)j, 64);
    memcpy(it.proof.r.data(), r + 64 * (size_t)j, 64);
    memcpy(it.proof.ok.data(), ok + 64 * (size_t)j, 64);
    memcpy(it.proof.s.data(), s + 32 * (size_t)j, 32);
    memcpy(it.proof.sb.data(), sb + 32 * (size_t)j, 32);
  }
  check(avrf_init(0));
  int fails = 0;
  auto expect = [&](const char* what, long got, long want) {
    std::printf("%-44s %ld (want %ld)\n", what, got, want);
    if (got != want) fails++;
  };
  pedersen::BatchVerifier<Suite, FMT> ref;
  check(avrf_pedersen_batch_push_many(ref.handle(), n, ios, io_off.data(), ad, ad_off.data(), pk_com, r, ok, s, sb));
  expect("push_many: Ok", ref.verify().status, AVRF_OK);
  {
    pedersen::BatchVerifier<Suite, FMT> bv;
    bv.reserve(n, io_off[n], ad_off[n]);
    for (const Item& it : items) bv.push(it.ios, it.ad, it.proof);
    expect("len after the push loop", (long)bv.len(), (long)n);
    expect("push loop: Ok", bv.verify().status, AVRF_OK);
    expect("push loop: the seed of push_many", seed_of(bv.handle()) == seed_of(ref.handle()), 1);
  }
  {
    pedersen::BatchVerifier<Suite, FMT> bv;
    const uint32_t bad = n - n / 3;
    for (uint32_t j = 0; j < n; j++) {
      pedersen::Proof pf = items[j].proof;
      if (j == bad) pf.sb[0] ^= 1;
      bv.push(items[j].ios, items[j].ad, pf);
    }
    expect("one tampered sb", bv.verify().status, AVRF_VERIFICATION_FAILURE);
    auto inv = bv.find_invalid();
    expect("find_invalid names it", inv.size() == 1 && inv[0] == bad, 1);
  }
  std::printf("%s\n", fails ? "FAIL" : "ALL OK");
  return fails ? 1 : 0;
}
