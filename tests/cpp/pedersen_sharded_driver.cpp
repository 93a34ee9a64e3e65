// GPU test driver, no Python in the process: one Pedersen batch over every GPU of the box through the C++ mirror
// (include/avrf.hpp: init_multi + pedersen::ShardedBatchVerifier over avrf_pedersen_sharded_* and avrf_thin_sharded_*).
// Reads oracle-made Pedersen proofs written by tests/test_gpu_pedersen_sharded.py, repeats them to a few thousand
// proofs so that every device gets a share, and checks accept / reject / InvalidData against a single-device
// pedersen::BatchVerifier.
//
// blob: u32 n, then per proof: n_ios(u32) ios[128*n_ios] ad_len(u32) ad[ad_len] pk_com[64] r[64] ok[64] s[32] sb[32]
//       (canonical)
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

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  std::ifstream f(argv[1], std::ios::binary);
  std::vector<uint8_t> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  size_t p = 0;
  auto u32 = [&]() { uint32_t v; memcpy(&v, &buf[p], 4); p += 4; return v; };
  auto bytes = [&](void* dst, size_t n) { memcpy(dst, &buf[p], n); p += n; };
  uint32_t n = u32();
  std::vector<Item> items(n);
  for (auto& it : items) {
    it.ios.resize(u32());
    for (auto& io : it.ios) { bytes(io.input.data(), 64); bytes(io.output.data(), 64); }
    it.ad.resize(u32());
    if (!it.ad.empty()) bytes(it.ad.data(), it.ad.size());
    bytes(it.proof.pk_com.data(), 64);
    bytes(it.proof.r.data(), 64);
    bytes(it.proof.ok.data(), 64);
    bytes(it.proof.s.data(), 32);
    bytes(it.proof.sb.data(), 32);
  }
  int ndev = pedersen::init_multi(0);
  std::printf("devices: %d\n", ndev);
  const size_t reps = 701;                       // 6 proofs x 701 = 4206 proofs
  // s + 1: a valid scalar but a wrong response (it would reach r only for s = r - 1, which no proof here holds)
  auto bump = [](ScalarField& x) {
    for (auto& byte : x)
      if (++byte != 0) break;
  };
  auto build = [&](long bad_s, long bad_sb, long ident_at) {
    pedersen::Batch b;
    for (size_t r = 0; r < reps; r++)
      for (size_t i = 0; i < items.size(); i++) {
        long idx = (long)(r * items.size() + i);
        auto pf = items[i].proof;
        if (idx == bad_s) bump(pf.s);
        if (idx == bad_sb) bump(pf.sb);
        if (idx == ident_at) { pf.pk_com.fill(0); pf.pk_com[32] = 1; }
        b.push(items[i].ios, items[i].ad, pf);
      }
    return b;
  };
  int fails = 0;
  auto expect = [&](const char* what, long got, long want) {
    std::printf("%-48s %ld (want %ld)\n", what, got, want);
    if (got != want) fails++;
  };
  long total = (long)(reps * items.size());
  pedersen::ShardedBatchVerifier<Suite, FMT> sh;
  expect("devices of the sharded handle", sh.devices(), ndev);
  uint8_t seed_sh[64], seed_one[64];
  {
    pedersen::Batch b = build(-1, -1, -1);
    sh.push_many(b);
    expect("sharded: proofs", sh.len(), total);
    expect("sharded: valid batch", sh.verify().status, AVRF_OK);
    expect("sharded: verify is repeatable", sh.verify().status, AVRF_OK);
    check(avrf_thin_sharded_seed(sh.handle(), seed_sh));
    pedersen::BatchVerifier<Suite, FMT> one;
    check(avrf_pedersen_batch_push_many(one.handle(), b.len(), b.ios[0].input.data(), b.io_offsets.data(), b.ad.data(),
                                        b.ad_offsets.data(), b.pk_com[0].data(), b.r[0].data(), b.ok[0].data(),
                                        b.s[0].data(), b.sb[0].data()));
    expect("single device: valid batch", one.verify().status, AVRF_OK);
    check(avrf_thin_batch_tap(one.handle(), AVRF_TAP_SEED, seed_one, 64));
    expect("seed equals the single-device seed", memcmp(seed_sh, seed_one, 64) == 0, 1);
    // a Thin push on a Pedersen handle is refused and changes nothing
    const AffinePoint pt{};
    const ScalarField sc{};
    const uint32_t off[2] = {0, 0};
    expect("thin push on a Pedersen handle",
           avrf_thin_sharded_push_many(sh.handle(), 1, pt.data(), nullptr, off, nullptr, off, pt.data(), sc.data()),
           AVRF_ERR_ARG);
    uint8_t seed_after[64];
    check(avrf_thin_sharded_seed(sh.handle(), seed_after));
    expect("... proofs kept", sh.len(), total);
    expect("... seed kept", memcmp(seed_sh, seed_after, 64) == 0, 1);
  }
  for (long bad : {0L, total / 2, total - 1}) {
    sh.clear();
    sh.push_many(build(bad, -1, -1));
    expect("sharded: one bad s", sh.verify().status, AVRF_VERIFICATION_FAILURE);
    sh.clear();
    sh.push_many(build(-1, bad, -1));
    expect("sharded: one bad sb", sh.verify().status, AVRF_VERIFICATION_FAILURE);
  }
  {
    sh.clear();
    sh.push_many(build(3, -1, total - 2));
    expect("sharded: identity pk_com + bad s", sh.verify().status, AVRF_INVALID_DATA);
  }
  {
    sh.clear();
    expect("sharded: empty batch", sh.verify().status, AVRF_OK);
  }
  std::printf("%s\n", fails ? "FAIL" : "ALL OK");
  return fails ? 1 : 0;
}
