// GPU test driver for ark_vrf::pedersen (include/avrf.hpp): reads oracle-made Pedersen proofs from a blob written by
// tests/test_gpu_pedersen.py, proves the same statements with prove_many, and verifies them one by one, as a batch and
// per proof.
//
// blob: u32 n, sk[32], pk[64], then per proof: n_ios(u32) ios[128*n_ios] ad_len(u32) ad[ad_len]
//       pk_com[64] r[64] ok[64] s[32] sb[32]      (canonical; every proof signed by sk)
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
  ScalarField sk;
  AffinePoint pk;
  bytes(sk.data(), 32);
  bytes(pk.data(), 64);
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
  check(avrf_init(0));
  int fails = 0;
  auto expect = [&](const char* what, int got, int want) {
    std::printf("%-40s %d (want %d)\n", what, got, want);
    if (got != want) fails++;
  };
  {  // prove the same statements: the same proofs, bit for bit
    std::vector<VrfIo> ios;
    std::vector<uint8_t> ad;
    std::vector<uint32_t> io_off{0}, ad_off{0};
    for (auto& it : items) {
      ios.insert(ios.end(), it.ios.begin(), it.ios.end());
      ad.insert(ad.end(), it.ad.begin(), it.ad.end());
      io_off.push_back((uint32_t)ios.size());
      ad_off.push_back((uint32_t)ad.size());
    }
    auto out = pedersen::prove_many<Suite, FMT>(std::vector<ScalarField>(n, sk), std::vector<AffinePoint>(n, pk), ios,
                                               io_off, ad, ad_off);
    int same = 0;
    for (uint32_t j = 0; j < n; j++) same += memcmp(&out.proofs[j], &items[j].proof, sizeof(pedersen::Proof)) == 0;
    expect("prove_many equals the oracle's proofs", same, (int)n);
  }
  for (auto& it : items) expect("verify", pedersen::verify<Suite, FMT>(it.ios, it.ad, it.proof).status, AVRF_OK);
  {
    pedersen::BatchVerifier<Suite, FMT> bv;
    for (auto& it : items) bv.push(it.ios, it.ad, it.proof);
    expect("batch of valid proofs", bv.verify().status, AVRF_OK);
    int ok = 0;
    for (int32_t s : bv.verify_each()) ok += s == AVRF_OK;
    expect("verify_each: all Ok", ok, (int)n);
  }
  {
    pedersen::BatchVerifier<Suite, FMT> bv;
    for (uint32_t j = 0; j < n; j++) {
      auto pf = items[j].proof;
      if (j == 3) pf.s[0] ^= 1;
      bv.push(items[j].ios, items[j].ad, pf);
    }
    expect("one bad s", bv.verify().status, AVRF_VERIFICATION_FAILURE);
    auto bad = bv.find_invalid();
    expect("find_invalid names it", bad.size() == 1 && bad[0] == 3, 1);
  }
  std::printf("%s\n", fails ? "FAIL" : "ALL OK");
  return fails ? 1 : 0;
}
