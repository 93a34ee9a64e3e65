// GPU test driver for ark_vrf::pedersen::BatchVerifier::push_compressed (include/avrf.hpp): reads wire-format Pedersen
// proofs from a blob written by tests/test_gpu_pedersen_wire.py, pushes them, then pushes them again with one
// undecodable public-key commitment (y >= p), which must be refused without touching the batch.
//
// blob: u32 n, u32 n_ios, u32 ad_len, proofs[160 n], ios32[64 n_ios], io_offsets[u32 (n+1)], ad_offsets[u32 (n+1)],
//       ad[ad_len]
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>
#include <vector>

#include "avrf.hpp"

using namespace ark_vrf;
using Suite = BandersnatchSha512Ell2;

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  std::ifstream f(argv[1], std::ios::binary);
  std::vector<uint8_t> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  size_t p = 0;
  auto u32 = [&]() { uint32_t v; memcpy(&v, &buf[p], 4); p += 4; return v; };
  auto bytes = [&](void* dst, size_t n) { if (n) memcpy(dst, &buf[p], n); p += n; };
  const uint32_t n = u32(), n_ios = u32(), ad_len = u32();
  std::vector<uint8_t> proofs(160 * (size_t)n), ios32(64 * (size_t)n_ios + 64), ad(ad_len + 16);
  std::vector<uint32_t> io_off(n + 1), ad_off(n + 1);
  bytes(proofs.data(), proofs.size());
  bytes(ios32.data(), 64 * (size_t)n_ios);
  bytes(io_off.data(), 4 * (size_t)(n + 1));
  bytes(ad_off.data(), 4 * (size_t)(n + 1));
  bytes(ad.data(), ad_len);
  check(avrf_init(0));
  int fails = 0;
  auto expect = [&](const char* what, long long got, long long want) {
    std::printf("%-44s %lld (want %lld)\n", what, got, want);
    if (got != want) fails++;
  };
  pedersen::BatchVerifier<Suite> bv;      // Montgomery handle: the wire format is the same for both
  std::vector<uint8_t> ok;
  uint64_t bad = bv.push_compressed(n, ios32.data(), io_off.data(), ad.data(), ad_off.data(), proofs.data(), &ok);
  expect("good proofs: undecodable", (long long)bad, 0);
  expect("good proofs: len", bv.len(), n);
  expect("good proofs: verify", bv.verify().status, AVRF_OK);
  const uint32_t victim = n / 2;
  std::vector<uint8_t> broken = proofs;
  memset(&broken[160 * (size_t)victim], 0xff, 31);          // pk_com: y = 2^255 - 1, above p for every suite
  broken[160 * (size_t)victim + 31] = 0x7f;
  bad = bv.push_compressed(n, ios32.data(), io_off.data(), ad.data(), ad_off.data(), broken.data(), &ok);
  expect("one y >= p: undecodable", (long long)bad, 1);
  int named = 0;
  for (uint32_t j = 0; j < n; j++) named += (ok[j] == 0) == (j == victim);
  expect("ok[] names exactly the victim", named, n);
  expect("len unchanged", bv.len(), n);
  expect("the pushed batch verifies", bv.verify().status, AVRF_OK);
  std::printf("%s\n", fails ? "FAIL" : "ALL OK");
  return fails ? 1 : 0;
}
