// GPU test driver for the batch servers of include/avrf.hpp with no Python in the process: a Pedersen server fed
// decoded and wire-format batches, and a Thin server fed wire-format batches.  Reads one batch of each kind from a blob
// written by tests/test_gpu_server_schemes.py (canonical format) and checks every verdict, including a refused decode
// and the job after it on the same worker.
//
// blob: 21 arrays, each u64 byte count then the bytes:
//   Pedersen decoded: ios, io_offsets, ad, ad_offsets, pk_com, r, ok, s, sb
//   Pedersen wire:    ios32, io_offsets, ad, ad_offsets, proofs (160 B each)
//   Thin wire:        pk32, ios32, io_offsets, ad, ad_offsets, r32, s
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>
#include <vector>

#include "avrf.hpp"

using namespace ark_vrf;
using Suite = BandersnatchSha512Ell2;
using Bytes = std::vector<uint8_t>;

static const uint32_t* u32p(const Bytes& b) { return reinterpret_cast<const uint32_t*>(b.data()); }

template <class T>
static std::vector<T> as(const Bytes& b) {
  std::vector<T> v(b.size() / sizeof(T));
  if (!b.empty()) memcpy(v.data(), b.data(), b.size());
  return v;
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  std::ifstream f(argv[1], std::ios::binary);
  Bytes buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  std::vector<Bytes> a;
  for (size_t p = 0; p + 8 <= buf.size();) {
    uint64_t len;
    memcpy(&len, &buf[p], 8);
    p += 8;
    a.emplace_back(buf.begin() + p, buf.begin() + p + len);
    p += len;
  }
  if (a.size() != 21) { std::printf("bad blob: %zu arrays\n", a.size()); return 2; }
  check(avrf_init(0));
  int fails = 0;
  auto expect = [&](const char* what, long long got, long long want) {
    std::printf("%-48s %lld (want %lld)\n", what, got, want);
    if (got != want) fails++;
  };

  {  // Pedersen server: decoded jobs (a pedersen::Batch) and wire jobs
    pedersen::Batch b;
    b.ios = as<VrfIo>(a[0]);
    b.io_offsets = as<uint32_t>(a[1]);
    b.ad = as<uint8_t>(a[2]);
    b.ad_offsets = as<uint32_t>(a[3]);
    b.pk_com = as<AffinePoint>(a[4]);
    b.r = as<AffinePoint>(a[5]);
    b.ok = as<AffinePoint>(a[6]);
    b.s = as<ScalarField>(a[7]);
    b.sb = as<ScalarField>(a[8]);
    const uint64_t n = b.len();
    pedersen::Batch bad = b;
    bad.s[n / 2][0] ^= 1;
    const Bytes &ios32 = a[9], &io_off = a[10], &ad = a[11], &ad_off = a[12], &proofs = a[13];
    Bytes broken = proofs;
    memset(&broken[160 * (n - 1)], 0xff, 31);              // the last pk_com: y = 2^255 - 1 >= p
    broken[160 * (n - 1) + 31] = 0x7f;
    pedersen::BatchServer<Suite, AVRF_FMT_CANONICAL> srv(1, 1);   // one worker: the job after a refusal reuses its handle
    Bytes ok_good(n, 9), ok_bad(n, 9);
    uint64_t nb_good = 77, nb_bad = 77;
    int64_t t0 = srv.submit(b), t1 = srv.submit(bad);
    int64_t t2 = srv.submit_compressed(n, ios32.data(), u32p(io_off), ad.data(), u32p(ad_off), proofs.data(), ok_good.data(), &nb_good);
    int64_t t3 = srv.submit_compressed(n, ios32.data(), u32p(io_off), ad.data(), u32p(ad_off), broken.data(), ok_bad.data(), &nb_bad);
    int64_t t4 = srv.submit_compressed(n, ios32.data(), u32p(io_off), ad.data(), u32p(ad_off), proofs.data());
    expect("pedersen decoded: valid", srv.wait(t0).status, AVRF_OK);
    expect("pedersen decoded: one s + 1", srv.wait(t1).status, AVRF_VERIFICATION_FAILURE);
    expect("pedersen wire: valid", srv.wait(t2).status, AVRF_OK);
    expect("pedersen wire: valid, undecodable", (long long)nb_good, 0);
    long long ones = 0;
    for (uint8_t x : ok_good) ones += x == 1;
    expect("pedersen wire: valid, decode flags set", ones, (long long)n);
    expect("pedersen wire: y >= p", srv.wait(t3).status, AVRF_INVALID_DATA);
    expect("pedersen wire: y >= p, undecodable", (long long)nb_bad, 1);
    long long named = 0;
    for (uint64_t j = 0; j < n; j++) named += (ok_bad[j] == 0) == (j == n - 1);
    expect("pedersen wire: ok[] names exactly the victim", named, (long long)n);
    expect("pedersen wire: the next job verifies", srv.wait(t4).status, AVRF_OK);
  }
  {  // Thin server: wire jobs
    const Bytes &pk32 = a[14], &ios32 = a[15], &io_off = a[16], &ad = a[17], &ad_off = a[18], &r32 = a[19], &s = a[20];
    const uint64_t n = pk32.size() / 32;
    Bytes s_bad = s;
    s_bad[32 * 3] ^= 1;
    thin::BatchServer<Suite, AVRF_FMT_CANONICAL> srv(2);
    uint64_t nb = 77;
    int64_t t0 = srv.submit_compressed(n, pk32.data(), ios32.data(), u32p(io_off), ad.data(), u32p(ad_off), r32.data(), s.data(),
                                       nullptr, &nb);
    int64_t t1 = srv.submit_compressed(n, pk32.data(), ios32.data(), u32p(io_off), ad.data(), u32p(ad_off), r32.data(), s_bad.data());
    expect("thin wire: valid", srv.wait(t0).status, AVRF_OK);
    expect("thin wire: valid, undecodable", (long long)nb, 0);
    expect("thin wire: one s + 1", srv.wait(t1).status, AVRF_VERIFICATION_FAILURE);
  }
  std::printf("%s\n", fails ? "FAIL" : "ALL OK");
  return fails ? 1 : 0;
}
