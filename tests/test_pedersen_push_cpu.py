"""CPU: the Pedersen single push (avrf_pedersen_batch_push) refuses a null handle without touching a device, and the
C++ classes that call it (pedersen::BatchVerifier::push / reserve in include/avrf.hpp) compile and link."""
import os
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_null_handle_is_an_argument_error():
    import ark_vrf_b200 as av
    lib = av.load()
    pt, sc = bytes(64), bytes(32)
    assert lib.avrf_pedersen_batch_push(None, None, 0, None, 0, pt, pt, pt, sc, sc) == -2
    assert b"null argument" in lib.avrf_last_error()


SRC = r'''
#include "avrf.hpp"
#include <cstdio>
using namespace ark_vrf;
int main() {
  try {
    pedersen::BatchVerifier<BandersnatchSha512Ell2> bv;
    bv.reserve(4, 4, 64);
    bv.push({}, {}, pedersen::Proof{});
    std::printf("len %lld\n", (long long)bv.len());
  } catch (const std::exception& e) {
    std::printf("error: %s\n", e.what());
  }
  return 0;
}
'''


def test_cpp_push_compiles_and_links():
    import ark_vrf_b200 as av
    av.load()
    pkg = os.path.join(ROOT, "ark_vrf_b200")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "p.cpp"), os.path.join(d, "p")
        open(src, "w").write(SRC)
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                               "-L", pkg, "-l:libavrf_gpu.so", "-Wl,-rpath," + pkg])
