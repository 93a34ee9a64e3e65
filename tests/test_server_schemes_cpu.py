"""CPU: the Pedersen batch server and the wire-format submits - the constructors refuse to run without a CUDA device
(no CPU fallback), the submits refuse a null server, and the C++ classes of include/avrf.hpp compile and link."""
import ctypes
import os
import subprocess
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def no_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")


def test_constructors_need_a_device(no_gpu):
    import ark_vrf_b200 as av
    from ark_vrf_b200 import pedersen as ped
    lib = av.load()
    assert lib.avrf_pedersen_server_new(0, 1, 2, 0, 0) is None
    assert b"no CUDA device" in lib.avrf_last_error()
    with pytest.raises(av.AvrfError, match="no CUDA device"):
        ped.BatchServer(0, workers=2)
    assert lib.avrf_pedersen_server_new(0, 2, 2, 0, 0) is None                # bad format: an argument error first
    assert b"bad suite/fmt" in lib.avrf_last_error()


def test_submits_refuse_a_null_server():
    import ark_vrf_b200 as av
    lib = av.load()
    nb = ctypes.c_uint64(5)
    assert lib.avrf_pedersen_server_submit(None, 0, *[None] * 9) == -2
    assert lib.avrf_server_submit_compressed(None, 0, *[None] * 7, None, ctypes.byref(nb)) == -2
    assert lib.avrf_pedersen_server_submit_compressed(None, 0, *[None] * 5, None, ctypes.byref(nb)) == -2
    assert b"null server" in lib.avrf_last_error()


SRC = r'''
#include "avrf.hpp"
#include <cstdio>
using namespace ark_vrf;
int main() {
  try {
    pedersen::BatchServer<BandersnatchSha512Ell2> srv(2, 1, 1);
    pedersen::Batch b;
    b.push({}, {}, pedersen::Proof{});
    std::printf("status %d\n", srv.wait(srv.submit(b)).status);
    uint8_t rec[160] = {};
    uint32_t off[2] = {0, 0};
    std::printf("status %d\n", srv.wait(srv.submit_compressed(1, nullptr, off, nullptr, off, rec)).status);
  } catch (const std::exception& e) {
    std::printf("error: %s\n", e.what());
  }
  try {
    thin::BatchServer<Ed25519Sha512Tai, AVRF_FMT_CANONICAL> srv(1);
    uint8_t pt[32] = {}, s[32] = {}, ok[1];
    uint32_t off[2] = {0, 0};
    uint64_t bad = 0;
    std::printf("status %d\n", srv.wait(srv.submit_compressed(1, pt, nullptr, off, nullptr, off, pt, s, ok, &bad)).status);
  } catch (const std::exception& e) {
    std::printf("error: %s\n", e.what());
  }
  return 0;
}
'''


def test_cpp_server_classes_compile_and_link():
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "t.cpp")
        open(src, "w").write(SRC)
        exe = os.path.join(d, "t")
        lib = os.path.join(ROOT, "ark_vrf_b200")
        subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                               "-L", lib, "-l:libavrf_gpu.so", "-Wl,-rpath," + lib])
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0
        assert out.stdout.count("error:") + out.stdout.count("status") >= 2
