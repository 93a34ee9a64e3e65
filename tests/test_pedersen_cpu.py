"""CPU: the Pedersen VRF without a GPU.

1. The oracle's pedersen_prove reproduces the reference's 21 Pedersen golden vectors (blinding included) and its
   pedersen_verify accepts them and rejects a small-order component on Ok.
2. The device prover and single verifier (csrc/pedersen.cuh), compiled for the host with the carry flag emulated,
   match the golden vectors and the oracle on random cases, and give the oracle's verdict on small-order faults.
3. The C++ mirror of the Pedersen API (include/avrf.hpp) compiles, links, and throws without a device."""
import ctypes
import json
import os
import random
import subprocess
import tempfile

import pytest

from oracle import pyref as o

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
R = 1 << 256


def _golden(S):
    with open(os.path.join(HERE, "golden", f"{S.name}_pedersen.json")) as f:
        return json.load(f)


def _t2(S):
    return (0, S.p - 1)                   # the point of order 2


def _proof_of(S, v):
    d = lambda k: o.dec_point(S, bytes.fromhex(v[k]))
    i = lambda k: int.from_bytes(bytes.fromhex(v[k]), "little")
    return o.PedersenProof(d("proof_pk_com"), d("proof_r"), d("proof_ok"), i("proof_s"), i("proof_sb"))


@pytest.mark.parametrize("sid", [0, 1, 2])
def test_oracle_reproduces_golden_vectors(sid):
    S = o.SUITES[sid]
    vs = _golden(S)
    assert len(vs) == 7
    for v in vs:
        sk = int.from_bytes(bytes.fromhex(v["sk"]), "little")
        ios = [(o.dec_point(S, bytes.fromhex(v["h"])), o.dec_point(S, bytes.fromhex(v["gamma"])))]
        ad = bytes.fromhex(v["ad"])
        pf, blinding = o.pedersen_prove(S, sk, ios, ad)
        assert o.enc_point(S, pf.pk_com).hex() == v["proof_pk_com"]
        assert o.enc_point(S, pf.r).hex() == v["proof_r"]
        assert o.enc_point(S, pf.ok).hex() == v["proof_ok"]
        assert o.enc_scalar(pf.s).hex() == v["proof_s"]
        assert o.enc_scalar(pf.sb).hex() == v["proof_sb"]
        assert o.enc_scalar(blinding).hex() == v["blinding"]
        assert o.pedersen_verify(S, ios, ad, pf) == o.OK
        bad = o.PedersenProof(pf.pk_com, pf.r, o.pt_add(S, pf.ok, _t2(S)), pf.s, pf.sb)
        assert o.pedersen_verify(S, ios, ad, bad) == o.VERIFICATION_FAILURE


# ---- host emulation of the device functions -------------------------------------------------------------------------

@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    src = os.path.join(HERE, "hostemu", "pedersen_emu.cpp")
    so = str(tmp_path_factory.mktemp("pedersen_emu") / "libpedersen_emu.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so, src])
    return ctypes.CDLL(so)


def _w(x):
    return [(x >> (32 * i)) & 0xFFFFFFFF for i in range(8)]


def _sc(x):
    return (ctypes.c_uint32 * 8)(*_w(x))


def _aff(S, *pts):
    return (ctypes.c_uint32 * (16 * max(1, len(pts))))(*[w for P in pts for c in P for w in _w(c * R % S.p)])


def _unaff(S, a):
    ri = pow(R, -1, S.p)
    u = lambda k: sum(int(a[k + i]) << (32 * i) for i in range(8))
    return (u(0) * ri % S.p, u(8) * ri % S.p)


def _uint(a):
    return sum(int(a[i]) << (32 * i) for i in range(8))


def _emu_prove(emu, sid, sk, ios, ad):
    S = o.SUITES[sid]
    pk = o.public_key(S, sk)
    flat = [P for io in ios for P in io]
    outs = [(ctypes.c_uint32 * 16)() for _ in range(3)] + [(ctypes.c_uint32 * 8)() for _ in range(3)]
    emu.emu_ped_prove(sid, _sc(sk), _aff(S, pk), _aff(S, *flat), len(ios), ad, len(ad), *outs)
    pf = o.PedersenProof(_unaff(S, outs[0]), _unaff(S, outs[1]), _unaff(S, outs[2]), _uint(outs[3]), _uint(outs[4]))
    return pf, _uint(outs[5])


def _emu_verify(emu, sid, ios, ad, pf):
    S = o.SUITES[sid]
    flat = [P for io in ios for P in io]
    return emu.emu_ped_verify(sid, _aff(S, *flat), len(ios), ad, len(ad), _aff(S, pf.pk_com), _aff(S, pf.r),
                              _aff(S, pf.ok), _sc(pf.s), _sc(pf.sb))


@pytest.mark.parametrize("sid", [0, 1, 2])
def test_emulated_prover_and_verifier_golden(emu, sid):
    S = o.SUITES[sid]
    for v in _golden(S):
        sk = int.from_bytes(bytes.fromhex(v["sk"]), "little")
        ios = [(o.dec_point(S, bytes.fromhex(v["h"])), o.dec_point(S, bytes.fromhex(v["gamma"])))]
        ad = bytes.fromhex(v["ad"])
        pf, blinding = _emu_prove(emu, sid, sk, ios, ad)
        assert o.enc_point(S, pf.pk_com).hex() == v["proof_pk_com"]
        assert o.enc_point(S, pf.r).hex() == v["proof_r"]
        assert o.enc_point(S, pf.ok).hex() == v["proof_ok"]
        assert o.enc_scalar(pf.s).hex() == v["proof_s"]
        assert o.enc_scalar(pf.sb).hex() == v["proof_sb"]
        assert o.enc_scalar(blinding).hex() == v["blinding"]
        assert _emu_verify(emu, sid, ios, ad, _proof_of(S, v)) == o.OK


def test_emulated_prover_and_verifier_vs_oracle(emu):
    """50 random cases: ragged M in {0, 1, 2, 5}, ad of 0..300 bytes, all three suites; the small-order faults
    Ok + T2 and R + T2 get the oracle's verdict."""
    rnd = random.Random(0x9ed)
    for case in range(50):
        sid = case % 3
        S = o.SUITES[sid]
        sk = o.secret_from_seed(S, rnd.randrange(1 << 64).to_bytes(8, "little") + bytes(24))
        m = rnd.choice([0, 1, 2, 5])
        ios = []
        for i in range(m):
            inp = o.data_to_point(S, b"ped-%d-%d" % (case, i))
            ios.append((inp, o.pt_mul(S, inp, sk)))
        ad = bytes(rnd.randrange(256) for _ in range(rnd.randrange(301)))
        want, want_bl = o.pedersen_prove(S, sk, ios, ad)
        got, got_bl = _emu_prove(emu, sid, sk, ios, ad)
        assert (got, got_bl) == (want, want_bl), (case, sid, m)
        assert _emu_verify(emu, sid, ios, ad, got) == o.pedersen_verify(S, ios, ad, got) == o.OK
        for bad in (o.PedersenProof(got.pk_com, got.r, o.pt_add(S, got.ok, _t2(S)), got.s, got.sb),
                    o.PedersenProof(got.pk_com, o.pt_add(S, got.r, _t2(S)), got.ok, got.s, got.sb)):
            assert _emu_verify(emu, sid, ios, ad, bad) == o.pedersen_verify(S, ios, ad, bad) == o.VERIFICATION_FAILURE


# ---- C++ mirror -----------------------------------------------------------------------------------------------------

CPP = r'''
#include "avrf.hpp"
#include <cstdio>
using namespace ark_vrf;
int main() {
  using Suite = BandersnatchSha512Ell2;
  int threw = 0;
  pedersen::Proof p{};
  try {
    Result r = pedersen::verify<Suite>({}, {}, p);
    std::printf("verdict %d\n", r.status);
  } catch (const std::exception& e) { threw++; }
  try {
    pedersen::BatchVerifier<Suite> bv;
    bv.push({}, {}, p);
    std::printf("verdict %d\n", bv.verify().status);
    std::printf("each %zu\n", bv.verify_each().size());
  } catch (const std::exception& e) { threw++; }
  try {
    std::vector<ScalarField> sk(1);
    std::vector<AffinePoint> pk(1);
    std::vector<uint32_t> io_off{0, 0}, ad_off{0, 0};
    auto out = pedersen::prove_many<Suite>(sk, pk, {}, io_off, {}, ad_off);
    std::printf("proofs %zu\n", out.proofs.size());
  } catch (const std::exception& e) { threw++; }
  std::printf("threw %d\n", threw);
  return 0;
}
'''


def test_cpp_pedersen_mirror_compiles_links_and_throws_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "t.cpp")
        open(src, "w").write(CPP)
        exe = os.path.join(d, "t")
        lib = os.path.join(ROOT, "ark_vrf_b200")
        subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                               "-L", lib, "-l:libavrf_gpu.so", "-Wl,-rpath," + lib])
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stderr
        assert "threw 3" in out.stdout and "verdict" not in out.stdout, out.stdout
