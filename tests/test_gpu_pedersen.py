"""GPU: the Pedersen VRF prover, exact single verifier and per-proof verdicts (avrf_pedersen_prove_many,
avrf_pedersen_verify_one, avrf_pedersen_batch_verify_each) against the reference's golden vectors and the oracle."""
import copy
import json
import os
import random

import numpy as np
import pytest

from oracle import pyref as o
from helpers import pt_bytes, pt_from_bytes, sc_bytes

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FULL = os.environ.get("AVRF_FULL_CONFIGS", "1") == "1"


@pytest.fixture(scope="module")
def av():
    import ark_vrf_b200 as a
    a.load().avrf_init(0)
    return a


def _golden(S):
    with open(os.path.join(HERE, "golden", f"{S.name}_pedersen.json")) as f:
        return json.load(f)


def _fp(S, x, mont):
    return ((x << 256) % S.p if mont else x).to_bytes(32, "little")


def _fr(S, x, mont):
    return ((x << 256) % S.r if mont else x).to_bytes(32, "little")


def _pb(S, P, mont):
    return _fp(S, P[0], mont) + _fp(S, P[1], mont)


def _arr(b, w):
    return np.frombuffer(b, dtype=np.uint8).reshape(-1, w).copy()


def _blob(cases, S, mont):
    """cases: (ios, ad, ...) -> ios array, io_offsets, ad blob, ad_offsets"""
    iob = b"".join(_pb(S, i, mont) + _pb(S, x, mont) for c in cases for (i, x) in c[0])
    io_off = np.zeros(len(cases) + 1, dtype=np.uint32)
    io_off[1:] = np.cumsum([len(c[0]) for c in cases])
    ad_off = np.zeros(len(cases) + 1, dtype=np.uint32)
    ad_off[1:] = np.cumsum([len(c[1]) for c in cases])
    return (np.frombuffer(iob + bytes(128), dtype=np.uint8).copy(), io_off,
            np.frombuffer(b"".join(c[1] for c in cases) + bytes(16), dtype=np.uint8).copy(), ad_off)


def _prove(av, sid, sks, cases, mont):
    from ark_vrf_b200 import ops
    S = o.SUITES[sid]
    ios, io_off, ad, ad_off = _blob(cases, S, mont)
    sk = _arr(b"".join(_fr(S, k, mont) for k in sks), 32)
    pk = _arr(b"".join(_pb(S, o.public_key(S, k), mont) for k in sks), 64)
    fmt = av.Format.MONTGOMERY if mont else av.Format.CANONICAL
    return ops.pedersen_prove_many(sid, sk, pk, ios, io_off, ad, ad_off, fmt)


def _unfmt_pt(S, b, mont):
    x, y = pt_from_bytes(b)
    if mont:
        ri = pow(1 << 256, -1, S.p)
        x, y = x * ri % S.p, y * ri % S.p
    return (x, y)


def _unfmt_sc(S, b, mont):
    k = int.from_bytes(bytes(b), "little")
    return k * pow(1 << 256, -1, S.r) % S.r if mont else k


def _proof_arrays(S, pfs, mont):
    return (_arr(b"".join(_pb(S, p.pk_com, mont) for p in pfs), 64), _arr(b"".join(_pb(S, p.r, mont) for p in pfs), 64),
            _arr(b"".join(_pb(S, p.ok, mont) for p in pfs), 64), _arr(b"".join(_fr(S, p.s, mont) for p in pfs), 32),
            _arr(b"".join(_fr(S, p.sb, mont) for p in pfs), 32))


def _ped_proof(S, p, mont):
    from ark_vrf_b200 import pedersen as ped
    return ped.Proof(_pb(S, p.pk_com, mont), _pb(S, p.r, mont), _pb(S, p.ok, mont), _fr(S, p.s, mont), _fr(S, p.sb, mont))


def _verify_one(av, sid, ios, ad, pf, mont=False):
    """status of avrf_pedersen_verify_one"""
    from ark_vrf_b200 import pedersen as ped
    S = o.SUITES[sid]
    fmt = av.Format.MONTGOMERY if mont else av.Format.CANONICAL
    try:
        ped.verify(sid, [(_pb(S, i, mont), _pb(S, x, mont)) for i, x in ios], ad, _ped_proof(S, pf, mont), fmt)
        return 0
    except av.VerificationFailure:
        return 1
    except av.InvalidData:
        return 2


def _batch(av, sid, cases, mont=False):
    from ark_vrf_b200 import pedersen as ped
    S = o.SUITES[sid]
    bv = ped.BatchVerifier(sid, av.Format.MONTGOMERY if mont else av.Format.CANONICAL)
    ios, io_off, ad, ad_off = _blob(cases, S, mont)
    bv.push_many(ios, io_off, ad, ad_off, *_proof_arrays(S, [c[2] for c in cases], mont))
    return bv


@pytest.mark.parametrize("sid", [0, 1, 2])
@pytest.mark.parametrize("mont", [False, True])
def test_golden_vectors(av, sid, mont):
    from ark_vrf_b200 import ops
    S = o.SUITES[sid]
    vs = _golden(S)
    sks = [int.from_bytes(bytes.fromhex(v["sk"]), "little") for v in vs]
    cases = [([(o.dec_point(S, bytes.fromhex(v["h"])), o.dec_point(S, bytes.fromhex(v["gamma"])))], bytes.fromhex(v["ad"]))
             for v in vs]
    pkc, r, ok, s, sb, bl = _prove(av, sid, sks, cases, mont)
    fmt = av.Format.MONTGOMERY if mont else av.Format.CANONICAL
    for arr, key in ((pkc, "proof_pk_com"), (r, "proof_r"), (ok, "proof_ok")):
        assert [bytes(x).hex() for x in ops.point_compress(sid, arr, fmt)] == [v[key] for v in vs]
    for arr, key in ((s, "proof_s"), (sb, "proof_sb"), (bl, "blinding")):
        assert [sc_bytes(_unfmt_sc(S, x, mont)).hex() for x in arr] == [v[key] for v in vs]
    pfs = [o.PedersenProof(_unfmt_pt(S, pkc[j], mont), _unfmt_pt(S, r[j], mont), _unfmt_pt(S, ok[j], mont),
                           _unfmt_sc(S, s[j], mont), _unfmt_sc(S, sb[j], mont)) for j in range(len(vs))]
    full = [(c[0], c[1], pf) for c, pf in zip(cases, pfs)]
    for ios, ad, pf in full:
        assert _verify_one(av, sid, ios, ad, pf, mont) == 0
    bv = _batch(av, sid, full, mont)
    assert list(bv.verify_each()) == [0] * len(vs)
    assert bv.verify_status() == 0


@pytest.mark.parametrize("sid", [0, 1, 2])
def test_prover_vs_oracle(av, sid):
    """Bit-exact against pyref.pedersen_prove: M in {0, 1, 2, 3, 5, 12}, ragged ad."""
    S = o.SUITES[sid]
    rnd = random.Random(100 + sid)
    sks, cases = [], []
    for j, m in enumerate([0, 1, 2, 3, 5, 12, 1, 0]):
        sk = o.secret_from_seed(S, rnd.randrange(1 << 64).to_bytes(8, "little") + bytes(24))
        ios = []
        for i in range(m):
            inp = o.data_to_point(S, b"pv-%d-%d" % (j, i))
            ios.append((inp, o.pt_mul(S, inp, sk)))
        sks.append(sk)
        cases.append((ios, bytes(rnd.randrange(256) for _ in range(rnd.choice([0, 1, 17, 128, 300])))))
    pkc, r, ok, s, sb, bl = _prove(av, sid, sks, cases, False)
    for j, (ios, ad) in enumerate(cases):
        want, wbl = o.pedersen_prove(S, sks[j], ios, ad)
        got = o.PedersenProof(pt_from_bytes(pkc[j]), pt_from_bytes(r[j]), pt_from_bytes(ok[j]),
                              int.from_bytes(bytes(s[j]), "little"), int.from_bytes(bytes(sb[j]), "little"))
        assert got == want, (sid, j)
        assert int.from_bytes(bytes(bl[j]), "little") == wbl


def _fault_cases(sid):
    """Valid proofs, then each fault of the list; returns [(ios, ad, proof)]."""
    S = o.SUITES[sid]
    t2 = (0, S.p - 1)
    sk = o.secret_from_seed(S, bytes(32))
    good = []
    for j, m in enumerate([1, 2, 0, 1, 3, 1, 4, 1]):
        ios = []
        for i in range(m):
            inp = o.data_to_point(S, b"f-%d-%d" % (j, i))
            ios.append((inp, o.pt_mul(S, inp, sk)))
        ad = b"ad-%d" % j
        good.append((ios, ad, o.pedersen_prove(S, sk, ios, ad)[0]))
    cases = list(copy.deepcopy(good))
    bad = copy.deepcopy(good)
    bad[0][2].s = (bad[0][2].s + 1) % S.r
    bad[1][2].sb = (bad[1][2].sb + 1) % S.r
    bad[2] = (bad[2][0], bad[2][1][:-1] + bytes([bad[2][1][-1] ^ 1]), bad[2][2])
    bad[3] = ([(bad[3][0][0][0], good[5][0][0][1])], bad[3][1], bad[3][2])            # O swapped with a neighbour's
    bad[4][2].r = o.pt_add(S, bad[4][2].r, S.G)
    bad[5][2].ok = o.pt_add(S, bad[5][2].ok, t2)
    bad[7][2].r = o.pt_add(S, bad[7][2].r, t2)
    cases += [bad[i] for i in (0, 1, 2, 3, 4, 5, 7)]
    f = copy.deepcopy(good[0]); f[2].pk_com = o.IDENTITY
    cases.append(f)
    ios = [(o.data_to_point(S, b"h-%d" % i), None) for i in range(4)]
    ios = [(i, o.pt_mul(S, i, sk)) for i, _ in ios]
    ios[2] = (o.IDENTITY, ios[2][1])                                                   # identity I hidden at M = 4
    cases.append((ios, b"id", o.pedersen_prove(S, sk, ios, b"id")[0]))
    f = copy.deepcopy(good[1]); f[2].pk_com = o.IDENTITY; f[2].s = (f[2].s + 1) % S.r
    cases.append(f)
    return cases


@pytest.mark.parametrize("sid", [0, 1, 2])
def test_verdicts_vs_oracle(av, sid):
    S = o.SUITES[sid]
    cases = _fault_cases(sid)
    want = [o.pedersen_verify(S, ios, ad, pf) for ios, ad, pf in cases]
    assert want.count(0) == 8 and want.count(1) == 7 and want.count(2) == 3
    bv = _batch(av, sid, cases)
    assert list(bv.verify_each()) == want
    assert [_verify_one(av, sid, ios, ad, pf) for ios, ad, pf in cases] == want
    items = [o.pedersen_batch_prepare(S, ios, ad, pf) for ios, ad, pf in cases]
    assert bv.verify_status() == o.pedersen_batch_verify(S, items) == 2
    ok_only = [c for c, w in zip(cases, want) if w != 2]
    bv2 = _batch(av, sid, ok_only)
    items = [o.pedersen_batch_prepare(S, ios, ad, pf) for ios, ad, pf in ok_only]
    assert bv2.verify_status() == o.pedersen_batch_verify(S, items) == 1
    assert list(bv2.find_invalid()) == [j for j, c in enumerate(ok_only) if o.pedersen_verify(S, *c) != 0]


def test_argument_errors_and_wrong_schemes(av):
    from ark_vrf_b200 import pedersen as ped
    import ctypes
    sid, S = 0, o.BANDERSNATCH
    ios, ad, pf = _fault_cases(sid)[0]
    lib = av.load()
    for bad_s in (S.r, (1 << 256) - 1):
        p = copy.deepcopy(pf); p.s = bad_s
        with pytest.raises(av.AvrfError):
            _verify_one(av, sid, ios, ad, p)
        st = ctypes.c_int32(-7)
        iob = b"".join(pt_bytes(a) + pt_bytes(b) for a, b in ios)
        rc = lib.avrf_pedersen_verify_one(sid, 1, iob, len(ios), ad, len(ad), pt_bytes(p.pk_com), pt_bytes(p.r),
                                          pt_bytes(p.ok), bad_s.to_bytes(32, "little"), sc_bytes(p.sb), ctypes.byref(st))
        assert rc == -2 and st.value == -7
        bv = _batch(av, sid, [(ios, ad, pf), (ios, ad, p)])
        with pytest.raises(av.AvrfError):
            bv.verify_each()
    tb = av.BatchVerifier(sid)
    out = np.zeros(1, dtype=np.int32)
    assert lib.avrf_pedersen_batch_verify_each(tb._h, out.ctypes.data) == -2
    pb = ped.BatchVerifier(sid)
    assert lib.avrf_thin_batch_verify_each(pb._h, out.ctypes.data) == -2


def test_full_size(av):
    """make_pedersen_batch(0, 2^20, 1, 4096 signers): sampled proofs equal the oracle's prover, the batch verifies,
    and with s corrupted at {0, 17, n/2, n-1} the batch fails and find_invalid names exactly those."""
    from ark_vrf_b200 import pedersen as ped, synth
    sid, S = 0, o.BANDERSNATCH
    n = 1 << (20 if FULL else 14)
    b = synth.make_pedersen_batch(sid, n, 1, 4096, av.Format.CANONICAL)
    pos = {0, n - 1} | {synth.splitmix64(i) % n for i in range(62)}
    sks = {}
    for j in sorted(pos):
        k = j % 4096
        if k not in sks:
            sks[k] = o.secret_from_seed(S, k.to_bytes(8, "little") + bytes(24))
        assert int.from_bytes(bytes(b.sk[j]), "little") == sks[k]
        ios = [(pt_from_bytes(b.ios[j][:64]), pt_from_bytes(b.ios[j][64:]))]
        want, wbl = o.pedersen_prove(S, sks[k], ios, b"ad-%d" % j)
        got = o.PedersenProof(pt_from_bytes(b.pk_com[j]), pt_from_bytes(b.r[j]), pt_from_bytes(b.ok[j]),
                              int.from_bytes(bytes(b.s[j]), "little"), int.from_bytes(bytes(b.sb[j]), "little"))
        assert got == want and int.from_bytes(bytes(b.blinding[j]), "little") == wbl, j
    bv = ped.BatchVerifier(sid, av.Format.CANONICAL)
    bv.push_many(b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.pk_com, b.r, b.ok, b.s, b.sb)
    assert bv.verify_status() == 0
    bad = [0, 17, n // 2, n - 1]
    s2 = b.s.copy()
    for j in bad:
        s2[j, 0] ^= 1
    bv.clear()
    bv.push_many(b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.pk_com, b.r, b.ok, s2, b.sb)
    assert bv.verify_status() == 1
    assert list(bv.find_invalid()) == bad


def test_reserve_slices_and_invalidate(av):
    """A Pedersen handle through avrf_thin_batch_reserve (smaller than the batch), two uneven push_many slices (the
    second one longer than a k_prepare chunk of 75 776 proofs) and, after avrf_thin_batch_invalidate, the prepare of
    the resident inputs: seed, C, W and SCALARS taps bit-identical to one push_many of the whole batch, and one
    corrupted sb named by find_invalid."""
    from ark_vrf_b200 import pedersen as ped, synth
    n, k, bad = 100_000, 20_000, 77_777
    b = synth.make_pedersen_batch(0, n, 1)
    taps = (av.Tap.SEED, av.Tap.C, av.Tap.W, av.Tap.SCALARS)
    ref = ped.BatchVerifier(0, b.fmt)
    ref.push_many(b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.pk_com, b.r, b.ok, b.s, b.sb)
    assert ref.verify_status() == 0
    want = [bytes(ref.tap(t)) for t in taps]
    lib = av.load()

    def push_two(bv, sb):
        h, ao = b.io_offsets, b.ad_offsets
        bv.push_many(b.ios, h[:k + 1], b.ad_blob, ao[:k + 1], b.pk_com[:k], b.r[:k], b.ok[:k], b.s[:k], sb[:k])
        q, a = int(h[k]), int(ao[k])
        bv.push_many(b.ios[q:], (h[k:] - q).astype(np.uint32), b.ad_blob[a:], (ao[k:] - a).astype(np.uint32),
                     b.pk_com[k:], b.r[k:], b.ok[k:], b.s[k:], sb[k:])

    bv = ped.BatchVerifier(0, b.fmt)
    assert lib.avrf_thin_batch_reserve(bv._h, n // 2, n // 2, len(b.ad_blob) // 2) == 0
    push_two(bv, b.sb)
    assert bv.verify_status() == 0
    assert [bytes(bv.tap(t)) for t in taps] == want
    assert lib.avrf_thin_batch_invalidate(bv._h) == 0
    assert bv.verify_status() == 0
    assert [bytes(bv.tap(t)) for t in taps] == want
    sb2 = b.sb.copy()
    sb2[bad, 0] ^= 1
    bv.clear()
    push_two(bv, sb2)
    assert bv.verify_status() == 1
    assert list(bv.find_invalid()) == [bad]


def test_cpp_pedersen_driver(av):
    """include/avrf.hpp's ark_vrf::pedersen through a compiled driver: prove, verify, batch verify, verify_each."""
    import struct
    import subprocess
    import tempfile
    S = o.BANDERSNATCH
    cases = _fault_cases(0)[:8]
    sk = o.secret_from_seed(S, bytes(32))
    blob = struct.pack("<I", len(cases)) + sc_bytes(sk) + pt_bytes(o.public_key(S, sk))
    for ios, ad, pf in cases:
        blob += struct.pack("<I", len(ios)) + b"".join(pt_bytes(a) + pt_bytes(x) for a, x in ios)
        blob += struct.pack("<I", len(ad)) + ad
        blob += pt_bytes(pf.pk_com) + pt_bytes(pf.r) + pt_bytes(pf.ok) + sc_bytes(pf.s) + sc_bytes(pf.sb)
    root = os.path.dirname(HERE)
    with tempfile.TemporaryDirectory() as d:
        exe, data = os.path.join(d, "pedersen_driver"), os.path.join(d, "proofs.bin")
        open(data, "wb").write(blob)
        lib = os.path.join(root, "ark_vrf_b200")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"),
                               os.path.join(HERE, "cpp", "pedersen_driver.cpp"), "-o", exe,
                               "-L", lib, "-l:libavrf_gpu.so", "-Wl,-rpath," + lib])
        out = subprocess.run([exe, data], capture_output=True, text=True, timeout=300)
        print(out.stdout, out.stderr)
        assert out.returncode == 0 and "ALL OK" in out.stdout
