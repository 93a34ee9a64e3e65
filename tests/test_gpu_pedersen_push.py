"""GPU: Pedersen VRF single pushes (avrf_pedersen_batch_push, pedersen.BatchVerifier.push): staged in pinned memory and
shipped in chunks like the Thin verifier's, compared with one push_many of the same arrays on a fresh handle through the
SEED, C, W and SCALARS taps and the verdict; and the handle controls pedersen.BatchVerifier shares with
thin.BatchVerifier."""
import json
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import pyref as o
from helpers import pt_bytes, sc_bytes, to_mont_bytes

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PREP_CHUNK = 148 * 4 * 128          # proofs per k_prepare launch (avrf_gpu.cu)
STAGE_CHUNK = PREP_CHUNK // 2       # proofs per shipment of staged single pushes
TAPS = ("SEED", "C", "W", "SCALARS")


@pytest.fixture(scope="module")
def av():
    import ark_vrf_b200 as a
    a.load().avrf_init(0)
    return a


def _offsets(lens):
    off = np.zeros(len(lens) + 1, dtype=np.uint32)
    off[1:] = np.cumsum(lens)
    return off


def _proven(sid, fmt, m, ad_lens, signers=64):
    """Proofs by the GPU prover: proof j has m[j] I/O pairs and ad_lens[j] bytes of ad (both may be ragged).
    -> the arguments of push_many: ios, io_offsets, ad_blob, ad_offsets, pk_com, r, ok, s, sb."""
    from ark_vrf_b200 import ops, synth
    n, mmax = len(m), max(1, int(max(m)))
    sk, pk, ios, _, _, _ = synth._inputs(synth.Suite(sid), n, mmax, signers, fmt, 0)
    m = np.asarray(m)
    rows = ((np.arange(n) * mmax)[:, None] + np.arange(mmax)[None, :])[np.arange(mmax)[None, :] < m[:, None]]
    ios = np.ascontiguousarray(np.concatenate([ios[rows], np.zeros((1, 128), np.uint8)]))
    io_off, ad_off = _offsets(m), _offsets(ad_lens)
    ad = np.random.default_rng(n).integers(0, 256, int(ad_off[-1]) + 16, dtype=np.uint8)
    return (ios, io_off, ad, ad_off) + tuple(ops.pedersen_prove_many(sid, sk, pk, ios, io_off, ad, ad_off, fmt)[:5])


def _ragged(sid, fmt, n):
    """M cycling 1, 2, 3; ad of 0 to 40 bytes, empty for every seventh proof."""
    return _proven(sid, fmt, [1 + j % 3 for j in range(n)], [0 if j % 7 == 0 else (5 * j) % 41 for j in range(n)])


def _slice(arrs, lo, hi):
    """Proofs [lo, hi) of push_many arguments, offsets rebased to 0."""
    ios, io_off, ad, ad_off, *cols = arrs
    q0, q1, a0, a1 = int(io_off[lo]), int(io_off[hi]), int(ad_off[lo]), int(ad_off[hi])
    return (np.ascontiguousarray(np.concatenate([ios[q0:q1], np.zeros((1, 128), np.uint8)])),
            (io_off[lo:hi + 1] - q0).astype(np.uint32), np.ascontiguousarray(np.concatenate([ad[a0:a1], np.zeros(16, np.uint8)])),
            (ad_off[lo:hi + 1] - a0).astype(np.uint32)) + tuple(np.ascontiguousarray(c[lo:hi]) for c in cols)


def _concat(parts):
    ios = np.concatenate([p[0][:int(p[1][-1])] for p in parts] + [np.zeros((1, 128), np.uint8)])
    ad = np.concatenate([p[2][:int(p[3][-1])] for p in parts] + [np.zeros(16, np.uint8)])
    io_off = _offsets(np.concatenate([np.diff(p[1]) for p in parts]))
    ad_off = _offsets(np.concatenate([np.diff(p[3]) for p in parts]))
    return (ios, io_off, ad, ad_off) + tuple(np.concatenate([p[k] for p in parts]) for k in range(4, 9))


def _singles(av, h, arrs, lo=0, hi=None):
    """avrf_pedersen_batch_push for proofs [lo, hi)."""
    ios, io_off, ad, ad_off, pk_com, r, ok, s, sb = arrs
    push = av.load().avrf_pedersen_batch_push
    base = [x.ctypes.data for x in (ios, ad, pk_com, r, ok, s, sb)]
    hi = len(io_off) - 1 if hi is None else hi
    for j in range(lo, hi):
        q0, q1, a0, a1 = int(io_off[j]), int(io_off[j + 1]), int(ad_off[j]), int(ad_off[j + 1])
        rc = push(h, base[0] + 128 * q0 if q1 > q0 else None, q1 - q0, base[1] + a0 if a1 > a0 else None, a1 - a0,
                  base[2] + 64 * j, base[3] + 64 * j, base[4] + 64 * j, base[5] + 32 * j, base[6] + 32 * j)
        assert rc == 0, av.load().avrf_last_error()


def _ped(av, sid, fmt):
    from ark_vrf_b200 import pedersen as ped
    return ped.BatchVerifier(sid, fmt)


def _assert_same(av, bv, ref, status=0):
    """Same verdict as the reference handle, and the same SEED, C, W and SCALARS taps."""
    assert len(bv) == len(ref)
    assert bv.verify_status() == status
    assert ref.verify_status() == status
    for t in TAPS:
        assert (bv.tap(av.Tap[t]) == ref.tap(av.Tap[t])).all(), t


def _reference(av, sid, fmt, arrs):
    ref = _ped(av, sid, fmt)
    ref.push_many(*arrs)
    return ref


def _wire(sid, fmt, arrs):
    from ark_vrf_b200 import ops, pedersen as ped
    ios, io_off, ad, ad_off, pk_com, r, ok, s, sb = arrs
    nio = int(io_off[-1])
    ios32 = ops.point_compress(sid, ios[:nio].reshape(-1, 64), fmt).reshape(-1)
    return (np.concatenate([ios32, np.zeros(64, np.uint8)]), io_off, ad, ad_off,
            ped.serialize_proofs(sid, pk_com, r, ok, s, sb, fmt))


# ---- golden vectors ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sid", [0, 1, 2])
def test_golden_vectors_one_by_one(av, sid):
    """The reference's published proofs pushed one by one through pedersen.BatchVerifier.push, on handles of both
    formats: Ok, the oracle's batch seed, and the taps of one push_many."""
    from ark_vrf_b200 import pedersen as ped
    S = o.SUITES[sid]
    with open(os.path.join(HERE, "golden", f"{S.name}_pedersen.json")) as f:
        vs = json.load(f)
    h = lambda v, k: bytes.fromhex(v[k])
    cases = [([(o.dec_point(S, h(v, "h")), o.dec_point(S, h(v, "gamma")))], h(v, "ad"),
              o.PedersenProof(o.dec_point(S, h(v, "proof_pk_com")), o.dec_point(S, h(v, "proof_r")),
                              o.dec_point(S, h(v, "proof_ok")), int.from_bytes(h(v, "proof_s"), "little"),
                              int.from_bytes(h(v, "proof_sb"), "little"))) for v in vs]
    seed = o.pedersen_batch_seed(S, [o.pedersen_batch_prepare(S, ios, ad, pf) for ios, ad, pf in cases])
    for fmt in (av.Format.CANONICAL, av.Format.MONTGOMERY):
        mont = fmt == av.Format.MONTGOMERY
        pb = lambda P: (to_mont_bytes(pt_bytes(P)[:32], S.p) + to_mont_bytes(pt_bytes(P)[32:], S.p)) if mont else pt_bytes(P)
        sc = lambda k: to_mont_bytes(sc_bytes(k), S.r) if mont else sc_bytes(k)
        bv = _ped(av, sid, fmt)
        for ios, ad, pf in cases:
            bv.push([(pb(i), pb(x)) for i, x in ios], ad, ped.Proof(pb(pf.pk_com), pb(pf.r), pb(pf.ok), sc(pf.s), sc(pf.sb)))
        assert len(bv) == len(cases)
        u8 = lambda b, w: np.frombuffer(b, dtype=np.uint8).reshape(-1, w).copy()
        arrs = (u8(b"".join(pb(i) + pb(x) for c in cases for i, x in c[0]) + bytes(128), 128),
                _offsets([len(c[0]) for c in cases]), u8(b"".join(c[1] for c in cases) + bytes(16), 1).reshape(-1),
                _offsets([len(c[1]) for c in cases])) + tuple(
            u8(b"".join(f(getattr(c[2], k)) for c in cases), w)
            for k, f, w in (("pk_com", pb, 64), ("r", pb, 64), ("ok", pb, 64), ("s", sc, 32), ("sb", sc, 32)))
        _assert_same(av, bv, _reference(av, sid, fmt, arrs))
        assert bytes(bv.tap(av.Tap.SEED)) == seed


# ---- bulk, ragged, staging reuse and growth ------------------------------------------------------------------------
def test_ragged_bulk_and_reuse(av):
    """160 000 proofs (more than two PREP_CHUNKs), M from 1 to 3, ad from empty to 40 bytes: identical taps; then clear
    and the same again on the same handle, which reuses its staging buffers."""
    F = av.Format.MONTGOMERY
    n = 160000
    arrs = _ragged(0, F, n)
    ref = _reference(av, 0, F, arrs)
    bv = _ped(av, 0, F)
    for _ in range(2):
        _singles(av, bv._h, arrs)
        assert len(bv) == n                     # staged proofs count
        _assert_same(av, bv, ref)
        bv.clear()
        assert len(bv) == 0


def test_staging_room_grows(av):
    """Proofs at M = 8 fill the first staging buffer's I/O room (2 x PREP_CHUNK pairs) before it holds STAGE_CHUNK
    proofs, and one proof carries more ad than the whole first buffer's room (16 x PREP_CHUNK bytes): the room grows,
    keeping what is staged, and the taps are still identical."""
    F = av.Format.CANONICAL
    n = 24000
    ad_lens = [80] * n
    ad_lens[20000] = 16 * PREP_CHUNK + 4321
    arrs = _proven(0, F, [8] * n, ad_lens, signers=16)
    bv = _ped(av, 0, F)
    _singles(av, bv._h, arrs)
    _assert_same(av, bv, _reference(av, 0, F, arrs))


# ---- interleavings -------------------------------------------------------------------------------------------------
def test_interleaved_pushes(av):
    """push_many, singles, push_compressed, singles: the batch of one push_many of the concatenation."""
    F = av.Format.CANONICAL
    arrs = _ragged(2, F, 4000)
    cut = [0, 700, 1900, 3100, 4000]
    parts = [_slice(arrs, cut[k], cut[k + 1]) for k in range(4)]
    bv = _ped(av, 2, F)
    bv.push_many(*parts[0])
    _singles(av, bv._h, parts[1])
    assert bv.push_compressed(*_wire(2, F, parts[2])).all()
    _singles(av, bv._h, parts[3])
    assert len(bv) == 4000
    _assert_same(av, bv, _reference(av, 2, F, _concat(parts)))


def test_refused_wire_push_keeps_staged_proofs(av):
    """A refused push_compressed between single pushes: the staged proofs survive it, len is right, and the seed is
    that of the batch without the refused proofs."""
    F = av.Format.CANONICAL
    arrs = _ragged(0, F, 3000)
    parts = [_slice(arrs, 0, 1000), _slice(arrs, 1000, 2000), _slice(arrs, 2000, 3000)]
    bad = _wire(0, F, parts[1])
    bad[4][500, 96:128] = np.frombuffer(o.BANDERSNATCH.r.to_bytes(32, "little"), dtype=np.uint8)     # s = r
    bv = _ped(av, 0, F)
    _singles(av, bv._h, parts[0])
    ok = bv.push_compressed(*bad)
    assert np.nonzero(ok == 0)[0].tolist() == [500]
    assert len(bv) == 1000
    _singles(av, bv._h, parts[2])
    assert len(bv) == 2000
    _assert_same(av, bv, _reference(av, 0, F, _concat([parts[0], parts[2]])))


# ---- rejections ----------------------------------------------------------------------------------------------------
def test_tampered_proofs(av):
    """A tampered s, and separately sb, at STAGE_CHUNK - 1, STAGE_CHUNK and the last proof: verdict 1, find_invalid
    names exactly that proof, and the taps equal push_many of the same tampered arrays."""
    F = av.Format.MONTGOMERY
    n = STAGE_CHUNK + 1500
    arrs = _ragged(0, F, n)
    bv = _ped(av, 0, F)
    for col in (7, 8):                          # s, sb
        for j in (STAGE_CHUNK - 1, STAGE_CHUNK, n - 1):
            bad = arrs[col].copy()
            bad[j, 0] ^= 1
            tampered = arrs[:col] + (bad,) + arrs[col + 1:]
            bv.clear()
            _singles(av, bv._h, tampered)
            _assert_same(av, bv, _reference(av, 0, F, tampered), status=1)
            assert bv.find_invalid().tolist() == [j], (col, j)


def test_identity_pk_com(av):
    """A single push whose pk_com is the identity: InvalidData, as pedersen::Verifier::verify reports it."""
    from ark_vrf_b200 import synth
    F = av.Format.CANONICAL
    arrs = _ragged(1, F, 40)
    pk_com = arrs[4].copy()
    pk_com[13] = synth.identity_point(1, F)
    arrs = arrs[:4] + (pk_com,) + arrs[5:]
    bv = _ped(av, 1, F)
    _singles(av, bv._h, arrs)
    _assert_same(av, bv, _reference(av, 1, F, arrs), status=2)
    assert bv.find_invalid().tolist() == [13]


# ---- handle state --------------------------------------------------------------------------------------------------
def test_non_eager_handle(av):
    """set_eager(0): single pushes wait in host memory until prepare; the same seed and taps."""
    lib = av.load()
    F = av.Format.CANONICAL
    arrs = _ragged(0, F, 5000)
    bv = _ped(av, 0, F)
    assert lib.avrf_thin_batch_set_eager(bv._h, 0) == 0
    _singles(av, bv._h, arrs)
    assert len(bv) == 5000
    _assert_same(av, bv, _reference(av, 0, F, arrs))


def test_set_eager_with_pending_pushes(av):
    lib = av.load()
    F = av.Format.CANONICAL
    arrs = _ragged(0, F, 3)
    bv = _ped(av, 0, F)
    _singles(av, bv._h, arrs, 0, 1)
    assert lib.avrf_thin_batch_set_eager(bv._h, 0) == -5
    assert b"pending" in lib.avrf_last_error()
    _singles(av, bv._h, arrs, 1, 3)
    _assert_same(av, bv, _reference(av, 0, F, arrs))


def test_push_completes_verify_in_flight(av):
    """verify_async in flight, then single pushes: the push completes the verify first (verify_wait then finds none
    in flight), and the next verify covers both parts - for a good first part and for one with a bad proof."""
    from ark_vrf_b200 import _lib
    F = av.Format.CANONICAL
    arrs = _ragged(0, F, 3000)
    first, second = _slice(arrs, 0, 2000), _slice(arrs, 2000, 3000)
    s_bad = first[7].copy()
    s_bad[77, 0] ^= 1
    for a, want in ((first, 0), (first[:7] + (s_bad,) + first[8:], 1)):
        bv = _ped(av, 0, F)
        bv.push_many(*a)
        bv.verify_async()
        _singles(av, bv._h, second)
        with pytest.raises(_lib.AvrfError, match="no verify in flight"):
            bv.verify_wait()
        _assert_same(av, bv, _reference(av, 0, F, _concat([a, second])), status=want)
        if want:
            assert bv.find_invalid().tolist() == [77]


def test_argument_errors(av):
    """Null pointers, a Thin handle, a Pedersen handle for avrf_thin_batch_push: AVRF_ERR_ARG with nothing pushed; a
    proof without I/O pairs or ad may pass null for both."""
    lib = av.load()
    F = av.Format.CANONICAL
    arrs = _proven(0, F, [0, 1], [0, 3])
    ios, io_off, ad, ad_off, pk_com, r, ok, s, sb = arrs
    bv = _ped(av, 0, F)
    cols = [x[1].ctypes.data for x in (pk_com, r, ok, s, sb)]
    io1, ad1 = ios.ctypes.data, ad.ctypes.data
    push = lib.avrf_pedersen_batch_push
    assert push(None, io1, 1, ad1, 3, *cols) == -2
    for k in range(5):
        assert push(bv._h, io1, 1, ad1, 3, *(cols[:k] + [None] + cols[k + 1:])) == -2
    assert push(bv._h, None, 1, ad1, 3, *cols) == -2
    assert push(bv._h, io1, 1, None, 3, *cols) == -2
    thin = av.BatchVerifier(0, F)
    assert push(thin._h, io1, 1, ad1, 3, *cols) == -2
    assert b"not a Pedersen batch" in lib.avrf_last_error()
    assert lib.avrf_thin_batch_push(bv._h, pk_com[1].ctypes.data, io1, 1, ad1, 3, r[1].ctypes.data, s[1].ctypes.data) == -2
    assert len(thin) == 0 and len(bv) == 0
    assert push(bv._h, None, 0, None, 0, *[x[0].ctypes.data for x in (pk_com, r, ok, s, sb)]) == 0
    assert push(bv._h, io1, 1, ad1, 3, *cols) == 0
    assert len(bv) == 2
    _assert_same(av, bv, _reference(av, 0, F, arrs))


def test_python_handle_controls(av):
    """The controls pedersen.BatchVerifier shares with thin.BatchVerifier, on a Pedersen handle: the same seed and
    verdict as the plain calls."""
    from ark_vrf_b200 import pedersen as ped, thin
    F = av.Format.CANONICAL
    arrs = _ragged(0, F, 6000)
    bad = arrs[7].copy()
    bad[4321, 0] ^= 1
    ref = _reference(av, 0, F, arrs)
    assert ref.verify_status() == 0
    seed = bytes(ref.tap(av.Tap.SEED))
    items = [(arrs[0][int(arrs[1][j]):int(arrs[1][j + 1])].tobytes(), arrs[2][int(arrs[3][j]):int(arrs[3][j + 1])].tobytes(),
              ped.Proof(*(bytes(arrs[k][j]) for k in range(4, 9)))) for j in range(6000)]
    bv = ped.BatchVerifier(0, F)
    bv.reserve(6000, int(arrs[1][-1]), int(arrs[3][-1]))
    pool = thin.HashPool(2)
    bv.set_hash_pool(pool)
    bv.set_blocking(True)
    for ios, ad, pf in items:
        bv.push(ios, ad, pf)
    assert len(bv) == 6000
    bv.verify_async()
    assert bv.verify_wait() == 0
    assert bytes(bv.tap(av.Tap.SEED)) == seed
    t = bv.timings()
    assert t["n_points"] == 5 * 6000 + 2 and t["total_ms"] > 0
    assert isinstance(bv.stream, int) and bv.stream != 0
    bv.invalidate()
    bv.verify()                                  # prepare again on the resident inputs
    assert bytes(bv.tap(av.Tap.SEED)) == seed
    bv.set_hash_pool(None)
    bv.set_blocking(False)
    bv.clear()
    for j, (ios, ad, pf) in enumerate(items):
        bv.push_prepared(ped.BatchVerifier.prepare(ios, ad, pf if j != 4321 else ped.Proof(pf.pk_com, pf.r, pf.ok,
                                                                                          bytes(bad[j]), pf.sb)))
    bv.verify_async()
    assert bv.verify_wait() == 1
    with pytest.raises(thin.VerificationFailure):
        bv.verify()
    assert bv.find_invalid().tolist() == [4321]
    bv.close()
    pool.close()


# ---- C++ -----------------------------------------------------------------------------------------------------------
def test_cpp_push_driver(av):
    """include/avrf.hpp's pedersen::BatchVerifier::push for 2^17 proofs through a compiled driver: the verdict and
    seed of push_many, and a tampered proof rejected."""
    F = av.Format.CANONICAL
    n = 1 << 17
    arrs = _ragged(0, F, n)
    ios, io_off, ad, ad_off, *cols = arrs
    blob = struct.pack("<I", n) + b"".join(np.ascontiguousarray(c).tobytes() for c in cols) + io_off.tobytes()
    blob += ad_off.tobytes() + ios[:int(io_off[-1])].tobytes() + ad[:int(ad_off[-1])].tobytes()
    root = os.path.dirname(HERE)
    with tempfile.TemporaryDirectory() as d:
        exe, data = os.path.join(d, "pedersen_push_driver"), os.path.join(d, "proofs.bin")
        open(data, "wb").write(blob)
        lib = os.path.join(root, "ark_vrf_b200")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(root, "include"),
                               os.path.join(HERE, "cpp", "pedersen_push_driver.cpp"), "-o", exe,
                               "-L", lib, "-l:libavrf_gpu.so", "-Wl,-rpath," + lib])
        out = subprocess.run([exe, data], capture_output=True, text=True, timeout=600)
        print(out.stdout, out.stderr)
        assert out.returncode == 0 and "ALL OK" in out.stdout
