"""GPU: Pedersen VRF proofs pushed in wire format (avrf_pedersen_batch_push_compressed): decoded and validated on the
device, against the reference's golden vectors, the decoded push (avrf_pedersen_batch_push_many) and the oracle's
deserialiser."""
import ctypes
import json
import os
import random
import struct

import numpy as np
import pytest

from oracle import pyref as o
from helpers import pt_bytes, pt_from_bytes, sc_bytes

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FULL = os.environ.get("AVRF_FULL_CONFIGS", "1") == "1"
PREP_CHUNK = 148 * 4 * 128          # proofs per decode chunk of the library (avrf_gpu.cu)


@pytest.fixture(scope="module")
def av():
    import ark_vrf_b200 as a
    a.load().avrf_init(0)
    return a


def _u8(b, w=None):
    a = np.frombuffer(bytes(b), dtype=np.uint8).copy()
    return a.reshape(-1, w) if w else a


def _t2(S):
    return (0, S.p - 1)             # the point of order 2


def _offsets(lens):
    off = np.zeros(len(lens) + 1, dtype=np.uint32)
    off[1:] = np.cumsum(lens)
    return off


# ---- oracle cases [(ios, ad, PedersenProof)] -> the arrays of both pushes -----------------------------------------
def _wire(S, cases):
    """-> (ios32, io_offsets, ad_blob, ad_offsets, proofs (n, 160))"""
    recs = b"".join(o.enc_point(S, p.pk_com) + o.enc_point(S, p.r) + o.enc_point(S, p.ok) + sc_bytes(p.s) + sc_bytes(p.sb)
                    for _, _, p in cases)
    ios32 = b"".join(o.enc_point(S, i) + o.enc_point(S, x) for c in cases for (i, x) in c[0])
    return (_u8(ios32 + bytes(64)), _offsets([len(c[0]) for c in cases]), _u8(b"".join(c[1] for c in cases) + bytes(16)),
            _offsets([len(c[1]) for c in cases]), _u8(recs, 160))


def _decoded(S, cases):
    """-> the canonical arguments of BatchVerifier.push_many"""
    ios = b"".join(pt_bytes(i) + pt_bytes(x) for c in cases for (i, x) in c[0])
    pfs = [c[2] for c in cases]
    return (_u8(ios + bytes(128)), _offsets([len(c[0]) for c in cases]), _u8(b"".join(c[1] for c in cases) + bytes(16)),
            _offsets([len(c[1]) for c in cases]), _u8(b"".join(pt_bytes(p.pk_com) for p in pfs), 64),
            _u8(b"".join(pt_bytes(p.r) for p in pfs), 64), _u8(b"".join(pt_bytes(p.ok) for p in pfs), 64),
            _u8(b"".join(sc_bytes(p.s) for p in pfs), 32), _u8(b"".join(sc_bytes(p.sb) for p in pfs), 32))


def _oracle_cases(sid, n, m, tag):
    """n proofs by the oracle's prover, M_j cycling through 0..m, three signers."""
    S = o.SUITES[sid]
    sks = [o.secret_from_seed(S, o.synth_seed(k)) for k in range(3)]
    cases = []
    for j in range(n):
        sk = sks[j % 3]
        ios = []
        for i in range(j % (m + 1)):
            inp = o.data_to_point(S, b"%s-%d-%d" % (tag, j, i))
            ios.append((inp, o.pt_mul(S, inp, sk)))
        ad = b"pw-%d" % j
        cases.append((ios, ad, o.pedersen_prove(S, sk, ios, ad)[0]))
    return cases


def _gpu_batch(av, sid, n, m, signers=64):
    """make_pedersen_batch (canonical) -> (decoded push arguments, wire push arguments)"""
    from ark_vrf_b200 import ops, pedersen as ped, synth
    F = av.Format.CANONICAL
    b = synth.make_pedersen_batch(sid, n, m, signers, F)
    nio = int(b.io_offsets[n])
    ios32 = ops.point_compress(sid, b.ios[:nio].reshape(-1, 64), F).reshape(-1) if nio else np.zeros(0, np.uint8)
    wire = (np.concatenate([ios32, np.zeros(64, np.uint8)]), b.io_offsets, b.ad_blob, b.ad_offsets,
            ped.serialize_proofs(sid, b.pk_com, b.r, b.ok, b.s, b.sb, F))
    dec = (b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.pk_com, b.r, b.ok, b.s, b.sb)
    return dec, wire


@pytest.fixture(scope="module")
def bulk(av):
    """200 000 Bandersnatch proofs at M = 1: three decode chunks."""
    return _gpu_batch(av, 0, 200000, 1)


def _ped(av, sid, fmt=None, eager=True):
    from ark_vrf_b200 import pedersen as ped
    bv = ped.BatchVerifier(sid, av.Format.CANONICAL if fmt is None else fmt)
    if not eager:
        assert av.load().avrf_thin_batch_set_eager(bv._h, 0) == 0
    return bv


def _copy(wire):
    return tuple(np.array(x, copy=True) for x in wire)


# ---- 1. golden vectors ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sid", [0, 1, 2])
def test_golden_vectors(av, sid):
    """The reference's published proofs, taken as the hex strings they are (proof_pk_com | proof_r | proof_ok |
    proof_s | proof_sb, with h | gamma as the pair): accepted, verified, and challenges / seed / weights / MSM scalars
    bit-identical to the same proofs pushed decoded - on handles of either in-memory format."""
    S = o.SUITES[sid]
    with open(os.path.join(HERE, "golden", f"{S.name}_pedersen.json")) as f:
        vs = json.load(f)
    n = len(vs)
    h = lambda v, k: bytes.fromhex(v[k])
    proofs = _u8(b"".join(h(v, "proof_pk_com") + h(v, "proof_r") + h(v, "proof_ok") + h(v, "proof_s") + h(v, "proof_sb")
                          for v in vs), 160)
    ios32 = _u8(b"".join(h(v, "h") + h(v, "gamma") for v in vs))
    ads = [h(v, "ad") for v in vs]
    io_off, ad_off, ad = np.arange(n + 1, dtype=np.uint32), _offsets([len(a) for a in ads]), _u8(b"".join(ads) + bytes(16))
    cases = [([(o.dec_point(S, h(v, "h")), o.dec_point(S, h(v, "gamma")))], h(v, "ad"),
              o.PedersenProof(o.dec_point(S, h(v, "proof_pk_com")), o.dec_point(S, h(v, "proof_r")),
                              o.dec_point(S, h(v, "proof_ok")), int.from_bytes(h(v, "proof_s"), "little"),
                              int.from_bytes(h(v, "proof_sb"), "little"))) for v in vs]
    assert _wire(S, cases)[4].tobytes() == proofs.tobytes()
    ref = _ped(av, sid)
    ref.push_many(*_decoded(S, cases))
    assert ref.verify_status() == 0
    for fmt in (av.Format.CANONICAL, av.Format.MONTGOMERY):
        bv = _ped(av, sid, fmt)
        ok = bv.push_compressed(ios32, io_off, ad, ad_off, proofs)
        assert ok.all() and len(bv) == n
        assert bv.verify_status() == 0
        assert list(bv.verify_each()) == [0] * n
        for tap in (av.Tap.C, av.Tap.SEED, av.Tap.W, av.Tap.SCALARS):
            assert (bv.tap(tap) == ref.tap(tap)).all(), (sid, fmt, tap)


def test_serialize_proofs_formats(av):
    """serialize_proofs: the same records from canonical and Montgomery prover output, equal to the oracle's
    encodings of the proofs."""
    from ark_vrf_b200 import pedersen as ped, synth
    for sid in (0, 1, 2):
        S = o.SUITES[sid]
        recs = []
        for fmt in (av.Format.CANONICAL, av.Format.MONTGOMERY):
            b = synth.make_pedersen_batch(sid, 40, 2, 8, fmt)
            recs.append(ped.serialize_proofs(sid, b.pk_com, b.r, b.ok, b.s, b.sb, fmt))
            if fmt == av.Format.CANONICAL:
                for j in (0, 17, 39):
                    want = b"".join(o.enc_point(S, pt_from_bytes(x[j])) for x in (b.pk_com, b.r, b.ok)) + bytes(b.s[j]) + bytes(b.sb[j])
                    assert recs[0][j].tobytes() == want
        assert recs[0].shape == (40, 160) and (recs[0] == recs[1]).all()


# ---- 2. bulk and ragged --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sid,m,n", [(0, 1, 200000), (2, 3, 24), (1, 0, 24), (0, 4, 24)])
def test_bulk_and_ragged(av, bulk, sid, m, n):
    """Same seed, weights and verdict as the decoded push; a second wire push appends."""
    if n == 200000:
        dec, wire = bulk
    else:
        S = o.SUITES[sid]
        cases = _oracle_cases(sid, n, m, b"rg")
        dec, wire = _decoded(S, cases), _wire(S, cases)
    ref = _ped(av, sid)
    ref.push_many(*dec)
    assert ref.verify_status() == 0
    bv = _ped(av, sid, av.Format.MONTGOMERY)
    ok = bv.push_compressed(*wire)
    assert ok.all() and len(bv) == n
    assert bv.verify_status() == 0
    assert bytes(bv.tap(av.Tap.SEED)) == bytes(ref.tap(av.Tap.SEED))
    assert (bv.tap(av.Tap.W) == ref.tap(av.Tap.W)).all()
    ok = bv.push_compressed(*wire)
    assert ok.all() and len(bv) == 2 * n and bv.verify_status() == 0
    ref.push_many(*dec)
    assert ref.verify_status() == 0
    assert bytes(bv.tap(av.Tap.SEED)) == bytes(ref.tap(av.Tap.SEED))


# ---- 3. refusals ---------------------------------------------------------------------------------------------------
def _flags_oracle(S, wire, j):
    """Proof j of a wire push decodes under the reference's deserialisers (and its scalars are canonical)."""
    ios32, io_off, _, _, proofs = wire
    rec = bytes(proofs[j])
    good = all(o.deserialize_point(S, rec[32 * k:32 * k + 32], False) is not None for k in range(3))
    good = good and int.from_bytes(rec[96:128], "little") < S.r and int.from_bytes(rec[128:160], "little") < S.r
    for i in range(2 * int(io_off[j]), 2 * int(io_off[j + 1])):
        good = good and o.deserialize_point(S, bytes(ios32[32 * i:32 * i + 32]), True) is not None
    return good


def _corrupt(S, wire, victims, rnd):
    """Each victim gets one fault, in this order: pk_com with y >= p, R with no square root, Ok + T2, R + T2, an
    identity input, an output (0, -1), s = r, sb = 2^256 - 1."""
    ios32, io_off, ad, ad_off, proofs = _copy(wire)
    while True:
        e = rnd.randrange(S.p).to_bytes(32, "little")
        if o.dec_point(S, e) is None:
            break
    faults = [
        lambda j: proofs[j].__setitem__(slice(0, 32), _u8(S.p.to_bytes(32, "little"))),
        lambda j: proofs[j].__setitem__(slice(32, 64), _u8(e)),
        lambda j: proofs[j].__setitem__(slice(64, 96), _u8(o.enc_point(S, o.pt_add(S, o.dec_point(S, bytes(proofs[j][64:96])), _t2(S))))),
        lambda j: proofs[j].__setitem__(slice(32, 64), _u8(o.enc_point(S, o.pt_add(S, o.dec_point(S, bytes(proofs[j][32:64])), _t2(S))))),
        lambda j: ios32.__setitem__(slice(64 * int(io_off[j]), 64 * int(io_off[j]) + 32), _u8(o.enc_point(S, o.IDENTITY))),
        lambda j: ios32.__setitem__(slice(64 * int(io_off[j]) + 32, 64 * int(io_off[j]) + 64), _u8(o.enc_point(S, _t2(S)))),
        lambda j: proofs[j].__setitem__(slice(96, 128), _u8(S.r.to_bytes(32, "little"))),
        lambda j: proofs[j].__setitem__(slice(128, 160), _u8(b"\xff" * 32)),
    ]
    for j, f in zip(victims, faults):
        f(j)
    return ios32, io_off, ad, ad_off, proofs


def test_refusals(av, bulk):
    """Encodings the reference's deserialisers refuse - among them the cofactor-tainted Ok + T2 and R + T2, which
    push_many accepts and verification then fails - are named in ok[] and push nothing; the flags agree with the
    oracle; a handle that already holds the batch keeps its proofs and seed and takes a later good push."""
    S = o.BANDERSNATCH
    rnd = random.Random(7)
    dec, wire = bulk
    n = len(wire[1]) - 1
    victims = [0, PREP_CHUNK - 1, PREP_CHUNK, n - 1] + rnd.sample(range(1, n - 1), 4)
    assert len(set(victims)) == 8
    bad = _corrupt(S, wire, victims, rnd)
    fresh = _ped(av, 0)
    ok = fresh.push_compressed(*bad)
    assert sorted(np.nonzero(ok == 0)[0].tolist()) == sorted(victims)
    assert len(fresh) == 0 and av.load().avrf_thin_batch_len(fresh._h) == 0
    for j in sorted(set(victims) | set(rnd.sample(range(n), 40))):
        assert bool(ok[j]) == _flags_oracle(S, bad, j), j
    # a handle that already holds the batch
    held = _ped(av, 0, av.Format.MONTGOMERY)
    assert held.push_compressed(*wire).all() and held.verify_status() == 0
    seed = bytes(held.tap(av.Tap.SEED))
    ok = held.push_compressed(*bad)
    assert sorted(np.nonzero(ok == 0)[0].tolist()) == sorted(victims)
    assert len(held) == n and av.load().avrf_thin_batch_len(held._h) == n
    assert held.verify_status() == 0 and bytes(held.tap(av.Tap.SEED)) == seed
    # after the rollback the handle is no longer hashed eagerly: this push copies the decoded proofs from the device
    assert held.push_compressed(*wire).all() and len(held) == 2 * n
    assert held.verify_status() == 0
    ref = _ped(av, 0)
    ref.push_many(*dec)
    ref.push_many(*dec)
    assert ref.verify_status() == 0
    assert bytes(held.tap(av.Tap.SEED)) == bytes(ref.tap(av.Tap.SEED))
    assert (held.tap(av.Tap.W) == ref.tap(av.Tap.W)).all()


@pytest.mark.parametrize("sid", [1, 2])
def test_refusals_small(av, sid):
    """The same faults on the other suites, one decode chunk, ragged I/O counts."""
    S = o.SUITES[sid]
    rnd = random.Random(20 + sid)
    cases = _oracle_cases(sid, 24, 2, b"rf")
    wire = _wire(S, cases)
    io_off = wire[1]
    owners = [j for j in range(24) if io_off[j + 1] > io_off[j]]
    order = list(range(24))
    rnd.shuffle(order)
    victims = []
    for k in range(8):                  # the I/O faults (4, 5) need a proof with pairs
        victims.append(next(j for j in (owners if k in (4, 5) else order) if j not in victims))
    bad = _corrupt(S, wire, victims, rnd)
    bv = _ped(av, sid, av.Format.MONTGOMERY)
    ok = bv.push_compressed(*bad)
    assert sorted(np.nonzero(ok == 0)[0].tolist()) == sorted(victims) and len(bv) == 0
    for j in range(24):
        assert bool(ok[j]) == _flags_oracle(S, bad, j), j
    assert bv.push_compressed(*wire).all() and len(bv) == 24 and bv.verify_status() == 0


# ---- 4. decodes, then verify decides -------------------------------------------------------------------------------
def test_identity_pk_com_and_r(av):
    """pk_com and R are bare points: an identity decodes.  verify then gives InvalidData for the pk_com (verify_each 2)
    and VerificationFailure for the R (verify_each 1)."""
    S = o.BANDERSNATCH
    cases = _oracle_cases(0, 8, 1, b"id")
    wire = _wire(S, cases)
    for field, j, want in ((0, 3, 2), (32, 5, 1)):
        w = _copy(wire)
        w[4][j, field:field + 32] = _u8(o.enc_point(S, o.IDENTITY))
        bv = _ped(av, 0)
        assert bv.push_compressed(*w).all() and len(bv) == 8
        assert bv.verify_status() == want
        assert list(bv.verify_each()) == [want if i == j else 0 for i in range(8)]


# ---- 5. non-eager handle -------------------------------------------------------------------------------------------
def test_non_eager_handle(av, bulk):
    _, wire = bulk
    n = len(wire[1]) - 1
    eager = _ped(av, 0)
    assert eager.push_compressed(*wire).all() and eager.verify_status() == 0
    for fmt in (av.Format.CANONICAL, av.Format.MONTGOMERY):
        lazy = _ped(av, 0, fmt, eager=False)
        assert lazy.push_compressed(*wire).all() and len(lazy) == n
        assert lazy.verify_status() == 0
        assert bytes(lazy.tap(av.Tap.SEED)) == bytes(eager.tap(av.Tap.SEED))
    # a refused push on a non-eager handle that holds proofs
    bad = _copy(wire)
    bad[4][n - 1, 96:128] = _u8(o.BANDERSNATCH.r.to_bytes(32, "little"))
    ok = lazy.push_compressed(*bad)
    assert np.nonzero(ok == 0)[0].tolist() == [n - 1] and len(lazy) == n
    assert lazy.verify_status() == 0 and bytes(lazy.tap(av.Tap.SEED)) == bytes(eager.tap(av.Tap.SEED))


# ---- 6. argument errors --------------------------------------------------------------------------------------------
def test_argument_errors(av):
    from ark_vrf_b200.thin import ptr
    S = o.BANDERSNATCH
    lib = av.load()
    cases = _oracle_cases(0, 6, 2, b"ae")
    ios32, io_off, ad, ad_off, proofs = _wire(S, cases)
    n = len(cases)
    held = _ped(av, 0)
    assert held.push_compressed(ios32, io_off, ad, ad_off, proofs).all()
    assert held.verify_status() == 0
    seed = bytes(held.tap(av.Tap.SEED))
    thin = av.BatchVerifier(0)
    nb = ctypes.c_uint64(77)

    def call(h, n, io, ao, pr):
        return lib.avrf_pedersen_batch_push_compressed(h, n, ptr(ios32), ptr(io), ptr(ad), ptr(ao), pr, None,
                                                       ctypes.byref(nb))
    assert call(thin._h, n, io_off, ad_off, ptr(proofs)) == -2
    assert len(thin) == 0 and lib.avrf_thin_batch_len(thin._h) == 0
    assert call(held._h, n, io_off, ad_off, None) == -2
    assert call(held._h, n, io_off + 1, ad_off, ptr(proofs)) == -2
    assert call(held._h, n, io_off, ad_off + 1, ptr(proofs)) == -2
    assert call(None, n, io_off, ad_off, ptr(proofs)) == -2
    assert call(held._h, 0, io_off, ad_off, ptr(proofs)) == 0 and nb.value == 0          # n == 0: a no-op
    assert lib.avrf_thin_batch_len(held._h) == n
    assert held.verify_status() == 0 and bytes(held.tap(av.Tap.SEED)) == seed


# ---- 7. full size --------------------------------------------------------------------------------------------------
def test_full_size(av):
    """2^20 Bandersnatch proofs, M = 1, 4096 signers: the serialised batch verifies; with four corrupted encodings the
    call names exactly those four and pushes nothing."""
    S = o.BANDERSNATCH
    n = 1 << (20 if FULL else 14)
    _, wire = _gpu_batch(av, 0, n, 1, 4096)
    bv = _ped(av, 0)
    assert bv.push_compressed(*wire).all() and len(bv) == n
    assert bv.verify_status() == 0
    ios32, io_off, ad, ad_off, proofs = _copy(wire)
    victims = [0, 17, n // 2, n - 1]
    proofs[0, 0:32] = _u8((S.p + 5).to_bytes(32, "little"))                                     # pk_com: y >= p
    proofs[17, 32:64] = _u8(o.enc_point(S, o.pt_add(S, o.dec_point(S, bytes(proofs[17, 32:64])), _t2(S))))   # R + T2
    ios32[64 * (n // 2) + 32:64 * (n // 2) + 64] = _u8(o.enc_point(S, o.IDENTITY))             # identity output
    proofs[n - 1, 128:160] = _u8(S.r.to_bytes(32, "little"))                                     # sb = r
    fresh = _ped(av, 0)
    ok = fresh.push_compressed(ios32, io_off, ad, ad_off, proofs)
    assert np.nonzero(ok == 0)[0].tolist() == victims
    assert len(fresh) == 0 and av.load().avrf_thin_batch_len(fresh._h) == 0


# ---- 8. C++ --------------------------------------------------------------------------------------------------------
def test_cpp_driver(av):
    """include/avrf.hpp's pedersen::BatchVerifier::push_compressed through a compiled driver."""
    import subprocess
    import tempfile
    S = o.BANDERSNATCH
    cases = _oracle_cases(0, 12, 2, b"cpp")
    ios32, io_off, ad, ad_off, proofs = _wire(S, cases)
    n, nio, nad = len(cases), int(io_off[-1]), int(ad_off[-1])
    blob = struct.pack("<III", n, nio, nad) + proofs.tobytes() + ios32[:64 * nio].tobytes() + io_off.tobytes()
    blob += ad_off.tobytes() + ad[:nad].tobytes()
    root = os.path.dirname(HERE)
    with tempfile.TemporaryDirectory() as d:
        exe, data = os.path.join(d, "pedersen_wire_driver"), os.path.join(d, "wire.bin")
        open(data, "wb").write(blob)
        lib = os.path.join(root, "ark_vrf_b200")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"),
                               os.path.join(HERE, "cpp", "pedersen_wire_driver.cpp"), "-o", exe,
                               "-L", lib, "-l:libavrf_gpu.so", "-Wl,-rpath," + lib])
        out = subprocess.run([exe, data], capture_output=True, text=True, timeout=300)
        print(out.stdout, out.stderr)
        assert out.returncode == 0 and "ALL OK" in out.stdout
