"""GPU: the batch server for both proof schemes and both input forms - Pedersen servers (avrf_pedersen_server_*) and
wire-format jobs (avrf_server_submit_compressed, avrf_pedersen_server_submit_compressed).  Every expected verdict comes
from a single batch handle fed the same arrays in the same process; refused decodes name the same proofs as the
handle's wire push; wire pushes on different handles run concurrently with each other and with the handle-less entry
points (their decode buffers belong to the handle)."""
import ctypes
import os
import random
import struct
import subprocess
import tempfile
import threading

import numpy as np
import pytest

from oracle import pyref as o
from helpers import pt_bytes, sc_bytes

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FULL = os.environ.get("AVRF_FULL_CONFIGS", "1") == "1"
PREP_CHUNK = 148 * 4 * 128          # proofs per decode chunk of the library (avrf_gpu.cu)
EDGES = [PREP_CHUNK - 1, PREP_CHUNK, 2 * PREP_CHUNK - 1, 2 * PREP_CHUNK]
SHAPES = [dict(workers=3, hashers=0), dict(workers=3, hashers=1), dict(workers=4, hashers=1, own_hash_workers=2)]


@pytest.fixture(scope="module")
def av():
    import ark_vrf_b200 as a
    a.load().avrf_init(0)
    return a


def _u8(b, w=None):
    a = np.frombuffer(bytes(b), dtype=np.uint8).copy()
    return a.reshape(-1, w) if w else a


def _offsets(lens):
    off = np.zeros(len(lens) + 1, dtype=np.uint32)
    off[1:] = np.cumsum(lens)
    return off


def _t2(S):
    return (0, S.p - 1)             # the point of order 2


def _no_sqrt(S, rnd):
    while True:
        e = rnd.randrange(S.p).to_bytes(32, "little")
        if o.dec_point(S, e) is None:
            return _u8(e)


def _copy(arrays):
    return tuple(np.array(x, copy=True) for x in arrays)


# ---- single-handle references --------------------------------------------------------------------------------------
def _ped_status(av, sid, fmt, dec):
    from ark_vrf_b200 import pedersen as ped
    bv = ped.BatchVerifier(sid, fmt)
    bv.push_many(*dec)
    st = bv.verify_status()
    bv.close()
    return st


def _thin_status(av, sid, fmt, dec):
    bv = av.BatchVerifier(sid, fmt)
    bv.push_many(*dec)
    st = bv.verify_status()
    bv.close()
    return st


def _ped_wire_ref(av, sid, wire):
    """-> (decode flags, status or None when refused) of one Pedersen handle's wire push"""
    from ark_vrf_b200 import pedersen as ped
    bv = ped.BatchVerifier(sid, av.Format.CANONICAL)
    ok = bv.push_compressed(*wire)
    st = bv.verify_status() if ok.all() else None
    bv.close()
    return ok, st


def _thin_wire_ref(av, sid, wire):
    bv = av.BatchVerifier(sid, av.Format.CANONICAL)
    ok = bv.push_compressed(*wire)
    st = bv.verify_status() if ok.all() else None
    bv.close()
    return ok, st


# ---- batches -------------------------------------------------------------------------------------------------------
def _ped_batch(av, sid, n, m, fmt, signers=64):
    """-> (decoded push arguments in `fmt`, wire push arguments)"""
    from ark_vrf_b200 import ops, pedersen as ped, synth
    b = synth.make_pedersen_batch(sid, n, m, signers, fmt)
    nio = int(b.io_offsets[n])
    ios32 = ops.point_compress(sid, b.ios[:nio].reshape(-1, 64), fmt).reshape(-1) if nio else np.zeros(0, np.uint8)
    wire = (np.concatenate([ios32, np.zeros(64, np.uint8)]), b.io_offsets, b.ad_blob, b.ad_offsets,
            ped.serialize_proofs(sid, b.pk_com, b.r, b.ok, b.s, b.sb, fmt))
    return (b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.pk_com, b.r, b.ok, b.s, b.sb), wire


def _thin_batch(av, sid, n, m, signers=64):
    """-> (decoded push arguments, canonical, and wire push arguments)"""
    from ark_vrf_b200 import ops, synth
    F = av.Format.CANONICAL
    b = synth.make_batch(sid, n, m, signers, F)
    nio = int(b.io_offsets[n])
    ios32 = np.concatenate([ops.point_compress(sid, b.ios[:nio].reshape(-1, 64), F).reshape(-1), np.zeros(64, np.uint8)])
    wire = (ops.point_compress(sid, b.pk, F), ios32, b.io_offsets, b.ad_blob, b.ad_offsets, ops.point_compress(sid, b.r, F), b.s)
    return (b.pk, b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.r, b.s), wire


def _ped_oracle_ragged(sid, n, m, tag):
    """Canonical decoded arrays of n oracle proofs, M_j cycling through 0..m (ragged), three signers."""
    S = o.SUITES[sid]
    sks = [o.secret_from_seed(S, o.synth_seed(k)) for k in range(3)]
    cases = []
    for j in range(n):
        sk = sks[j % 3]
        ios = []
        for i in range(j % (m + 1)):
            inp = o.data_to_point(S, b"%s-%d-%d" % (tag, j, i))
            ios.append((inp, o.pt_mul(S, inp, sk)))
        ad = b"sv-%d" % j
        cases.append((ios, ad, o.pedersen_prove(S, sk, ios, ad)[0]))
    ios = b"".join(pt_bytes(i) + pt_bytes(x) for c in cases for (i, x) in c[0])
    pfs = [c[2] for c in cases]
    return (_u8(ios + bytes(128)), _offsets([len(c[0]) for c in cases]), _u8(b"".join(c[1] for c in cases) + bytes(16)),
            _offsets([len(c[1]) for c in cases]), _u8(b"".join(pt_bytes(p.pk_com) for p in pfs), 64),
            _u8(b"".join(pt_bytes(p.r) for p in pfs), 64), _u8(b"".join(pt_bytes(p.ok) for p in pfs), 64),
            _u8(b"".join(sc_bytes(p.s) for p in pfs), 32), _u8(b"".join(sc_bytes(p.sb) for p in pfs), 32))


def _ped_variants(av, sid, fmt, dec):
    """{name: decoded arrays}: the batch and its faulty twins (one proof each, proofs with at least one pair)."""
    from ark_vrf_b200 import synth
    ios, io_off, ad, ad_off, pk_com, r, okp, s, sb = dec
    n = len(io_off) - 1
    owners = [j for j in range(n) if io_off[j + 1] > io_off[j] and ad_off[j + 1] > ad_off[j]]
    j1, j2 = owners[len(owners) // 3], owners[-1]
    ident = synth.identity_point(sid, fmt)
    out = {"valid": dec}

    def variant(name, f):
        v = list(_copy(dec))
        f(v)
        out[name] = tuple(v)
    variant("s+1", lambda v: v[7].__setitem__((j1, 0), v[7][j1, 0] ^ 1))
    variant("sb+1", lambda v: v[8].__setitem__((j2, 0), v[8][j2, 0] ^ 1))
    variant("ad", lambda v: v[2].__setitem__(int(ad_off[j1]), v[2][int(ad_off[j1])] ^ 0x20))
    variant("identity pk_com", lambda v: v[4].__setitem__(j2, ident))
    variant("identity O", lambda v: v[0].reshape(-1, 128).__setitem__((int(io_off[j1]), slice(64, 128)), ident))

    def both(v):                         # InvalidData wins over a bad scalar elsewhere
        v[4][j1] = ident
        v[7][j2, 0] ^= 1
    variant("identity + bad s", both)
    return out


# ---- 1. Pedersen decoded jobs --------------------------------------------------------------------------------------
@pytest.mark.parametrize("sid,fmt,n,m", [(0, 1, 300, 1), (0, 0, 300, 2), (1, 1, 40, 1), (2, 0, 40, 1)])
def test_pedersen_decoded_jobs(av, sid, fmt, n, m):
    """Every variant's verdict on every server shape equals a fresh handle's; waits in reverse order."""
    from ark_vrf_b200 import pedersen as ped
    dec, _ = _ped_batch(av, sid, n, m, fmt)
    variants = _ped_variants(av, sid, fmt, dec)
    want = {k: _ped_status(av, sid, fmt, v) for k, v in variants.items()}
    assert want == {"valid": 0, "s+1": 1, "sb+1": 1, "ad": 1, "identity pk_com": 2, "identity O": 2, "identity + bad s": 2}
    for shape in SHAPES:
        srv = ped.BatchServer(sid, fmt, **shape)
        tickets = [(k, srv.submit(*v)) for k, v in variants.items() for _ in range(2)]
        for k, t in reversed(tickets):
            assert srv.wait(t) == want[k], (shape, k)
        with pytest.raises(av.AvrfError):
            srv.wait(10 ** 6)            # unknown ticket
        srv.close()


def test_pedersen_ragged_and_empty(av):
    """Ragged I/O counts (0..3 pairs per proof) from the oracle's prover, and an empty job."""
    from ark_vrf_b200 import pedersen as ped
    F = av.Format.CANONICAL
    dec = _ped_oracle_ragged(0, 12, 3, b"rg")
    bad = list(_copy(dec))
    bad[8][5, 0] ^= 1
    want = [_ped_status(av, 0, F, dec), _ped_status(av, 0, F, tuple(bad))]
    assert want == [0, 1]
    srv = ped.BatchServer(0, F, workers=2)
    empty = (np.zeros(128, np.uint8), np.zeros(1, np.uint32), np.zeros(16, np.uint8), np.zeros(1, np.uint32)) + (None,) * 5
    t = [srv.submit(*dec), srv.submit(*bad), srv.submit(*empty)]
    assert [srv.wait(x) for x in t] == want + [0]
    srv.verify(srv.submit(*dec))
    with pytest.raises(av.VerificationFailure):
        srv.verify(srv.submit(*bad))
    srv.close()


def test_close_finishes_queued_jobs(av):
    """close() with jobs still queued runs them: their borrowed decode flags and counts are filled."""
    from ark_vrf_b200 import pedersen as ped
    from ark_vrf_b200.thin import ptr
    lib = av.load()
    _, wire = _ped_batch(av, 0, 5000, 1, av.Format.CANONICAL)
    ios32, io_off, ad, ad_off, proofs = wire
    bad = proofs.copy()
    bad[77, 96:128] = _u8(o.BANDERSNATCH.r.to_bytes(32, "little"))      # s = r
    n = len(io_off) - 1
    srv = ped.BatchServer(0, av.Format.CANONICAL, workers=1)
    flags = [np.full(n, 9, np.uint8) for _ in range(6)]
    counts = [ctypes.c_uint64(12345) for _ in range(6)]
    for k in range(6):
        t = lib.avrf_pedersen_server_submit_compressed(srv._h, n, ptr(ios32), ptr(io_off), ptr(ad), ptr(ad_off),
                                                        ptr(bad if k == 3 else proofs), ptr(flags[k]), ctypes.byref(counts[k]))
        assert t == k
    srv.close()
    for k in range(6):
        assert counts[k].value == (1 if k == 3 else 0), k
        assert np.nonzero(flags[k] == 0)[0].tolist() == ([77] if k == 3 else []) and (flags[k] <= 1).all()


# ---- 2. / 3. wire jobs, refusals at chunk edges ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def thin_bulk(av):
    """2 PREP_CHUNKs + 1000 Bandersnatch Thin proofs at M = 1: three decode chunks."""
    return _thin_batch(av, 0, 2 * PREP_CHUNK + 1000, 1)


@pytest.fixture(scope="module")
def ped_bulk(av):
    return _ped_batch(av, 0, 2 * PREP_CHUNK + 1000, 1, av.Format.CANONICAL)


def _n_bad_of(lib, fn, h, arrays, n):
    from ark_vrf_b200.thin import ptr
    nb = ctypes.c_uint64(99)
    t = fn(h, n, *[ptr(a) for a in arrays], None, ctypes.byref(nb))
    return t, nb


def test_thin_wire_jobs(av, thin_bulk):
    S = o.BANDERSNATCH
    rnd = random.Random(5)
    lib = av.load()
    dec, wire = thin_bulk
    n = len(wire[2]) - 1
    pk32, ios32, io_off, ad, ad_off, r32, s = wire
    s_bad = s.copy()
    s_bad[n // 2, 0] ^= 1
    dec_bad = dec[:6] + (s_bad,)
    wire_bad = wire[:6] + (s_bad,)
    assert _thin_status(av, 0, av.Format.CANONICAL, dec) == 0 and _thin_status(av, 0, av.Format.CANONICAL, dec_bad) == 1
    srv = av.BatchServer(0, av.Format.CANONICAL, workers=1)          # one worker: every job reuses its handle
    t = [srv.submit(*dec), srv.submit_compressed(*wire), srv.submit(*dec_bad), srv.submit_compressed(*wire_bad)]
    assert srv.wait(t[0]) == 0 and srv.wait_compressed(t[1])[0] == 0
    assert srv.wait(t[2]) == 1 and srv.wait_compressed(t[3])[0] == 1
    # encodings the deserialisers refuse, on both sides of each chunk edge
    pk32, ios32, r32 = pk32.copy(), ios32.copy(), r32.copy()
    v = [0] + EDGES + [n - 1]
    pk32[v[0]] = _u8(S.p.to_bytes(32, "little"))                                              # y >= p
    r32[v[1]] = _no_sqrt(S, rnd)                                                               # x with no square root
    r32[v[2]] = _u8(o.enc_point(S, o.pt_add(S, o.dec_point(S, bytes(r32[v[2]])), _t2(S))))    # R + T2
    pk32[v[3]] = _u8(o.enc_point(S, o.IDENTITY))                                               # identity pk
    ios32[64 * v[4] + 32:64 * v[4] + 64] = _u8(o.enc_point(S, o.IDENTITY))                    # identity O
    pk32[v[5]] = _u8((S.p + 3).to_bytes(32, "little"))
    refused = (pk32, ios32, io_off, ad, ad_off, r32, s)
    ok_ref, st_ref = _thin_wire_ref(av, 0, refused)
    assert st_ref is None and np.nonzero(ok_ref == 0)[0].tolist() == sorted(v)
    t = srv.submit_compressed(*refused)
    st, ok = srv.wait_compressed(t)
    assert st == 2 and (ok == ok_ref.astype(bool)).all()
    t, nb = _n_bad_of(lib, lib.avrf_server_submit_compressed, srv._h, refused, n)
    assert t >= 0 and srv.wait(t) == 2 and nb.value == len(v)
    # the worker's handle was left empty: the next job verifies normally
    st, ok = srv.wait_compressed(srv.submit_compressed(*wire))
    assert st == 0 and ok.all() and len(ok) == n
    assert srv.wait(srv.submit(*dec)) == 0
    srv.close()


def test_pedersen_wire_jobs(av, ped_bulk):
    from ark_vrf_b200 import pedersen as ped
    S = o.BANDERSNATCH
    rnd = random.Random(6)
    lib = av.load()
    dec, wire = ped_bulk
    n = len(wire[1]) - 1
    ios32, io_off, ad, ad_off, proofs = wire
    pbad = proofs.copy()
    pbad[n // 3, 96] ^= 1                                                                      # s + 1: still decodes
    assert _ped_status(av, 0, av.Format.CANONICAL, dec) == 0
    srv = ped.BatchServer(0, av.Format.CANONICAL, workers=1)
    t = [srv.submit(*dec), srv.submit_compressed(*wire), srv.submit_compressed(ios32, io_off, ad, ad_off, pbad)]
    assert srv.wait(t[0]) == 0 and srv.wait_compressed(t[1])[0] == 0
    st, ok = srv.wait_compressed(t[2])
    assert st == 1 and ok.all() and _ped_wire_ref(av, 0, (ios32, io_off, ad, ad_off, pbad))[1] == 1
    # an identity pk_com decodes (a bare point): InvalidData from verify, with every proof decoded
    pid = proofs.copy()
    pid[EDGES[1], 0:32] = _u8(o.enc_point(S, o.IDENTITY))
    t, nb = _n_bad_of(lib, lib.avrf_pedersen_server_submit_compressed, srv._h, (ios32, io_off, ad, ad_off, pid), n)
    assert srv.wait(t) == 2 and nb.value == 0
    # refused encodings on both sides of each chunk edge
    ios32, pr = ios32.copy(), proofs.copy()
    v = [0] + EDGES + [n // 2, n - 1]
    pr[v[0], 0:32] = _u8(S.p.to_bytes(32, "little"))                                           # pk_com: y >= p
    pr[v[1], 32:64] = _no_sqrt(S, rnd)                                                          # R: no square root
    pr[v[2], 32:64] = _u8(o.enc_point(S, o.pt_add(S, o.dec_point(S, bytes(pr[v[2], 32:64])), _t2(S))))   # R + T2
    ios32[64 * v[3] + 32:64 * v[3] + 64] = _u8(o.enc_point(S, o.IDENTITY))                     # identity O
    pr[v[4], 96:128] = _u8(S.r.to_bytes(32, "little"))                                          # s = r
    pr[v[5], 128:160] = _u8(b"\xff" * 32)                                                       # sb = 2^256 - 1
    pr[v[6], 64:96] = _u8(o.enc_point(S, o.pt_add(S, o.dec_point(S, bytes(pr[v[6], 64:96])), _t2(S))))   # Ok + T2
    refused = (ios32, io_off, ad, ad_off, pr)
    ok_ref, st_ref = _ped_wire_ref(av, 0, refused)
    assert st_ref is None and np.nonzero(ok_ref == 0)[0].tolist() == sorted(v)
    st, ok = srv.wait_compressed(srv.submit_compressed(*refused))
    assert st == 2 and (ok == ok_ref.astype(bool)).all()
    t, nb = _n_bad_of(lib, lib.avrf_pedersen_server_submit_compressed, srv._h, refused, n)
    assert srv.wait(t) == 2 and nb.value == len(v)
    st, ok = srv.wait_compressed(srv.submit_compressed(*wire))
    assert st == 0 and ok.all()
    srv.close()


# ---- 4. two schemes at once ----------------------------------------------------------------------------------------
def test_two_schemes_at_once(av):
    from ark_vrf_b200 import pedersen as ped
    F = av.Format.CANONICAL
    tdec, twire = _thin_batch(av, 0, 3000, 1)
    pdec, pwire = _ped_batch(av, 0, 3000, 1, F)
    ts = tdec[6].copy()
    ts[11, 0] ^= 1
    pp = pwire[4].copy()
    pp[29, 128] ^= 1                                                                           # sb + 1
    jobs = {  # name: (server kind, wire?, arrays, expected)
        "thin": ("t", False, tdec, 0), "thin bad": ("t", False, tdec[:6] + (ts,), 1),
        "thin wire": ("t", True, twire, 0), "thin wire bad": ("t", True, twire[:6] + (ts,), 1),
        "ped": ("p", False, pdec, 0), "ped wire": ("p", True, pwire, 0), "ped wire bad": ("p", True, pwire[:4] + (pp,), 1)}
    assert _thin_status(av, 0, F, jobs["thin bad"][2]) == 1 and _ped_wire_ref(av, 0, jobs["ped wire bad"][2])[1] == 1
    servers = {"t": av.BatchServer(0, F, workers=3), "p": ped.BatchServer(0, F, workers=3, hashers=1)}
    results, errors = [], []

    def client(order):
        try:
            mine = []
            for name in order:
                kind, wire, arrays, want = jobs[name]
                srv = servers[kind]
                mine.append((name, srv, wire, (srv.submit_compressed if wire else srv.submit)(*arrays)))
            for name, srv, wire, t in mine:
                st = srv.wait_compressed(t)[0] if wire else srv.wait(t)
                results.append((name, st))
        except Exception as e:                 # noqa: BLE001  (reported by the main thread)
            errors.append(e)
    names = list(jobs)
    th = [threading.Thread(target=client, args=(names * 2,)), threading.Thread(target=client, args=(names[::-1] * 2,))]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors
    assert len(results) == 4 * len(jobs)
    for name, st in results:
        assert st == jobs[name][3], name
    for s in servers.values():
        s.close()


# ---- 5. handle-owned decode buffers --------------------------------------------------------------------------------
def test_concurrent_wire_pushes_and_feeders(av, thin_bulk, ped_bulk):
    """Two handles push in wire format from two threads while a third thread hashes to the curve: every result equals
    the one the same call gives alone."""
    from ark_vrf_b200 import ops, pedersen as ped
    F = av.Format.CANONICAL
    msgs = [b"h2c-%d" % i for i in range(20000)]

    def thin_job():
        bv = av.BatchVerifier(0, F)
        ok = bv.push_compressed(*thin_bulk[1])
        out = (ok.copy(), bv.verify_status(), bytes(bv.tap(av.Tap.SEED)))
        bv.close()
        return out

    def ped_job():
        bv = ped.BatchVerifier(0, F)
        ok = bv.push_compressed(*ped_bulk[1])
        out = (ok.copy(), bv.verify_status(), bytes(bv.tap(av.Tap.SEED)))
        bv.close()
        return out

    def h2c_job():
        return [ops.hash_to_curve(0, msgs, want_compressed=True) for _ in range(4)]

    alone = [thin_job(), ped_job(), h2c_job()]
    together, errors = [None] * 3, []

    def run(k, f):
        try:
            together[k] = f()
        except Exception as e:                 # noqa: BLE001
            errors.append(e)
    th = [threading.Thread(target=run, args=(k, f)) for k, f in enumerate((thin_job, ped_job, h2c_job))]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors
    for k in (0, 1):
        assert (together[k][0] == alone[k][0]).all() and together[k][0].all()
        assert together[k][1:] == alone[k][1:] and alone[k][1] == 0
    for a, b in zip(alone[2], together[2]):
        assert len(a) == len(b) and all((x == y).all() for x, y in zip(a, b))


def test_wire_buffers_grow_after_clear(av, thin_bulk):
    """A wire push, clear, then a larger wire push (the handle's decode buffers grow) still verifies."""
    from ark_vrf_b200 import pedersen as ped
    F = av.Format.CANONICAL
    _, wire = _ped_batch(av, 2, 300, 1, F)
    big_dec, big_wire = _ped_batch(av, 2, PREP_CHUNK + 500, 2, F)
    bv = ped.BatchVerifier(2, F)
    assert bv.push_compressed(*wire).all() and bv.verify_status() == 0
    bv.clear()
    assert bv.push_compressed(*big_wire).all() and len(bv) == PREP_CHUNK + 500 and bv.verify_status() == 0
    ref = ped.BatchVerifier(2, F)
    ref.push_many(*big_dec)
    assert ref.verify_status() == 0 and bytes(ref.tap(av.Tap.SEED)) == bytes(bv.tap(av.Tap.SEED))
    _, small = _thin_batch(av, 0, 300, 1)
    tv = av.BatchVerifier(0, F)
    assert tv.push_compressed(*small).all() and tv.verify_status() == 0
    tv.clear()
    assert tv.push_compressed(*thin_bulk[1]).all() and tv.verify_status() == 0


# ---- 6. argument errors --------------------------------------------------------------------------------------------
def test_argument_errors(av):
    from ark_vrf_b200 import pedersen as ped
    from ark_vrf_b200.thin import ptr
    lib = av.load()
    F = av.Format.CANONICAL
    tdec, twire = _thin_batch(av, 0, 40, 1)
    pdec, pwire = _ped_batch(av, 0, 40, 1, F)
    n = 40
    tsrv, psrv = av.BatchServer(0, F, workers=1), ped.BatchServer(0, F, workers=1)
    P = lambda arrays: [ptr(a) for a in arrays]
    submits = {  # entry point: (its server, the other server, arguments after n)
        "avrf_server_submit": (tsrv, psrv, P(tdec)),
        "avrf_server_submit_compressed": (tsrv, psrv, P(twire) + [None, None]),
        "avrf_pedersen_server_submit": (psrv, tsrv, P(pdec)),
        "avrf_pedersen_server_submit_compressed": (psrv, tsrv, P(pwire) + [None, None])}
    required = {"avrf_server_submit": [0, 2, 4, 5, 6], "avrf_server_submit_compressed": [0, 2, 4, 5, 6],
                "avrf_pedersen_server_submit": [1, 3, 4, 5, 6, 7, 8], "avrf_pedersen_server_submit_compressed": [1, 3, 4]}
    for name, (own, other, args) in submits.items():
        fn = getattr(lib, name)
        assert fn(other._h, n, *args) == -2, name                                  # cross-scheme: no ticket
        assert b"server" in lib.avrf_last_error() and b"job on a" in lib.avrf_last_error()
        assert fn(None, n, *args) == -2
        for k in required[name]:
            a = list(args)
            a[k] = None
            assert fn(own._h, n, *a) == -2, (name, k)
        t = fn(own._h, n, *args)                                                    # ok / n_bad NULL: accepted
        assert t >= 0 and own.wait(t) == 0, name
        assert own.wait(fn(own._h, 0, *args)) == 0                                   # empty job
    # the refusals issued no ticket: the next one follows the last issued
    t = tsrv.submit(*tdec)
    assert tsrv.wait(t) == 0 and t == 4
    with pytest.raises(ValueError):
        tsrv.wait_compressed(tsrv.submit(*tdec))
    assert av.load().avrf_pedersen_server_new(0, 2, 1, 0, 0) is None             # bad format
    tsrv.close()
    psrv.close()


# ---- 7. full size --------------------------------------------------------------------------------------------------
def test_full_size_burst(av):
    """A burst of 20 Pedersen batches of 2^20 proofs (M = 1, 4096 signers); exactly the one with a corrupted s fails."""
    from ark_vrf_b200 import pedersen as ped
    F = av.Format.MONTGOMERY
    n = 1 << (20 if FULL else 14)
    dec, _ = _ped_batch(av, 0, n, 1, F, signers=4096)
    s_bad = dec[7].copy()
    s_bad[n // 2, 0] ^= 1
    bad = dec[:7] + (s_bad,) + dec[8:]
    srv = ped.BatchServer(0, F, workers=max(2, min(8, os.cpu_count() or 2)))
    tickets = [srv.submit(*(bad if k == 13 else dec)) for k in range(20)]
    got = [srv.wait(t) for t in tickets]
    srv.close()
    assert got == [1 if k == 13 else 0 for k in range(20)]


# ---- C++ -----------------------------------------------------------------------------------------------------------
def test_cpp_server_driver(av, thin_bulk):
    """include/avrf.hpp's pedersen::BatchServer and both servers' submit_compressed through a compiled C++ host."""
    F = av.Format.CANONICAL
    pdec, pwire = _ped_batch(av, 0, 2000, 1, F)
    _, twire = _thin_batch(av, 0, 2000, 1)
    blob = b""
    for a in pdec + pwire + twire:
        a = np.ascontiguousarray(a)
        blob += struct.pack("<Q", a.nbytes) + a.tobytes()
    root = os.path.dirname(HERE)
    with tempfile.TemporaryDirectory() as d:
        exe, data = os.path.join(d, "server_driver"), os.path.join(d, "jobs.bin")
        open(data, "wb").write(blob)
        lib = os.path.join(root, "ark_vrf_b200")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"),
                               os.path.join(HERE, "cpp", "server_driver.cpp"), "-o", exe,
                               "-L", lib, "-l:libavrf_gpu.so", "-Wl,-rpath," + lib, "-lpthread"])
        out = subprocess.run([exe, data], capture_output=True, text=True, timeout=600)
        print(out.stdout, out.stderr)
        assert out.returncode == 0 and "ALL OK" in out.stdout
