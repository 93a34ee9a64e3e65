"""GPU: the batch MSM's exact value (csrc/msm.cuh), not only whether it is the identity.

A verdict cannot see an error that maps zero to zero and non-zero to non-zero (a sign flipped on one sort path, a
scalar factor on the whole sum, a small-order component handled wrongly).  So every case here decodes the PARTIAL tap
(the MSM sum, Montgomery extended X, Y, Z, T) and requires it to equal the C oracle's independent MSM (`corc.msm`,
signed-digit Pippenger with window ln(n) + 2) of the pushed bases, in the documented MSM order, under the SCALARS tap:
the MSM as a function of its own inputs.  Where the oracle computes the scalars too (Thin), they are compared bit for
bit.  The cases cover both sort paths (`k_scatter` below 2^18 points, `k_sort_transpose` + `k_scatter_window` from
2^18 on), Pedersen's 5N+2 points, ragged M, adversarial buckets, shard partials whose cuts split a weight block, and
batches whose R or O carry a point of order 2, 4 or 8, where the verdict depends on the exact residue of the summed
scalars."""
import hashlib
import os
import random
import time
from dataclasses import dataclass

import numpy as np
import pytest

from oracle import corc, pyref as o
from helpers import pt_bytes, pt_from_bytes, sc_bytes, torsion_points

pytestmark = pytest.mark.gpu

NT = max(1, min(os.cpu_count() or 1, 64))
LARGE = 1 << 18                        # run_msm: k_scatter_window from this many points on


@pytest.fixture(scope="module")
def av():
    import ark_vrf_b200 as a
    a.load().avrf_init(0)
    return a


def _pt(row) -> tuple:
    return pt_from_bytes(bytes(row))


def _int(row) -> int:
    return int.from_bytes(bytes(row), "little")


def _pt_arr(P) -> np.ndarray:
    return np.frombuffer(pt_bytes(P), np.uint8).copy()


def _sc_arr(k) -> np.ndarray:
    return np.frombuffer(sc_bytes(k), np.uint8).copy()


@dataclass
class Thin:
    """A Thin batch in canonical form: one row per proof, `ios` one row per pair (input || output)."""
    pk: np.ndarray
    ios: np.ndarray
    io_off: np.ndarray
    ads: list
    r: np.ndarray
    s: np.ndarray
    sk: np.ndarray = None                # the signer's secret per proof (canonical), when known

    @staticmethod
    def of(b) -> "Thin":
        ads = [bytes(b.ad_blob[b.ad_offsets[j]:b.ad_offsets[j + 1]]) for j in range(b.n)]
        nio = int(b.io_offsets[b.n])
        return Thin(b.pk.copy(), b.ios[:nio].copy(), b.io_offsets.astype(np.uint32), ads, b.r.copy(), b.s.copy(),
                    b.sk.copy())

    @property
    def n(self) -> int:
        return len(self.ads)

    @property
    def npoints(self) -> int:
        return 2 * self.n + 2 * int(self.io_off[-1]) + 1

    def arrays(self):
        """The arrays avrf_thin_batch_push_many and corc.thin_batch_verify take."""
        ad_off = np.zeros(self.n + 1, np.uint32)
        ad_off[1:] = np.cumsum([len(a) for a in self.ads], dtype=np.uint64)
        ad = np.frombuffer(b"".join(self.ads) + bytes(16), np.uint8).copy()
        ios = np.ascontiguousarray(np.concatenate([self.ios, np.zeros((1, 128), np.uint8)]))
        return (np.ascontiguousarray(self.pk), ios, self.io_off, ad, ad_off, np.ascontiguousarray(self.r),
                np.ascontiguousarray(self.s))

    def take(self, order) -> "Thin":
        order = np.asarray(order, dtype=np.int64)
        cnt = np.diff(self.io_off.astype(np.int64))[order]
        off = np.zeros(len(order) + 1, np.int64)
        off[1:] = np.cumsum(cnt)
        rows = np.repeat(self.io_off[:-1].astype(np.int64)[order] - off[:-1], cnt) + np.arange(off[-1])
        return Thin(self.pk[order], self.ios[rows], off.astype(np.uint32), [self.ads[j] for j in order],
                    self.r[order], self.s[order], None if self.sk is None else self.sk[order])

    def bases(self, S) -> np.ndarray:
        """MSM bases in thin.rs:291-317 order: per proof R, pk, (O_i, I_i)..., then G."""
        n, nio = self.n, int(self.io_off[-1])
        out = np.zeros((self.npoints, 64), np.uint8)
        j = np.arange(n, dtype=np.int64)
        pb = 2 * j + 2 * self.io_off[:-1].astype(np.int64)
        out[pb] = self.r
        out[pb + 1] = self.pk
        owner = np.repeat(j, np.diff(self.io_off.astype(np.int64)))
        pos = 2 * owner + 2 * np.arange(nio, dtype=np.int64) + 2
        out[pos] = self.ios[:, 64:]
        out[pos + 1] = self.ios[:, :64]
        out[-1] = _pt_arr(S.G)
        return out


def _partial(S, part) -> tuple:
    """The PARTIAL tap (Montgomery extended X, Y, Z, T) as a canonical affine point, checked to be one."""
    part = bytes(part)
    assert len(part) == 128
    p, rinv = S.p, pow(1 << 256, -1, S.p)
    X, Y, Z, T = [int.from_bytes(part[32 * i:32 * i + 32], "little") * rinv % p for i in range(4)]
    assert Z != 0 and T * Z % p == X * Y % p
    zi = pow(Z, -1, p)
    P = (X * zi % p, Y * zi % p)
    assert o.on_curve(S, P)
    return P


def _oracle_msm(sid, bases, scalars):
    t = time.time()
    got, ident = corc.msm(sid, bases, scalars, nthreads=NT)
    P = pt_from_bytes(got)
    assert ident == (P == o.IDENTITY)
    return P, time.time() - t


def _check_value(av, sid, bv, bases, repeat=False):
    """PARTIAL == corc.msm(bases, SCALARS tap).  With `repeat`: the same point after verify, after the SCALARS tap
    (which runs the MSM again) and after a second verify.  Points, not bytes: the order of the entries inside a bucket
    follows the counting sort's atomic ranks, so the projective representation (Z) may differ from run to run."""
    S = o.SUITES[sid]
    P = _partial(S, bv.tap(av.Tap.PARTIAL))
    sc = bv.tap(av.Tap.SCALARS).reshape(-1, 32)
    assert sc.shape[0] == bases.shape[0]
    if repeat:
        assert _partial(S, bv.tap(av.Tap.PARTIAL)) == P
        bv.verify_status()
        assert _partial(S, bv.tap(av.Tap.PARTIAL)) == P
        assert bytes(bv.tap(av.Tap.SCALARS)) == sc.tobytes()
    want, dt = _oracle_msm(sid, bases, sc)
    assert P == want
    return P, sc, dt


def _run_thin(av, sid, tb: Thin, oracle_scalars=True, repeat=False):
    """Push, verify, check PARTIAL against corc.msm and (optionally) status and SCALARS against the C batch verifier."""
    bv = av.BatchVerifier(sid, av.Format.CANONICAL)
    arrs = tb.arrays()
    bv.push_many(*arrs)
    st = bv.verify_status()
    P, sc, dt = _check_value(av, sid, bv, tb.bases(o.SUITES[sid]), repeat=repeat)
    if oracle_scalars:
        cst, _, taps = corc.thin_batch_verify(sid, *arrs, nthreads=NT, taps=True)
        assert st == cst
        assert (sc == taps["scalars"]).all()
    assert st == (0 if P == o.IDENTITY else 1)
    return bv, st, P, sc


def _flip_s(tb: Thin, rows, S):
    for j in rows:
        tb.s[j] = _sc_arr((_int(tb.s[j]) + 1) % S.r)


def _batch(av, sid, n, m=1, signers=4096):
    from ark_vrf_b200 import synth
    return Thin.of(synth.make_batch(sid, n, m, signers=signers, fmt=av.Format.CANONICAL))


# ---- (a) both sides of the k_scatter / k_scatter_window switch, (h) repeatability ------------------------------------
@pytest.mark.parametrize("sid", [0, 1, 2])
@pytest.mark.parametrize("n", [65535, 65536])
def test_thin_sort_switch(av, sid, n):
    tb = _batch(av, sid, n)
    assert (tb.npoints >= LARGE) == (n == 65536)
    S = o.SUITES[sid]
    _flip_s(tb, random.Random(n + sid).sample(range(n), n // 100), S)
    bv, st, P, _ = _run_thin(av, sid, tb, repeat=True)
    assert st == 1 and P != o.IDENTITY


# ---- (b) tiny batches: most accumulation threads exit, one crosses many bins ------------------------------------------
@pytest.mark.parametrize("sid", [0, 1, 2])
@pytest.mark.parametrize("m", [0, 1])
@pytest.mark.parametrize("n", [1, 2, 3, 7])
def test_thin_tiny(av, sid, m, n):
    tb = _batch(av, sid, n, m)
    _, st, P, _ = _run_thin(av, sid, tb)
    assert st == 0 and P == o.IDENTITY
    _flip_s(tb, [n - 1], o.SUITES[sid])
    _, st, P, _ = _run_thin(av, sid, tb, repeat=True)
    assert st == 1


# ---- (c) ragged M on the large path: point index 2j + 2 io_off[j] ------------------------------------------------------
@pytest.mark.parametrize("sid,n,mmax,ragged", [(0, 40000, 5, True), (2, 26215, 4, False)])
def test_thin_ragged_large(av, sid, n, mmax, ragged):
    from ark_vrf_b200 import ops
    tb = _batch(av, sid, n, mmax)
    if ragged:
        ms = np.random.default_rng(7).integers(0, mmax + 1, n)
        keep = np.concatenate([np.arange(mmax * j, mmax * j + ms[j]) for j in range(n)]).astype(np.int64)
        off = np.zeros(n + 1, np.uint32)
        off[1:] = np.cumsum(ms)
        tb.ios, tb.io_off = np.ascontiguousarray(tb.ios[keep]), off
        arrs = tb.arrays()
        tb.r, tb.s = ops.thin_prove_many(sid, tb.sk, arrs[0], arrs[1], arrs[2], arrs[3], arrs[4])
    assert tb.npoints >= LARGE
    _, st, P, _ = _run_thin(av, sid, tb)
    assert st == 0
    _flip_s(tb, [0, n // 3, n - 1], o.SUITES[sid])
    _, st, P, _ = _run_thin(av, sid, tb)
    assert st == 1


# ---- (d) the bench.py workload ------------------------------------------------------------------------------------------
def test_thin_bench_shape(av):
    """Bandersnatch 2^20, M = 1, the last proof's s flipped: the production shape, with the weight-carry bucket of
    about n/2 entries going through k_combine_big."""
    sid, n = 0, 1 << 20
    tb = _batch(av, sid, n)
    _flip_s(tb, [n - 1], o.SUITES[sid])
    bv = av.BatchVerifier(sid, av.Format.CANONICAL)
    bv.push_many(*tb.arrays())
    assert bv.verify_status() == 1
    P, _, dt = _check_value(av, sid, bv, tb.bases(o.SUITES[sid]))
    assert P != o.IDENTITY
    print(f"\n2^20 Bandersnatch: C oracle MSM of {tb.npoints} points took {dt:.1f} s on {NT} threads")


# ---- (e) adversarial buckets ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sid,n", [(0, 65536), (2, 65536), (1, 4096)])
def test_thin_adversarial_buckets(av, sid, n):
    """One signer and the same I/O pair on every proof (P + P in one bucket and one segment), R_j = -R_{j+1} on one
    stride (P + (-P)), R = identity on another."""
    from ark_vrf_b200 import ops
    S = o.SUITES[sid]
    tb = _batch(av, sid, n, 1, signers=1)
    tb.ios[:] = tb.ios[0]
    arrs = tb.arrays()
    tb.r, tb.s = ops.thin_prove_many(sid, tb.sk, arrs[0], arrs[1], arrs[2], arrs[3], arrs[4])
    assert (tb.pk == tb.pk[0]).all()
    _, st, P, _ = _run_thin(av, sid, tb)
    assert st == 0 and P == o.IDENTITY
    for j in range(0, n - 1, 97):
        x, y = _pt(tb.r[j + 1])
        tb.r[j] = _pt_arr(((S.p - x) % S.p, y))
    for j in range(5, n, 101):
        tb.r[j] = _pt_arr(o.IDENTITY)
    assert tb.npoints >= LARGE or n < 16384
    _, st, P, _ = _run_thin(av, sid, tb)
    assert st == 1


# ---- (f) Pedersen: 5N+2 points on both sides of the switch -------------------------------------------------------------
@pytest.mark.parametrize("sid,n", [(0, 52428), (0, 52429), (1, 52429), (2, 52428), (0, 1), (1, 3), (2, 1), (2, 3)])
def test_pedersen_value(av, sid, n):
    from ark_vrf_b200 import pedersen as ped, synth
    S = o.SUITES[sid]
    pb = synth.make_pedersen_batch(sid, n, 1, fmt=av.Format.CANONICAL)
    np_ = 5 * n + 2
    if n > 3:
        assert (np_ >= LARGE) == (n == 52429)
    bases = np.concatenate([np.stack([pb.ios[:, 64:], pb.ok, pb.ios[:, :64], pb.pk_com, pb.r], axis=1).reshape(-1, 64),
                            _pt_arr(S.G)[None], _pt_arr(S.B)[None]])

    def run(s, sb):
        bv = ped.BatchVerifier(sid, av.Format.CANONICAL)
        bv.push_many(np.ascontiguousarray(pb.ios), pb.io_offsets, pb.ad_blob, pb.ad_offsets, pb.pk_com, pb.r, pb.ok,
                     np.ascontiguousarray(s), np.ascontiguousarray(sb))
        st = bv.verify_status()
        P, sc, _ = _check_value(av, sid, bv, bases, repeat=True)
        assert st == (0 if P == o.IDENTITY else 1)
        if n <= 3:                                   # scalars against the Python oracle
            items = [o.pedersen_batch_prepare(S, [(_pt(pb.ios[j][:64]), _pt(pb.ios[j][64:]))],
                                              bytes(pb.ad_blob[pb.ad_offsets[j]:pb.ad_offsets[j + 1]]),
                                              o.PedersenProof(_pt(pb.pk_com[j]), _pt(pb.r[j]), _pt(pb.ok[j]), _int(s[j]),
                                                              _int(sb[j]))) for j in range(n)]
            _, want = o.pedersen_batch_terms(S, items)
            assert [bytes(x) for x in sc] == [sc_bytes(k) for k in want]
            assert st == o.pedersen_batch_verify(S, items)
        return st, P

    assert run(pb.s, pb.sb) == (0, o.IDENTITY)
    s, sb = pb.s.copy(), pb.sb.copy()
    s[n // 2] = _sc_arr((_int(s[n // 2]) + 1) % S.r)
    sb[n - 1] = _sc_arr((_int(sb[n - 1]) + 1) % S.r)
    st, P = run(s, sb)
    assert st == 1 and P != o.IDENTITY


# ---- (g) the same batch on a Montgomery and a canonical handle ----------------------------------------------------------
def test_formats_same_partial(av):
    """The same sum from a MONTGOMERY and a CANONICAL handle (as points: see _check_value)."""
    sid, n = 1, 65536
    S = o.SUITES[sid]
    tb = _batch(av, sid, n)
    _flip_s(tb, random.Random(3).sample(range(n), 64), S)
    arrs = tb.arrays()

    def mont(a, mod):
        a = np.ascontiguousarray(a)
        out = b"".join(((int.from_bytes(bytes(x), "little") << 256) % mod).to_bytes(32, "little") for x in a.reshape(-1, 32))
        return np.frombuffer(out, np.uint8).reshape(a.shape).copy()

    points, handles = [], []
    for fmt, conv in [(av.Format.CANONICAL, lambda a, mod: a), (av.Format.MONTGOMERY, mont)]:
        bv = av.BatchVerifier(sid, fmt)
        bv.push_many(conv(arrs[0], S.p), conv(arrs[1], S.p), arrs[2], arrs[3], arrs[4], conv(arrs[5], S.p),
                     conv(arrs[6], S.r))
        assert bv.verify_status() == 1
        points.append(_partial(S, bv.tap(av.Tap.PARTIAL)))
        handles.append(bv)
    assert points[0] == points[1] != o.IDENTITY
    P, _, _ = _check_value(av, sid, handles[0], tb.bases(S))
    assert P == points[0]


# ---- (i) shard partials cut inside a weight block -------------------------------------------------------------------------
def test_shard_partials(av):
    """avrf_thin_batch_partial(seed, first_index) at cuts that are not multiples of 4 (four proofs share one weight
    squeeze block): each partial equals corc.msm of its shard's terms under the global weights; combine_partials and
    the sum of the shard points equal the whole batch."""
    sid, n = 0, 1 << 17
    S = o.SUITES[sid]
    tb = _batch(av, sid, n)
    _flip_s(tb, random.Random(11).sample(range(n), n // 100), S)
    whole, st, Pw, scw = _run_thin(av, sid, tb, oracle_scalars=False)
    assert st == 1 and tb.npoints >= LARGE
    seed = bytes(whole.tap(av.Tap.SEED))
    cuts = [0, 43690, 87381, n]
    assert all(c % 4 for c in cuts[1:-1])
    parts, total, gsum = b"", o.IDENTITY, 0
    for lo, hi in zip(cuts, cuts[1:]):
        sh = tb.take(range(lo, hi))
        h = av.BatchVerifier(sid, av.Format.CANONICAL)
        h.push_many(*sh.arrays())
        assert h.prepare_device() is False
        part = h.partial(seed, lo)
        sc = h.tap(av.Tap.SCALARS).reshape(-1, 32)
        P = _partial(S, part)
        assert P == _oracle_msm(sid, sh.bases(S), sc)[0]
        a, b = 2 * lo + 2 * int(tb.io_off[lo]), 2 * hi + 2 * int(tb.io_off[hi])
        assert (sc[:-1] == scw[a:b]).all()          # the global weights, addressed by global index
        gsum = (gsum + _int(sc[-1])) % S.r
        parts += part
        total = o.pt_add(S, total, P)
    assert gsum == _int(scw[-1])
    assert total == Pw
    assert av.combine_partials(sid, parts) == st


# ---- small-order components in large batches ---------------------------------------------------------------------------
def _taint(S, tb: Thin, T, o_rows, r_rows, sks, rnd):
    """O taint: O' = O + T, proof re-made honestly over (I, O').  R taint: R' = R0 + T committed in the transcript,
    s = k + c'·sk.  Both with the Python oracle."""
    for j in o_rows:
        inp, out = _pt(tb.ios[j][:64]), _pt(tb.ios[j][64:])
        ios = [(inp, o.pt_add(S, out, T))]
        R, s = o.thin_prove(S, sks[j], ios, tb.ads[j])
        tb.ios[j] = np.frombuffer(pt_bytes(ios[0][0]) + pt_bytes(ios[0][1]), np.uint8)
        tb.r[j], tb.s[j] = _pt_arr(R), _sc_arr(s)
    for j in r_rows:
        pk, ios = _pt(tb.pk[j]), [(_pt(tb.ios[j][:64]), _pt(tb.ios[j][64:]))]
        t, zs = o.thin_transcript(S, pk, ios, tb.ads[j])
        im, _ = o.merged_io(S, pk, ios, zs)
        k = rnd.randrange(1, S.r)
        Rp = o.pt_add(S, o.ext_to_affine(S, o.ext_mul(S, im, k)), T)
        c = o.challenge(S, [Rp], t)
        tb.r[j], tb.s[j] = _pt_arr(Rp), _sc_arr((k + c * sks[j]) % S.r)


@pytest.mark.parametrize("sid,order", [(0, 2), (1, 2), (1, 4), (1, 8), (2, 2), (2, 4), (2, 8)])
def test_small_order_taints(av, sid, order):
    """2^16 proofs (2^18 + 1 points, the large path), some honest for O + T or committing R + T, T of order 2, 4, 8.
    The batch sees T under the O scalar w·c·z mod r and the R scalar w: the verdict depends on their exact residues mod
    ord(T).  The rotation of the batch (which changes the seed, so every weight) is chosen on the host so that one run
    has the small-order parts cancel - the batch must accept, as the reference does - and one has them not cancel.
    Each run: exact value, verdict and scalars as the oracle's; verify_each as the exact single verifier, proof by
    proof."""
    S = o.SUITES[sid]
    n = 1 << 16
    T = torsion_points(S)[order]
    rnd = random.Random(1000 * sid + order)
    tb = _batch(av, sid, n)
    rows = rnd.sample(range(n), 12)
    o_rows, r_rows = rows[:6], rows[6:]
    sks = {j: _int(tb.sk[j]) for j in rows}
    _taint(S, tb, T, o_rows, r_rows, sks, rnd)
    # c_j and z_j do not depend on the proof's position: read them once, then search rotations on the host
    bv = av.BatchVerifier(sid, av.Format.CANONICAL)
    bv.push_many(*tb.arrays())
    c = bv.tap(av.Tap.C).reshape(-1, 16)
    z = bv.tap(av.Tap.Z).reshape(-1, 16)
    cs64 = np.concatenate([c, np.zeros((n, 16), np.uint8), tb.s], axis=1)

    def residue(rot):
        seed = hashlib.sha512(S.suite_id + b"\x50" + np.roll(cs64, -rot, axis=0).tobytes()).digest()
        acc = 0
        for j in rows:
            pos = (j - rot) % n
            blk = hashlib.sha512(seed + (pos // 4).to_bytes(8, "little")).digest()
            w = int.from_bytes(blk[16 * (pos % 4):16 * (pos % 4) + 16], "little") % S.r
            acc += (w * _int(c[j]) * _int(z[j]) % S.r) if j in o_rows else w
        return acc % order

    found = {}
    for rot in range(256):
        found.setdefault(residue(rot) == 0, rot)
        if len(found) == 2:
            break
    assert set(found) == {True, False}, found
    for cancels, rot in sorted(found.items()):
        order_ = np.roll(np.arange(n), -rot)
        tr = tb.take(order_)
        bv, st, P, _ = _run_thin(av, sid, tr)
        assert st == (0 if cancels else 1)
        assert (P == o.IDENTITY) == cancels
        each = bv.verify_each()
        pos = {j: (j - rot) % n for j in rows}
        honest = np.ones(n, bool)
        honest[list(pos.values())] = False
        assert (each[honest] == 0).all()
        for j in rows:
            q = pos[j]
            pk, ios = _pt(tr.pk[q]), [(_pt(tr.ios[q][:64]), _pt(tr.ios[q][64:]))]
            R, s = _pt(tr.r[q]), _int(tr.s[q])
            want = o.thin_verify(S, pk, ios, tr.ads[q], R, s)
            assert corc.thin_verify(sid, pt_bytes(pk), pt_bytes(ios[0][0]) + pt_bytes(ios[0][1]), tr.ads[q],
                                    pt_bytes(R), sc_bytes(s)) == want
            assert each[q] == want
            if j in o_rows:
                assert want == (0 if _int(c[j]) * _int(z[j]) % order == 0 else 1)
            else:
                assert want == 1
