"""CPU: pin the C oracle (oracle/avrf_oracle.c) against the reference's golden vectors and
cross-check it with the independent Python restatement (oracle/pyref.py)."""
import numpy as np
import pytest

from oracle import corc, pyref as o
from helpers import (GOLDEN_SEEDS, arrays_from_proofs, golden_proofs, msm_py, oracle_items, point_order_2k, pt_bytes,
                     pt_from_bytes, sc_bytes, torsion_points)


@pytest.mark.parametrize("sid", [0, 1, 2])
def test_c_vectors_process(sid, golden):
    S = o.SUITES[sid]
    for v, sd in zip(golden[sid], GOLDEN_SEEDS):
        sk = corc.secret_from_seed(sid, bytes([sd]) + bytes(31))
        assert sk.hex() == v["sk"]
        pk = corc.scalar_mul(sid, sk)
        assert corc.point_compress(sid, pk).hex() == v["pk"]
        alpha, ad = bytes.fromhex(v["alpha"]), bytes.fromhex(v["ad"])
        h = corc.hash_to_curve(sid, alpha).tobytes()
        assert corc.point_compress(sid, h).hex() == v["h"]
        gamma = corc.scalar_mul(sid, sk, h)
        assert corc.point_compress(sid, gamma).hex() == v["gamma"]
        assert corc.point_to_hash(sid, gamma).hex() == v["beta"]
        r, s = corc.thin_prove(sid, sk, h + gamma, ad)
        assert corc.point_compress(sid, r).hex() == v["proof_r"]
        assert s.hex() == v["proof_s"]
        assert corc.thin_verify(sid, pk, h + gamma, ad, r, s) == 0
        assert corc.thin_verify(sid, pk, h + gamma, ad + b"x", r, s) == 1


@pytest.mark.parametrize("sid", [0, 1, 2])
@pytest.mark.parametrize("threads", [1, 4])
def test_c_batch_vs_python(sid, threads, golden):
    S = o.SUITES[sid]
    pr = golden_proofs(S, golden[sid])
    items = oracle_items(pr)
    st, _, taps = corc.thin_batch_verify(sid, *arrays_from_proofs(pr), nthreads=threads, taps=True)
    assert st == 0
    assert [bytes(x) for x in taps["c"]] == [e.c.to_bytes(16, "little") for e in items]
    assert [bytes(x) for x in taps["z"]] == [e.zs[1].to_bytes(16, "little") for e in items]
    seed = o.batch_seed(S, items)
    assert taps["seed"].tobytes() == seed
    assert [bytes(x) for x in taps["w"]] == [w.to_bytes(16, "little") for w in o.batch_weights(S, seed, 7)]
    _, scalars = o.batch_msm_terms(S, items)
    assert [bytes(x) for x in taps["scalars"]] == [sc_bytes(k) for k in scalars]
    pr.s[2] = (pr.s[2] + 1) % S.r
    assert corc.thin_batch_verify(sid, *arrays_from_proofs(pr), nthreads=threads)[0] == 1
    pr.pk[4] = o.IDENTITY
    assert corc.thin_batch_verify(sid, *arrays_from_proofs(pr), nthreads=threads)[0] == 2


@pytest.mark.parametrize("sid,m,n", [(0, 1, 40), (0, 3, 12), (0, 0, 9), (1, 1, 33), (2, 4, 10)])
def test_c_random_batches(sid, m, n):
    S = o.SUITES[sid]
    pr = o.synth_proofs(S, n, m, signers=3)
    arrs = arrays_from_proofs(pr)
    st, _, taps = corc.thin_batch_verify(sid, *arrs, nthreads=2, taps=True)
    items = oracle_items(pr)
    assert st == 0 == o.batch_verify(S, items)
    _, scalars = o.batch_msm_terms(S, items)
    assert [bytes(x) for x in taps["scalars"]] == [sc_bytes(k) for k in scalars]
    # C prover agrees with the Python prover
    sk = o.secret_from_seed(S, o.synth_seed(1 % 3))
    iob = b"".join(pt_bytes(a) + pt_bytes(b) for a, b in pr.ios[1])
    r, s = corc.thin_prove(sid, sc_bytes(sk), iob, pr.ad[1])
    assert r == pt_bytes(pr.r[1]) and s == sc_bytes(pr.s[1])
    assert corc.thin_verify(sid, pt_bytes(pr.pk[1]), iob, pr.ad[1], r, s) == 0
    pr.ad[n - 1] += b"?"
    assert corc.thin_batch_verify(sid, *arrays_from_proofs(pr), nthreads=2)[0] == 1


@pytest.mark.parametrize("sid", [0, 1, 2])
def test_c_msm_vs_python(sid):
    """orc_msm (the oracle's signed-digit Pippenger, exported) against sum k_i * P_i by plain double-and-add, before any
    GPU MSM is compared with it: repeated bases, P with -P, the identity, small-order bases and their sums with
    subgroup points, scalars 0, r - 1, r, 2^256 - 1 and every 16-bit chunk 0x8000 / 0x7fff (the signed-digit carry edge),
    none of them reduced mod r."""
    import random
    S = o.SUITES[sid]
    rnd = random.Random(0x5EED + sid)
    tors = torsion_points(S)
    assert set(tors) == ({2} if sid == 0 else {2, 4, 8})
    for k, T in tors.items():
        assert o.on_curve(S, T) and point_order_2k(S, T) == k
    sub = [o.pt_mul(S, S.G, rnd.randrange(1, S.r)) for _ in range(4)]
    mixed = [o.pt_add(S, sub[i % 4], T) for i, T in enumerate(tors.values())]
    pool = sub + [o.pt_neg(S, sub[0]), o.IDENTITY, S.G] + list(tors.values()) + mixed
    edge = [0, 1, 2, S.r - 1, S.r, S.r + 1, int("8000" * 16, 16), int("7fff" * 16, 16), (1 << 256) - 1,
            int("8000" * 15 + "7fff", 16), 1 << 255]
    cases = [([], []), ([sub[0]], [edge[3]]), ([tors[2]], [edge[8]]), ([o.IDENTITY], [edge[6]]),
             ([sub[1], sub[1]], [edge[6], edge[7]]), ([sub[2], o.pt_neg(S, sub[2])], [edge[8], edge[8]]),
             ([mixed[-1], tors[max(tors)]], [S.r, edge[9]])]
    for P in pool:                                      # every base alone under every edge scalar
        cases += [([P] * len(edge), edge)]
    for _ in range(4):                                  # n = 37: everything at once
        bases = [rnd.choice(pool) for _ in range(37)]
        scalars = [rnd.choice(edge) if rnd.random() < 0.5 else rnd.getrandbits(256) for _ in range(37)]
        cases.append((bases, scalars))
    for j, (bases, scalars) in enumerate(cases):
        want = msm_py(S, bases, scalars)
        b = np.frombuffer(b"".join(pt_bytes(P) for P in bases), np.uint8)
        k = np.frombuffer(b"".join(sc_bytes(x) for x in scalars), np.uint8)
        for threads in (1, 4):
            got, ident = corc.msm(sid, b, k, nthreads=threads)
            assert pt_from_bytes(got) == want, (j, threads)
            assert ident == (want == o.IDENTITY)
    # the small-order component follows the integer scalar, not its residue mod r
    T = tors[max(tors)]
    assert corc.msm(sid, np.frombuffer(pt_bytes(T), np.uint8), np.frombuffer(sc_bytes(S.r), np.uint8))[1] is False
    assert corc.msm(sid, np.frombuffer(pt_bytes(T), np.uint8), np.frombuffer(sc_bytes(S.r * max(tors)), np.uint8))[1]


def test_c_ragged_batch():
    """Ragged M_j and ad lengths in one batch: C oracle == Python oracle (seed, scalars, verdict)."""
    import random
    S = o.BANDERSNATCH
    rnd = random.Random(5)
    sk = o.secret_from_seed(S, bytes(32))
    pr = o.Proofs(S)
    for j, (m, al) in enumerate(zip([0, 1, 3, 2, 5, 1], [0, 1, 127, 128, 129, 300])):
        ios = []
        for i in range(m):
            inp = o.data_to_point(S, o.synth_msg(j, i))
            ios.append((inp, o.pt_mul(S, inp, sk)))
        ad = bytes(rnd.randrange(256) for _ in range(al))
        R, s = o.thin_prove(S, sk, ios, ad)
        pr.pk.append(o.public_key(S, sk)); pr.ios.append(ios); pr.ad.append(ad); pr.r.append(R); pr.s.append(s)
    items = oracle_items(pr)
    st, _, taps = corc.thin_batch_verify(0, *arrays_from_proofs(pr), nthreads=2, taps=True)
    assert st == 0 == o.batch_verify(S, items)
    assert taps["seed"].tobytes() == o.batch_seed(S, items)
    _, scalars = o.batch_msm_terms(S, items)
    assert [bytes(x) for x in taps["scalars"]] == [sc_bytes(k) for k in scalars]
