"""Shared helpers for the parity tests: oracle <-> byte-array conversions."""
import numpy as np

from oracle import pyref as o

GOLDEN_SEEDS = [1, 2, 3, 4, 5, 5, 6]           # reference src/testing.rs:291-299


def pt_bytes(P) -> bytes:
    return P[0].to_bytes(32, "little") + P[1].to_bytes(32, "little")


def pt_from_bytes(b) -> tuple:
    b = bytes(b)
    return (int.from_bytes(b[:32], "little"), int.from_bytes(b[32:64], "little"))


def sc_bytes(k: int) -> bytes:
    return int(k).to_bytes(32, "little")


def to_mont_bytes(b: bytes, mod: int) -> bytes:
    return ((int.from_bytes(b, "little") << 256) % mod).to_bytes(32, "little")


def arrays_from_proofs(pr: "o.Proofs", montgomery: bool = False):
    """Oracle Proofs -> the arrays avrf_thin_batch_push_many takes (canonical or Montgomery)."""
    S = pr.suite
    n = len(pr.pk)

    def fp(x):
        return ((x << 256) % S.p if montgomery else x).to_bytes(32, "little")

    def fr(x):
        return ((x << 256) % S.r if montgomery else x).to_bytes(32, "little")

    def pb(P):
        return fp(P[0]) + fp(P[1])

    pk = np.frombuffer(b"".join(pb(P) for P in pr.pk), dtype=np.uint8).reshape(n, 64).copy()
    r = np.frombuffer(b"".join(pb(P) for P in pr.r), dtype=np.uint8).reshape(n, 64).copy()
    s = np.frombuffer(b"".join(fr(x) for x in pr.s), dtype=np.uint8).reshape(n, 32).copy()
    iob = b"".join(pb(i) + pb(oo) for ios in pr.ios for (i, oo) in ios)
    ios = np.frombuffer(iob + bytes(128), dtype=np.uint8).copy()
    io_off = np.zeros(n + 1, dtype=np.uint32)
    io_off[1:] = np.cumsum([len(x) for x in pr.ios])
    ad_off = np.zeros(n + 1, dtype=np.uint32)
    ad_off[1:] = np.cumsum([len(a) for a in pr.ad])
    ad = np.frombuffer(b"".join(pr.ad) + bytes(16), dtype=np.uint8).copy()
    return pk, ios, io_off, ad, ad_off, r, s


def oracle_items(pr: "o.Proofs"):
    return [o.batch_prepare(pr.suite, pr.pk[j], pr.ios[j], pr.ad[j], pr.r[j], pr.s[j]) for j in range(len(pr.pk))]


def point_order_2k(S, T) -> int:
    """Order of a point of the 2-power torsion (1, 2, 4, 8 or 16)."""
    k = 1
    while T != o.IDENTITY:
        assert k < 16, "not a small-order point"
        T, k = o.pt_add(S, T, T), 2 * k
    return k


def torsion_points(S) -> dict:
    """{order: point} for the affine points of order 2, 4 and 8 the suite has: a curve point outside the prime-order
    subgroup (x solved from the curve equation at some y) multiplied by r, doubled down to each order.  With `a` a
    non-square (Bandersnatch) the other points of order 2 lie at infinity and nothing halves (0, -1): only T2 exists."""
    out = {2: (0, S.p - 1)}
    if pow(S.a, (S.p - 1) // 2, S.p) != 1:
        return out
    want = {d for d in (2, 4, 8) if S.cofactor % d == 0}
    for y in range(2, 200):
        P = o.x_from_y(S, y, False)
        if P is None:
            continue
        T = o.pt_mul_raw(S, P, S.r)
        k = point_order_2k(S, T)
        while k >= 2:
            out.setdefault(k, T)
            T, k = o.pt_add(S, T, T), k // 2
        if want <= set(out):
            break
    return out


def msm_py(S, bases, scalars):
    """sum k_i * P_i by scalar multiplication without any reduction of k_i (pyref.pt_mul_raw)."""
    acc = o.IDENTITY
    for P, k in zip(bases, scalars):
        acc = o.pt_add(S, acc, o.pt_mul_raw(S, P, k))
    return acc


def golden_proofs(S, vectors) -> "o.Proofs":
    pr = o.Proofs(S)
    for v in vectors:
        pk = o.dec_point(S, bytes.fromhex(v["pk"]))
        h = o.dec_point(S, bytes.fromhex(v["h"]))
        gamma = o.dec_point(S, bytes.fromhex(v["gamma"]))
        pr.pk.append(pk)
        pr.ios.append([(h, gamma)])
        pr.ad.append(bytes.fromhex(v["ad"]))
        pr.r.append(o.dec_point(S, bytes.fromhex(v["proof_r"])))
        pr.s.append(int.from_bytes(bytes.fromhex(v["proof_s"]), "little"))
    return pr
