"""ctypes binding of the C oracle (oracle/avrf_oracle.c -> oracle/liboracle.so).

TEST INFRASTRUCTURE / CPU BASELINE ONLY - see the header of avrf_oracle.c."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path):
            import subprocess
            subprocess.check_call(["make", "-s", "-C", _HERE])
        L = C.CDLL(path)
        L.orc_hash_to_curve.restype = C.c_int
        L.orc_hash_to_curve.argtypes = [C.c_int, C.c_char_p, C.c_size_t, C.c_void_p]
        L.orc_point_compress.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.orc_scalar_mul.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_secret_from_seed.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.orc_point_to_hash.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.orc_thin_prove.restype = C.c_int
        L.orc_thin_prove.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_char_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.orc_thin_verify.restype = C.c_int
        L.orc_thin_verify.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_char_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.orc_thin_batch_verify.restype = C.c_int
        L.orc_thin_batch_verify.argtypes = [C.c_int, C.c_size_t] + [C.c_void_p] * 7 + [C.c_int, C.c_void_p] + [C.c_void_p] * 5
        L.orc_msm.restype = C.c_int
        L.orc_msm.argtypes = [C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.orc_synth_batch.restype = C.c_int
        L.orc_synth_batch.argtypes = [C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data


def hash_to_curve(sid: int, msg: bytes):
    out = np.zeros(64, np.uint8)
    ok = lib().orc_hash_to_curve(sid, msg, len(msg), _p(out))
    return out if ok else None


def point_compress(sid: int, p64) -> bytes:
    a = np.frombuffer(bytes(p64), np.uint8).copy(); out = np.zeros(32, np.uint8)
    lib().orc_point_compress(sid, _p(a), _p(out)); return out.tobytes()


def scalar_mul(sid: int, k32: bytes, p64=None) -> bytes:
    k = np.frombuffer(bytes(k32), np.uint8).copy(); out = np.zeros(64, np.uint8)
    a = None if p64 is None else np.frombuffer(bytes(p64), np.uint8).copy()
    lib().orc_scalar_mul(sid, _p(k), _p(a), _p(out)); return out.tobytes()


def secret_from_seed(sid: int, seed: bytes) -> bytes:
    s = np.frombuffer(bytes(seed), np.uint8).copy(); out = np.zeros(32, np.uint8)
    lib().orc_secret_from_seed(sid, _p(s), _p(out)); return out.tobytes()


def point_to_hash(sid: int, p64) -> bytes:
    a = np.frombuffer(bytes(p64), np.uint8).copy(); out = np.zeros(32, np.uint8)
    lib().orc_point_to_hash(sid, _p(a), _p(out)); return out.tobytes()


def thin_prove(sid: int, sk32: bytes, ios: bytes, ad: bytes):
    k = np.frombuffer(bytes(sk32), np.uint8).copy()
    io = np.frombuffer(bytes(ios) + bytes(128), np.uint8).copy()
    r = np.zeros(64, np.uint8); s = np.zeros(32, np.uint8)
    rc = lib().orc_thin_prove(sid, _p(k), _p(io), len(ios) // 128, ad, len(ad), _p(r), _p(s))
    assert rc == 0
    return r.tobytes(), s.tobytes()


def thin_verify(sid: int, pk64, ios: bytes, ad: bytes, r64, s32) -> int:
    pk = np.frombuffer(bytes(pk64), np.uint8).copy(); io = np.frombuffer(bytes(ios) + bytes(128), np.uint8).copy()
    r = np.frombuffer(bytes(r64), np.uint8).copy(); s = np.frombuffer(bytes(s32), np.uint8).copy()
    return lib().orc_thin_verify(sid, _p(pk), _p(io), len(ios) // 128, ad, len(ad), _p(r), _p(s))


def thin_batch_verify(sid: int, pk, ios, io_off, ad, ad_off, r, s, nthreads=1, taps=False):
    """Arrays as for avrf_thin_batch_push_many (canonical).  Returns (status, (prepare_s, verify_s), taps dict)."""
    n = len(io_off) - 1
    nio = int(io_off[n]) if n else 0
    times = np.zeros(2, np.float64)
    t = {}
    if taps:
        t = dict(c=np.zeros((n, 16), np.uint8), z=np.zeros((max(nio, 1), 16), np.uint8), seed=np.zeros(64, np.uint8),
                 w=np.zeros((n, 16), np.uint8), scalars=np.zeros((2 * n + 2 * nio + 1, 32), np.uint8))
    args = [np.ascontiguousarray(x) for x in (pk, ios, io_off, ad, ad_off, r, s)]
    st = lib().orc_thin_batch_verify(sid, n, *[_p(a) for a in args], nthreads, _p(times),
                                     _p(t.get("c")), _p(t.get("z")), _p(t.get("seed")), _p(t.get("w")), _p(t.get("scalars")))
    if taps:
        t["z"] = t["z"][:nio]
    return st, (float(times[0]), float(times[1])), t


def msm(sid: int, bases, scalars, nthreads: int = 1):
    """sum_i k_i * P_i by the oracle's MSM (the one its batch verifier runs).  bases: (n, 64) canonical affine points,
    scalars: (n, 32) canonical little-endian integers below 2^256, not reduced mod r.  Returns (sum as 64 canonical
    bytes, is_identity)."""
    b = np.ascontiguousarray(np.asarray(bases, dtype=np.uint8).reshape(-1, 64))
    k = np.ascontiguousarray(np.asarray(scalars, dtype=np.uint8).reshape(-1, 32))
    assert b.shape[0] == k.shape[0]
    out = np.zeros(64, np.uint8)
    rc = lib().orc_msm(sid, b.shape[0], _p(b), _p(k), nthreads, _p(out))
    assert rc in (0, 1)
    return out.tobytes(), bool(rc)


def synth_batch(sid: int, n: int, m: int = 1, signers: int = 4096, first: int = 0, nthreads: int = 1):
    """The synthetic set of SURVEY.md 8(d) generated by the oracle's own prover (canonical arrays,
    same layout as avrf_thin_batch_push_many)."""
    pk = np.zeros((n, 64), np.uint8); ios = np.zeros((n * m + 1, 128), np.uint8)
    r = np.zeros((n, 64), np.uint8); s = np.zeros((n, 32), np.uint8)
    rc = lib().orc_synth_batch(sid, first, n, m, min(signers, max(n, 1)) if signers else 1, nthreads, _p(pk), _p(ios), _p(r), _p(s))
    assert rc == 0
    ads = [b"ad-%d" % (first + j) for j in range(n)]
    ad_off = np.zeros(n + 1, np.uint32)
    if n:
        ad_off[1:] = np.cumsum([len(a) for a in ads])
    ad = np.frombuffer(b"".join(ads) + bytes(16), np.uint8).copy()
    io_off = (np.arange(n + 1, dtype=np.uint64) * m).astype(np.uint32)
    return pk, ios, io_off, ad, ad_off, r, s
