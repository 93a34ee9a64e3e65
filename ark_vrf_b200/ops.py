"""Feeder operations of the hot path on the GPU (include/avrf.h, "Feeder operations").

    reference (Rust)                                  here
    ------------------------------------------------  -------------------------------
    Input::new(data)            src/lib.rs:500-502    hash_to_curve(suite, msgs)
    secret.output(input)        src/lib.rs:391-393    vrf_output(suite, sk, inputs)
    Secret::from_scalar().public src/lib.rs:331-334   public_keys(suite, sk)
    secret.prove(ios, ad)       src/thin.rs:111-129   thin_prove_many(...)
    pedersen Prover::prove      src/pedersen.rs:136-186  pedersen_prove_many(...)
    point.serialize_compressed  ark-serialize         point_compress(suite, points)
    output.hash::<32>()         common.rs:290-305     point_to_hash(suite, points)

All arrays are numpy uint8 (or pinned torch CPU tensors), little-endian field elements.
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence, Tuple

import numpy as np

from . import _lib
from .thin import Format, Suite, ptr


def _blob(msgs: Sequence[bytes]) -> Tuple[np.ndarray, np.ndarray]:
    off = np.zeros(len(msgs) + 1, dtype=np.uint32)
    if len(msgs):
        off[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64).astype(np.uint32)
    blob = np.frombuffer(b"".join(msgs) + b"\0", dtype=np.uint8).copy()
    return blob, off


def hash_to_curve(suite, msgs, offsets=None, fmt=Format.CANONICAL, want_compressed=False):
    """msgs: list of bytes, or (blob uint8 array, offsets uint32 array).  Returns (n,64) points
    (and (n,32) compressed encodings if asked) plus the per-message ok flags."""
    lib = _lib.load()
    if offsets is None:
        blob, offsets = _blob(msgs)
    else:
        blob = msgs
    n = len(offsets) - 1
    aff = np.zeros((n, 64), dtype=np.uint8)
    enc = np.zeros((n, 32), dtype=np.uint8) if want_compressed else None
    ok = np.zeros(n, dtype=np.uint8)
    _lib.check(lib.avrf_hash_to_curve(int(suite), int(fmt), ptr(blob), ptr(offsets), n, ptr(aff), ptr(enc), ptr(ok)))
    return (aff, enc, ok) if want_compressed else (aff, ok)


def vrf_output(suite, sk: np.ndarray, inputs: np.ndarray, fmt=Format.CANONICAL) -> np.ndarray:
    """sk: (32,) shared or (n,32) per item; inputs (n,64)."""
    lib = _lib.load()
    n = inputs.shape[0]
    sk = np.ascontiguousarray(sk, dtype=np.uint8)
    stride = 0 if sk.ndim == 1 else 32
    out = np.zeros((n, 64), dtype=np.uint8)
    _lib.check(lib.avrf_vrf_output(int(suite), int(fmt), ptr(sk), stride, ptr(np.ascontiguousarray(inputs)), n, ptr(out)))
    return out


def vrf_io_many(suite, msgs, offsets, sk: np.ndarray, fmt=Format.CANONICAL, want_inputs=True, want_outputs=True,
                want_hashes=False, out=None):
    """Input::new + Secret::output (+ Output::hash) in one call (BASELINE.json configs[4]).  msgs/offsets as for
    hash_to_curve; sk (32,) shared or (n,32).  Returns a dict with the requested arrays (and `ok`); `out` may supply
    preallocated (e.g. pinned) arrays under the same keys."""
    lib = _lib.load()
    if offsets is None:
        msgs, offsets = _blob(msgs)
    n = len(offsets) - 1
    sk = np.ascontiguousarray(sk, dtype=np.uint8)
    stride = 0 if sk.ndim == 1 else 32
    out = dict(out or {})
    if want_inputs and "inputs" not in out:
        out["inputs"] = np.zeros((n, 64), dtype=np.uint8)
    if want_outputs and "outputs" not in out:
        out["outputs"] = np.zeros((n, 64), dtype=np.uint8)
    if want_hashes and "hashes" not in out:
        out["hashes"] = np.zeros((n, 32), dtype=np.uint8)
    if "ok" not in out:
        out["ok"] = np.zeros(n, dtype=np.uint8)
    _lib.check(lib.avrf_vrf_io_many(int(suite), int(fmt), ptr(msgs), ptr(offsets), n, ptr(sk), stride, ptr(out.get("inputs")),
                                    ptr(out.get("outputs")), ptr(out.get("hashes")), ptr(out["ok"])))
    return out


def public_keys(suite, sk: np.ndarray, fmt=Format.CANONICAL) -> np.ndarray:
    lib = _lib.load()
    sk = np.ascontiguousarray(sk, dtype=np.uint8).reshape(-1, 32)
    out = np.zeros((sk.shape[0], 64), dtype=np.uint8)
    _lib.check(lib.avrf_public_keys(int(suite), int(fmt), ptr(sk), sk.shape[0], ptr(out)))
    return out


def thin_prove_many(suite, sk, pk, ios, io_offsets, ad_blob, ad_offsets, fmt=Format.CANONICAL):
    lib = _lib.load()
    n = len(io_offsets) - 1
    r = np.zeros((n, 64), dtype=np.uint8)
    s = np.zeros((n, 32), dtype=np.uint8)
    _lib.check(lib.avrf_thin_prove_many(int(suite), int(fmt), n, ptr(sk), ptr(pk), ptr(ios), ptr(io_offsets),
                                        ptr(ad_blob), ptr(ad_offsets), ptr(r), ptr(s)))
    return r, s


def pedersen_prove_many(suite, sk, pk, ios, io_offsets, ad_blob, ad_offsets, fmt=Format.CANONICAL):
    """pedersen::Prover::prove for n proofs (arrays as for thin_prove_many).  Returns (pk_com, r, ok, s, sb, blinding):
    (n,64) points and (n,32) scalars in `fmt`; `blinding` is the factor the reference returns beside each proof."""
    lib = _lib.load()
    n = len(io_offsets) - 1
    pk_com, r, ok = (np.zeros((n, 64), dtype=np.uint8) for _ in range(3))
    s, sb, blinding = (np.zeros((n, 32), dtype=np.uint8) for _ in range(3))
    _lib.check(lib.avrf_pedersen_prove_many(int(suite), int(fmt), n, ptr(sk), ptr(pk), ptr(ios), ptr(io_offsets),
                                            ptr(ad_blob), ptr(ad_offsets), ptr(pk_com), ptr(r), ptr(ok), ptr(s), ptr(sb),
                                            ptr(blinding)))
    return pk_com, r, ok, s, sb, blinding


def point_compress(suite, points: np.ndarray, fmt=Format.CANONICAL) -> np.ndarray:
    lib = _lib.load()
    points = np.ascontiguousarray(points, dtype=np.uint8).reshape(-1, 64)
    out = np.zeros((points.shape[0], 32), dtype=np.uint8)
    _lib.check(lib.avrf_point_compress(int(suite), int(fmt), ptr(points), points.shape[0], ptr(out)))
    return out


def points_deserialize(suite, enc: np.ndarray, kind: int = 1, fmt=Format.CANONICAL):
    """Compressed 32-byte encodings -> validated affine points (reference CanonicalDeserialize with
    Validate::Yes).  kind 1 = Public/Input/Output (identity rejected), 0 = bare point (Proof.r)."""
    lib = _lib.load()
    enc = np.ascontiguousarray(enc, dtype=np.uint8).reshape(-1, 32)
    n = enc.shape[0]
    out = np.zeros((n, 64), dtype=np.uint8)
    ok = np.zeros(n, dtype=np.uint8)
    _lib.check(lib.avrf_points_deserialize(int(suite), int(fmt), kind, ptr(enc), n, ptr(out), ptr(ok)))
    return out, ok


def point_to_hash(suite, points: np.ndarray, fmt=Format.CANONICAL) -> np.ndarray:
    lib = _lib.load()
    points = np.ascontiguousarray(points, dtype=np.uint8).reshape(-1, 64)
    out = np.zeros((points.shape[0], 32), dtype=np.uint8)
    _lib.check(lib.avrf_point_to_hash(int(suite), int(fmt), ptr(points), points.shape[0], ptr(out)))
    return out


def microbench(kind: int, iters: int) -> Tuple[float, float]:
    lib = _lib.load()
    v = C.c_double(0)
    ms = C.c_float(0)
    _lib.check(lib.avrf_microbench(kind, iters, C.byref(v), C.byref(ms)))
    return v.value, ms.value
