"""Pedersen VRF on the GPU (SURVEY.md 8f-3): proving, single and batch verification.

Mirror of `ark_vrf::pedersen` (reference src/pedersen.rs):
    Prover::prove                    prove_many(...)             (pedersen.rs:136-186, n proofs per call)
    Verifier::verify                 verify(suite, ios, ad, proof)  (pedersen.rs:188-253, exact)
    BatchVerifier::{new, push, push_prepared, verify}   BatchVerifier  (pedersen.rs:322-427; the MSM has 5N+2 points)
    (wire-format proofs)             BatchVerifier.push_compressed(), serialize_proofs()  (Proof::{de,}serialize_compressed)
    (per-proof verdicts)             BatchVerifier.verify_each() / find_invalid()
A proof is `(pk_com, r, ok, s, sb)` (pedersen.rs:43-50)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Union

import numpy as np

from . import _lib
from .ops import pedersen_prove_many as prove_many          # noqa: F401  (re-exported: pedersen.prove_many)
from .ops import point_compress
from .synth import ORDER
from .thin import Format, Suite, Tap, _bytes_of, _ios_bytes, _raise_for_status, ptr


@dataclass
class Proof:                              # pedersen::Proof (src/pedersen.rs:43-50)
    pk_com: bytes
    r: bytes
    ok: bytes
    s: bytes
    sb: bytes


@dataclass
class BatchItem:                          # pedersen::BatchItem; hashing deferred to the GPU
    ios: bytes
    n_ios: int
    ad: bytes
    proof: Proof


class BatchVerifier:
    def __init__(self, suite: Union[Suite, int], fmt: Union[Format, int] = Format.CANONICAL):
        self._lib = _lib.load()
        self.suite, self.fmt = Suite(suite), Format(fmt)
        self._h = self._lib.avrf_pedersen_batch_new(int(self.suite), int(self.fmt))
        if not self._h:
            msg = self._lib.avrf_last_error()
            raise _lib.AvrfError(msg.decode() if msg else "avrf_pedersen_batch_new failed")
        self._n = 0

    @staticmethod
    def prepare(ios, ad, proof: Proof) -> BatchItem:
        iob, k = _ios_bytes(ios)
        return BatchItem(iob, k, bytes(ad), proof)

    def push_prepared(self, e: BatchItem) -> None:
        io_off = np.array([0, e.n_ios], dtype=np.uint32)
        ad_off = np.array([0, len(e.ad)], dtype=np.uint32)
        f = lambda b, n: np.frombuffer(_bytes_of(b, n), dtype=np.uint8).copy()
        self.push_many(np.frombuffer(e.ios + bytes(128), dtype=np.uint8).copy(), io_off,
                       np.frombuffer(e.ad + bytes(16), dtype=np.uint8).copy(), ad_off,
                       f(e.proof.pk_com, 64), f(e.proof.r, 64), f(e.proof.ok, 64), f(e.proof.s, 32), f(e.proof.sb, 32))

    def push(self, ios, ad, proof: Proof) -> None:
        self.push_prepared(self.prepare(ios, ad, proof))

    def push_many(self, ios, io_offsets, ad_blob, ad_offsets, pk_com, r, ok, s, sb) -> None:
        n = len(io_offsets) - 1
        _lib.check(self._lib.avrf_pedersen_batch_push_many(self._h, n, ptr(ios), ptr(io_offsets), ptr(ad_blob),
                                                           ptr(ad_offsets), ptr(pk_com), ptr(r), ptr(ok), ptr(s), ptr(sb)))
        self._n += n

    def push_compressed(self, ios32, io_offsets, ad_blob, ad_offsets, proofs) -> np.ndarray:
        """`avrf_pedersen_batch_push_compressed`: proofs in wire format, (n, 160) records of
        `Proof::serialize_compressed` (see `serialize_proofs`), and 64 bytes of compressed (input, output) per pair;
        decoded and validated on the device.  Returns the per-proof decode flags; when any is 0 nothing was pushed -
        those proofs are the ones `Proof::deserialize_compressed` / `Input` / `Output` deserialisation would refuse."""
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        ok = np.zeros(max(n, 1), dtype=np.uint8)
        bad = C.c_uint64(0)
        _lib.check(self._lib.avrf_pedersen_batch_push_compressed(self._h, n, ptr(ios32), ptr(io_offsets), ptr(ad_blob),
                                                                 ptr(ad_offsets), ptr(proofs), ptr(ok), C.byref(bad)))
        if bad.value == 0:
            self._n += n
        return ok[:n]

    def clear(self) -> None:
        """Forget all pushed proofs, keep allocations."""
        _lib.check(self._lib.avrf_thin_batch_clear(self._h))
        self._n = 0

    def verify_status(self) -> int:
        st = C.c_int32(-1)
        _lib.check(self._lib.avrf_pedersen_batch_verify(self._h, C.byref(st)))
        return st.value

    def verify(self) -> None:
        _raise_for_status(self.verify_status())

    def verify_each(self) -> np.ndarray:
        """Per-proof status codes (0 Ok, 1 VerificationFailure, 2 InvalidData) under `pedersen::Verifier::verify`."""
        out = np.full(max(self._n, 1), -1, dtype=np.int32)
        _lib.check(self._lib.avrf_pedersen_batch_verify_each(self._h, ptr(out)))
        return out[:self._n]

    def find_invalid(self) -> np.ndarray:
        """Indices of the proofs a failed batch owes its verdict to; empty when every proof verifies."""
        return np.nonzero(self.verify_each() != 0)[0]

    def tap(self, what: Tap) -> np.ndarray:
        n = self._n
        size = {Tap.C: 16 * n, Tap.W: 32 * n, Tap.SEED: 64, Tap.SCALARS: 32 * (5 * n + 2)}[Tap(what)]
        buf = np.zeros(max(size, 1), dtype=np.uint8)
        _lib.check(self._lib.avrf_thin_batch_tap(self._h, int(what), ptr(buf), buf.nbytes))
        return buf

    def __len__(self) -> int:
        return self._n

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.avrf_thin_batch_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def verify(suite: Union[Suite, int], ios, ad, proof: Proof, fmt: Union[Format, int] = Format.CANONICAL) -> None:
    """`pedersen::Verifier::verify` (src/pedersen.rs:188-253) for one proof: returns None, or raises VerificationFailure
    / InvalidData like `thin.Public.verify`."""
    lib = _lib.load()
    iob, k = _ios_bytes(ios)
    st = C.c_int32(-1)
    _lib.check(lib.avrf_pedersen_verify_one(int(Suite(suite)), int(Format(fmt)), iob if k else None, k,
                                            bytes(ad) if ad else None, len(ad), _bytes_of(proof.pk_com, 64),
                                            _bytes_of(proof.r, 64), _bytes_of(proof.ok, 64), _bytes_of(proof.s, 32),
                                            _bytes_of(proof.sb, 32), C.byref(st)))
    _raise_for_status(st.value)


def serialize_proofs(suite: Union[Suite, int], pk_com, r, ok, s, sb, fmt: Union[Format, int] = Format.CANONICAL) -> np.ndarray:
    """`pedersen::Proof::serialize_compressed` for n proofs: (n, 64) points and (n, 32) scalars in `fmt` (the arrays
    `prove_many` returns) -> (n, 160) uint8 records pk_com | r | ok | s | sb, as `BatchVerifier.push_compressed` takes
    them.  The points are compressed on the device; Montgomery scalars are converted to canonical on the host."""
    suite, fmt = Suite(suite), Format(fmt)
    pts = np.ascontiguousarray(np.stack([np.asarray(x, dtype=np.uint8).reshape(-1, 64) for x in (pk_com, r, ok)], axis=1))
    n = pts.shape[0]
    out = np.empty((n, 160), dtype=np.uint8)
    out[:, :96] = point_compress(suite, pts.reshape(-1, 64), fmt).reshape(n, 96)
    for k, x in enumerate((s, sb)):
        x = np.ascontiguousarray(x, dtype=np.uint8).reshape(n, 32)
        out[:, 96 + 32 * k:128 + 32 * k] = x if fmt == Format.CANONICAL else _from_mont_scalars(suite, x)
    return out


def _from_mont_scalars(suite: Suite, x: np.ndarray) -> np.ndarray:
    """(n, 32) Montgomery-form scalars (a * 2^256 mod r) -> canonical little-endian."""
    mod = ORDER[suite]
    rinv = pow(1 << 256, -1, mod)
    return np.frombuffer(b"".join((int.from_bytes(bytes(v), "little") * rinv % mod).to_bytes(32, "little") for v in x),
                         dtype=np.uint8).reshape(-1, 32).copy()
