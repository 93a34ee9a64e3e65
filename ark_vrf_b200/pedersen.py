"""Pedersen VRF on the GPU (SURVEY.md 8f-3): proving, single and batch verification.

Mirror of `ark_vrf::pedersen` (reference src/pedersen.rs):
    Prover::prove                    prove_many(...)             (pedersen.rs:136-186, n proofs per call)
    Verifier::verify                 verify(suite, ios, ad, proof)  (pedersen.rs:188-253, exact)
    BatchVerifier::{new, push, push_prepared, verify}   BatchVerifier  (pedersen.rs:322-427; the MSM has 5N+2 points;
                                                    push stages each proof in pinned memory, shipped in chunks)
    (handle controls, as thin.BatchVerifier)        BatchVerifier.{verify_async, verify_wait, reserve, set_blocking,
                                                    set_hash_pool, invalidate, timings, stream, clear}
    (wire-format proofs)             BatchVerifier.push_compressed(), serialize_proofs()  (Proof::{de,}serialize_compressed)
    (per-proof verdicts)             BatchVerifier.verify_each() / find_invalid()
    (throughput mode)                BatchServer: whole batches on a native worker pool, decoded or in wire format
    (one batch over several GPUs)    ShardedBatchVerifier: every GPU of this process (init_multi);
                                     BatchVerifier.{prepare_device, cs_stream, cs_stream_dev, partial}, seed_of_stream,
                                     seed_of_device_stream: one process per GPU (dist.sharded_verify)
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
from .thin import (Format, Suite, Tap, _BatchBase, _ServerBase, _ShardedBase, _bytes_of, _ios_bytes, _raise_for_status,
                   ptr)


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


class BatchVerifier(_BatchBase):
    """pedersen::BatchVerifier<S> (src/pedersen.rs:322-427) on one B200; the handle controls are `thin.BatchVerifier`'s.
    `eager_seed=False` (a shard of a batch spread over processes: its seed comes from the gathered stream) and `device`
    as in `thin.BatchVerifier`."""

    cs_stride = 96                        # c || s || sb per proof (src/pedersen.rs:361-367)

    def __init__(self, suite: Union[Suite, int], fmt: Union[Format, int] = Format.CANONICAL, eager_seed: bool = True,
                 device: int = -1):
        self._lib = _lib.load()
        self.suite, self.fmt = Suite(suite), Format(fmt)
        self._open(self._lib.avrf_pedersen_batch_new_on(int(device), int(self.suite), int(self.fmt)),
                   "avrf_pedersen_batch_new")
        if not eager_seed:
            _lib.check(self._lib.avrf_thin_batch_set_eager(self._h, 0))

    @staticmethod
    def prepare(ios, ad, proof: Proof) -> BatchItem:
        iob, k = _ios_bytes(ios)
        return BatchItem(iob, k, bytes(ad), proof)

    def push_prepared(self, e: BatchItem) -> None:
        p = e.proof
        _lib.check(self._lib.avrf_pedersen_batch_push(self._h, e.ios if e.n_ios else None, e.n_ios, e.ad if e.ad else None,
                                                      len(e.ad), _bytes_of(p.pk_com, 64), _bytes_of(p.r, 64),
                                                      _bytes_of(p.ok, 64), _bytes_of(p.s, 32), _bytes_of(p.sb, 32)))

    def push(self, ios, ad, proof: Proof) -> None:
        self.push_prepared(self.prepare(ios, ad, proof))

    def push_many(self, ios, io_offsets, ad_blob, ad_offsets, pk_com, r, ok, s, sb) -> None:
        n = len(io_offsets) - 1
        _lib.check(self._lib.avrf_pedersen_batch_push_many(self._h, n, ptr(ios), ptr(io_offsets), ptr(ad_blob),
                                                           ptr(ad_offsets), ptr(pk_com), ptr(r), ptr(ok), ptr(s), ptr(sb)))

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
        return ok[:n]

    def verify_status(self) -> int:
        st = C.c_int32(-1)
        _lib.check(self._lib.avrf_pedersen_batch_verify(self._h, C.byref(st)))
        return st.value

    def verify_each(self) -> np.ndarray:
        """Per-proof status codes (0 Ok, 1 VerificationFailure, 2 InvalidData) under `pedersen::Verifier::verify`."""
        n = len(self)
        out = np.full(max(n, 1), -1, dtype=np.int32)
        _lib.check(self._lib.avrf_pedersen_batch_verify_each(self._h, ptr(out)))
        return out[:n]

    def find_invalid(self) -> np.ndarray:
        """Indices of the proofs a failed batch owes its verdict to; empty when every proof verifies."""
        return np.nonzero(self.verify_each() != 0)[0]

    def tap(self, what: Tap) -> np.ndarray:
        n = len(self)
        size = {Tap.C: 16 * n, Tap.W: 32 * n, Tap.SEED: 64, Tap.SCALARS: 32 * (5 * n + 2), Tap.PARTIAL: 128}[Tap(what)]
        buf = np.zeros(max(size, 1), dtype=np.uint8)
        _lib.check(self._lib.avrf_thin_batch_tap(self._h, int(what), ptr(buf), buf.nbytes))
        return buf


class _ShardView(BatchVerifier):
    """One device's Pedersen handle inside a `ShardedBatchVerifier` (taps, timings, verify_each; owned by the parent)."""

    def __init__(self, parent, handle):
        self._lib, self.suite, self.fmt, self._h, self._parent = parent._lib, parent.suite, parent.fmt, handle, parent

    def close(self) -> None:
        self._h = None


class ShardedBatchVerifier(_ShardedBase):
    """pedersen::BatchVerifier<S> (src/pedersen.rs:322-427) over every GPU initialised with `thin.init_multi`, inside
    ONE process: include/avrf.h, "Multi-GPU batches".  Seed, weights and verdict are those of one `BatchVerifier`
    holding the same proofs in the same order; the serial batch-seed hash still runs once, on one core."""

    def __init__(self, suite: Union[Suite, int], fmt: Union[Format, int] = Format.CANONICAL):
        self.suite, self.fmt = Suite(suite), Format(fmt)
        self._open(_lib.load().avrf_pedersen_sharded_new, "avrf_pedersen_sharded_new")

    def push_many(self, ios, io_offsets, ad_blob, ad_offsets, pk_com, r, ok, s, sb) -> None:
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        _lib.check(self._lib.avrf_pedersen_sharded_push_many(self._h, n, ptr(ios), ptr(io_offsets), ptr(ad_blob),
                                                             ptr(ad_offsets), ptr(pk_com), ptr(r), ptr(ok), ptr(s),
                                                             ptr(sb)))

    def shard(self, index: int) -> _ShardView:
        """Device `index`'s handle: `tap` (W: t_j || u_j, 32 bytes per proof; SCALARS: 5n + 2 terms), `timings` and
        `verify_each`, indexed by the proof's position on that device."""
        return _ShardView(self, self._shard_handle(index))


def seed_of_stream(suite: Union[Suite, int], stream) -> bytes:
    """SHA512(SUITE_ID || 0x50 || stream) of 96-byte records c || s || sb (src/pedersen.rs:361-367)."""
    lib = _lib.load()
    out = (C.c_uint8 * 64)()
    n = (stream.nbytes if isinstance(stream, np.ndarray) else len(stream)) // BatchVerifier.cs_stride
    _lib.check(lib.avrf_pedersen_seed(int(suite), ptr(stream), n, out))
    return bytes(out)


def seed_of_device_stream(suite: Union[Suite, int], dev_ptr: int, n_items: int) -> bytes:
    """The same seed of `n_items` records resident on the default device (`avrf_pedersen_seed_dev`)."""
    lib = _lib.load()
    out = (C.c_uint8 * 64)()
    _lib.check(lib.avrf_pedersen_seed_dev(int(suite), dev_ptr, n_items, out))
    return bytes(out)


class BatchServer(_ServerBase):
    """Throughput mode for the Pedersen VRF: a native pool of worker threads, one Pedersen `BatchVerifier` handle each
    (include/avrf.h, "Batch server").  `submit` / `submit_compressed` enqueue a whole batch (new + push + verify) and
    return a ticket; `wait` returns its status code, `wait_compressed` the status and the decode flags of a wire-format
    job.  Pool shapes as `thin.BatchServer`.  The arrays of a submitted batch are kept alive (and must not be modified)
    until its `wait` returns."""

    def __init__(self, suite: Union[Suite, int], fmt: Union[Format, int] = Format.CANONICAL, workers: int = 4,
                 hashers: int = 0, own_hash_workers: int = 0):
        self._start(_lib.load().avrf_pedersen_server_new, suite, fmt, workers, hashers, own_hash_workers)

    def submit(self, ios, io_offsets, ad_blob, ad_offsets, pk_com, r, ok, s, sb) -> int:
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        return self._submit(self._lib.avrf_pedersen_server_submit, (ios, io_offsets, ad_blob, ad_offsets, pk_com, r, ok, s, sb),
                            n, False)

    def submit_compressed(self, ios32, io_offsets, ad_blob, ad_offsets, proofs) -> int:
        """A job of proofs in wire format, arguments as `BatchVerifier.push_compressed`."""
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        return self._submit(self._lib.avrf_pedersen_server_submit_compressed, (ios32, io_offsets, ad_blob, ad_offsets, proofs),
                            n, True)


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
