"""Host-side mirror of the reference's Thin-VRF verification interface.

Same names, argument meaning and error behaviour as `ark_vrf::thin` (reference
src/thin.rs:95-109, 172-326), forwarding to the C ABI in include/avrf.h:

    reference (Rust)                         here
    ---------------------------------------  -----------------------------------------
    thin::BatchVerifier::<S>::new()          BatchVerifier(suite)
    BatchVerifier::prepare(pk, ios, ad, pf)  BatchVerifier.prepare(...) -> BatchItem
    bv.push_prepared(item)                   bv.push_prepared(item)
    bv.push(pk, ios, ad, proof)              bv.push(pk, ios, ad, proof)
    bv.verify() -> Result<(), Error>         bv.verify()  (raises VerificationFailure / InvalidData)
    public.verify(ios, ad, proof)            Public(suite, pk).verify(ios, ad, proof)

Points are 64-byte affine (x || y), scalars 32 bytes, little-endian, in the format given at
construction (`Format.CANONICAL` integers or `Format.MONTGOMERY` = arkworks memory image).
An I/O pair is `input || output` (128 bytes).  Hashing happens on the GPU, so `prepare`
only captures the inputs (it cannot fail, like the reference's).
"""
from __future__ import annotations

import ctypes as C
import enum
from dataclasses import dataclass
from typing import Iterable, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib


class Suite(enum.IntEnum):
    BANDERSNATCH_SHA512_ELL2 = 0      # src/suites/bandersnatch.rs:56-70
    ED25519_SHA512_TAI = 1            # src/suites/ed25519.rs
    BABYJUBJUB_SHA512_TAI = 2         # src/suites/baby_jubjub.rs


class Format(enum.IntEnum):
    MONTGOMERY = 0
    CANONICAL = 1


class Tap(enum.IntEnum):
    C = 0
    Z = 1
    W = 2
    SEED = 3
    R_COMPRESSED = 4
    PARTIAL = 5
    SCALARS = 6


class Error(Exception):
    """Mirror of `ark_vrf::Error` (src/lib.rs:136-147) - the variants reachable on this path."""


class VerificationFailure(Error):
    pass


class InvalidData(Error):
    pass


STATUS_OK, STATUS_VERIFICATION_FAILURE, STATUS_INVALID_DATA = 0, 1, 2


def _raise_for_status(status: int) -> None:
    if status == STATUS_OK:
        return
    if status == STATUS_INVALID_DATA:
        raise InvalidData("public key or I/O pair point is the group identity")
    raise VerificationFailure("batch equation does not hold")


def ptr(x) -> Optional[int]:
    """Host address of a numpy array / torch CPU tensor / bytes-like (None passes through)."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        assert x.flags["C_CONTIGUOUS"]
        return x.ctypes.data
    if hasattr(x, "data_ptr"):          # torch CPU tensor (possibly pinned)
        assert x.device.type == "cpu" and x.is_contiguous()
        return x.data_ptr()
    if isinstance(x, (bytes, bytearray)):
        return C.cast(C.c_char_p(bytes(x)), C.c_void_p).value
    raise TypeError(type(x))


def _bytes_of(x, n: int) -> bytes:
    b = bytes(x) if not isinstance(x, np.ndarray) else x.tobytes()
    if len(b) != n:
        raise ValueError(f"expected {n} bytes, got {len(b)}")
    return b


def _ios_bytes(ios) -> Tuple[bytes, int]:
    """Accept one pair or a sequence of pairs; a pair is 128 bytes or (input64, output64)."""
    if ios is None:
        return b"", 0
    if isinstance(ios, (bytes, bytearray)):
        if len(ios) % 128:
            raise ValueError("ios must be a multiple of 128 bytes")
        return bytes(ios), len(ios) // 128
    if isinstance(ios, np.ndarray):
        b = ios.tobytes()
        return b, len(b) // 128
    if isinstance(ios, tuple) and len(ios) == 2 and not isinstance(ios[0], tuple):
        ios = [ios]                      # single VrfIo (lib.rs:621-625: VrfIo: AsRef<[VrfIo]>)
    out = bytearray()
    k = 0
    for io in ios:
        if isinstance(io, (bytes, bytearray)):
            out += _bytes_of(io, 128)
        else:
            out += _bytes_of(io[0], 64) + _bytes_of(io[1], 64)
        k += 1
    return bytes(out), k


@dataclass
class Proof:                              # thin::Proof (src/thin.rs:42-48)
    r: bytes                              # 64-byte affine point
    s: bytes                              # 32-byte scalar


@dataclass
class BatchItem:                          # thin::BatchItem (src/thin.rs:172-179); hashing deferred to the GPU
    pk: bytes
    ios: bytes
    n_ios: int
    ad: bytes
    r: bytes
    s: bytes


class _BatchBase:
    """The controls of a batch handle that serve both schemes (include/avrf.h): `thin.BatchVerifier` and
    `pedersen.BatchVerifier` share them, and so do the building blocks of a batch sharded over processes
    (`dist.sharded_verify`).  Pushes, taps and per-proof verdicts are scheme-specific and stay in those classes."""

    cs_stride = 64                        # bytes per proof of the batch-seed stream (Thin: c || s; Pedersen: c || s || sb)

    def _open(self, handle, what: str) -> None:
        self._h = handle
        if not self._h:
            msg = self._lib.avrf_last_error()
            raise _lib.AvrfError(msg.decode() if msg else f"{what} failed")

    def verify(self) -> None:
        """Ok -> returns None; otherwise raises VerificationFailure or InvalidData."""
        _raise_for_status(self.verify_status())

    def verify_async(self) -> None:
        """Enqueue the verification on the GPU and return (pair with `verify_wait`)."""
        _lib.check(self._lib.avrf_thin_batch_verify_async(self._h))

    def verify_wait(self) -> int:
        st = C.c_int32(-1)
        _lib.check(self._lib.avrf_thin_batch_verify_wait(self._h, C.byref(st)))
        return st.value

    def set_blocking(self, blocking: bool = True) -> None:
        """Host waits sleep instead of spinning (use when several handles are driven from as many threads)."""
        _lib.check(self._lib.avrf_thin_batch_set_blocking(self._h, 1 if blocking else 0))

    def set_hash_pool(self, pool: Optional["HashPool"]) -> None:
        """Hash this handle's batch seeds in a lane of a shared multi-buffer pool (None: on its own thread)."""
        _lib.check(self._lib.avrf_thin_batch_set_hash_pool(self._h, pool._h if pool is not None else None))
        self._pool = pool                 # keep it alive

    def reserve(self, n: int, n_ios: int, ad_bytes: int) -> None:
        """Room for `n` proofs (like `Vec::with_capacity`): pushes up to that size never reallocate device memory."""
        _lib.check(self._lib.avrf_thin_batch_reserve(self._h, n, n_ios, ad_bytes))

    def clear(self) -> None:
        """Forget all pushed proofs, keep allocations."""
        _lib.check(self._lib.avrf_thin_batch_clear(self._h))

    def invalidate(self) -> None:
        """Forget c_j / z_ij / prepared bases; inputs stay resident (next verify redoes prepare)."""
        _lib.check(self._lib.avrf_thin_batch_invalidate(self._h))

    def __len__(self) -> int:
        return int(self._lib.avrf_thin_batch_len(self._h))

    @property
    def stream(self) -> int:
        """The handle's CUDA stream (a ``cudaStream_t`` as an integer) - record timing events on it."""
        return int(self._lib.avrf_thin_batch_stream(self._h))

    def timings(self) -> dict:
        t = _lib.Timings()
        _lib.check(self._lib.avrf_thin_batch_timings(self._h, C.byref(t)))
        return t.as_dict()

    # -- sharded path ------------------------------------------------------------------------
    def prepare_device(self) -> bool:
        """Runs the per-proof transcripts on the GPU; returns True if an identity pk (pk_com) / I / O was seen."""
        inv = C.c_int32(0)
        _lib.check(self._lib.avrf_thin_batch_prepare(self._h, C.byref(inv)))
        return bool(inv.value)

    def cs_stream(self) -> np.ndarray:
        """The batch-seed stream of this handle's proofs, one `cs_stride`-byte record per proof."""
        out = np.empty((len(self), self.cs_stride), dtype=np.uint8)
        _lib.check(self._lib.avrf_thin_batch_cs_stream(self._h, ptr(out)))
        return out

    def cs_stream_dev(self):
        """(device pointer, n_bytes) of the batch-seed stream after prepare (for a device-side all-gather)."""
        p = self._lib.avrf_thin_batch_cs_dev(self._h)
        if not p and len(self):
            _lib.check(-1)
        return p, self.cs_stride * len(self)

    def partial(self, seed: bytes, first_index: int) -> bytes:
        """This handle's share of the batch MSM under `seed`, its proofs at global indices first_index, ... (128 bytes,
        extended coordinates in Montgomery form)."""
        out = (C.c_uint8 * 128)()
        _lib.check(self._lib.avrf_thin_batch_partial(self._h, _bytes_of(seed, 64), first_index, out))
        return bytes(out)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.avrf_thin_batch_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchVerifier(_BatchBase):
    """thin::BatchVerifier<S> (src/thin.rs:188-326) on one B200."""

    def __init__(self, suite: Union[Suite, int], fmt: Union[Format, int] = Format.CANONICAL, eager_seed: bool = True,
                 device: int = -1):
        self._lib = _lib.load()
        self.suite = Suite(suite)
        self.fmt = Format(fmt)
        self._open(self._lib.avrf_thin_batch_new_on(int(device), int(self.suite), int(self.fmt)), "avrf_thin_batch_new")
        self._n_ios = 0
        if not eager_seed:
            _lib.check(self._lib.avrf_thin_batch_set_eager(self._h, 0))

    # -- reference API -------------------------------------------------------------------
    @staticmethod
    def prepare(public, ios, ad, proof: Proof) -> BatchItem:
        iob, k = _ios_bytes(ios)
        return BatchItem(_bytes_of(public, 64), iob, k, bytes(ad), _bytes_of(proof.r, 64), _bytes_of(proof.s, 32))

    def push_prepared(self, item: BatchItem) -> None:
        self._n_ios += item.n_ios
        _lib.check(self._lib.avrf_thin_batch_push(self._h, item.pk, item.ios if item.n_ios else None, item.n_ios,
                                                  item.ad if item.ad else None, len(item.ad), item.r, item.s))

    def push(self, public, ios, ad, proof: Proof) -> None:
        self.push_prepared(self.prepare(public, ios, ad, proof))

    # -- bulk / measurement API ---------------------------------------------------------------
    def push_many(self, pk, ios, io_offsets, ad_blob, ad_offsets, r, s) -> None:
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        self._n_ios += int(io_offsets[n])
        _lib.check(self._lib.avrf_thin_batch_push_many(self._h, n, ptr(pk), ptr(ios), ptr(io_offsets), ptr(ad_blob),
                                                       ptr(ad_offsets), ptr(r), ptr(s)))

    def push_compressed(self, pk32, ios32, io_offsets, ad_blob, ad_offsets, r32, s) -> np.ndarray:
        """`avrf_thin_batch_push_compressed`: proofs in wire format (32-byte compressed points, canonical scalars), decoded
        and validated on the device.  Returns the per-proof decode flags; when any is 0 nothing was pushed - those
        proofs are the ones `Proof::deserialize_compressed` / `Public::deserialize_compressed` would have refused."""
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        ok = np.zeros(max(n, 1), dtype=np.uint8)
        bad = C.c_uint64(0)
        _lib.check(self._lib.avrf_thin_batch_push_compressed(self._h, n, ptr(pk32), ptr(ios32), ptr(io_offsets), ptr(ad_blob),
                                                             ptr(ad_offsets), ptr(r32), ptr(s), ptr(ok), C.byref(bad)))
        if bad.value == 0:
            self._n_ios += int(io_offsets[n])
        return ok[:n]

    def verify_status(self) -> int:
        st = C.c_int32(-1)
        _lib.check(self._lib.avrf_thin_batch_verify(self._h, C.byref(st)))
        return st.value

    def verify_each(self) -> np.ndarray:
        """Per-proof status codes (0 Ok, 1 VerificationFailure, 2 InvalidData): names the bad proofs."""
        out = np.full(max(len(self), 1), -1, dtype=np.int32)
        _lib.check(self._lib.avrf_thin_batch_verify_each(self._h, ptr(out)))
        return out[:len(self)]

    def find_invalid(self) -> np.ndarray:
        """Indices of the proofs a failed batch owes its verdict to (status != Ok under `thin::Verifier::verify`,
        src/thin.rs:131-165); empty when every proof verifies.  The reference only reports that some proof is bad."""
        return np.nonzero(self.verify_each() != 0)[0]

    def clear(self) -> None:
        super().clear()
        self._n_ios = 0

    def set_weights_mode(self, mode: int) -> None:
        _lib.check(self._lib.avrf_thin_batch_set_weights_mode(self._h, mode))

    # -- sharded path (prepare_device, cs_stream, cs_stream_dev, partial: _BatchBase) --------------
    def tree_leaves(self, first_index: int = 0) -> np.ndarray:
        """Leaf digests of this handle's stream for AVRF_WEIGHTS_TREE (64 bytes per 32 proofs)."""
        out = np.zeros(((len(self) + 31) // 32 + 1, 64), dtype=np.uint8)
        n = C.c_uint64(0)
        _lib.check(self._lib.avrf_thin_batch_tree_leaves(self._h, first_index, ptr(out), C.byref(n)))
        return out[:n.value]

    def tap(self, what: Tap) -> np.ndarray:
        n = len(self)
        what = Tap(what)
        size = {Tap.C: 16 * n, Tap.W: 16 * n, Tap.SEED: 64, Tap.R_COMPRESSED: 32 * n, Tap.PARTIAL: 128,
                Tap.Z: 16 * self._n_ios, Tap.SCALARS: 32 * (2 * n + 2 * self._n_ios + 1)}[what]
        buf = np.zeros(max(size, 1), dtype=np.uint8)
        _lib.check(self._lib.avrf_thin_batch_tap(self._h, int(what), ptr(buf), buf.nbytes))
        return buf


class HashPool:
    """`avrf_hash_pool_*`: host threads that each advance up to eight batches' SHA-512 chains in lockstep (AVX-512)."""

    def __init__(self, n_threads: int):
        self._lib = _lib.load()
        self._h = self._lib.avrf_hash_pool_new(int(n_threads))
        if not self._h:
            msg = self._lib.avrf_last_error()
            raise _lib.AvrfError(msg.decode() if msg else "avrf_hash_pool_new failed")

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.avrf_hash_pool_free(self._h)
            self._h = None


def init_multi(n_dev: int = 0, dev_ids: Optional[Sequence[int]] = None) -> int:
    """`avrf_init_multi`: several GPUs in this process (n_dev <= 0: all).  Returns the number of devices."""
    lib = _lib.load()
    arr = (C.c_int * len(dev_ids))(*dev_ids) if dev_ids else None
    _lib.check(lib.avrf_init_multi(len(dev_ids) if dev_ids else int(n_dev), arr))
    return int(lib.avrf_device_count())


class _ShardView(BatchVerifier):
    """One device's ordinary handle inside a `ShardedBatchVerifier` (taps and timings only; owned by the parent)."""

    def __init__(self, parent, handle, n_ios):
        self._lib, self.suite, self.fmt, self._h, self._n_ios, self._parent = parent._lib, parent.suite, parent.fmt, handle, n_ios, parent

    def close(self) -> None:
        self._h = None


class _ShardedBase:
    """What the multi-GPU batches of both schemes share (include/avrf.h, "Multi-GPU batches"): every
    `avrf_thin_sharded_*` call but the constructor and the push serves either kind of handle."""

    def _open(self, new, what: str) -> None:
        self._lib = _lib.load()
        self._h = new(int(self.suite), int(self.fmt))
        if not self._h:
            msg = self._lib.avrf_last_error()
            raise _lib.AvrfError(msg.decode() if msg else f"{what} failed")

    def _shard_handle(self, index: int):
        h = self._lib.avrf_thin_sharded_shard(self._h, index)
        if not h:
            _lib.check(-2)
        return h

    @property
    def devices(self) -> int:
        return int(self._lib.avrf_thin_sharded_devices(self._h))

    def __len__(self) -> int:
        return int(self._lib.avrf_thin_sharded_len(self._h))

    def verify_status(self) -> int:
        st = C.c_int32(-1)
        _lib.check(self._lib.avrf_thin_sharded_verify(self._h, C.byref(st)))
        return st.value

    def verify(self) -> None:
        _raise_for_status(self.verify_status())

    def clear(self) -> None:
        _lib.check(self._lib.avrf_thin_sharded_clear(self._h))

    def seed(self) -> bytes:
        out = (C.c_uint8 * 64)()
        _lib.check(self._lib.avrf_thin_sharded_seed(self._h, out))
        return bytes(out)

    def timings(self) -> dict:
        t = _lib.ShardedTimings()
        _lib.check(self._lib.avrf_thin_sharded_timings(self._h, C.byref(t)))
        return t.as_dict()

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.avrf_thin_sharded_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ShardedBatchVerifier(_ShardedBase):
    """thin::BatchVerifier<S> (src/thin.rs:188-326) over every GPU initialised with `init_multi`, inside ONE
    process and without torch.distributed: include/avrf.h, "Multi-GPU batches"."""

    def __init__(self, suite: Union[Suite, int], fmt: Union[Format, int] = Format.CANONICAL):
        self.suite, self.fmt = Suite(suite), Format(fmt)
        self._open(_lib.load().avrf_thin_sharded_new, "avrf_thin_sharded_new")

    def push_many(self, pk, ios, io_offsets, ad_blob, ad_offsets, r, s) -> None:
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        _lib.check(self._lib.avrf_thin_sharded_push_many(self._h, n, ptr(pk), ptr(ios), ptr(io_offsets), ptr(ad_blob),
                                                         ptr(ad_offsets), ptr(r), ptr(s)))

    def shard(self, index: int, n_ios: int) -> "_ShardView":
        """Device `index`'s handle (taps / timings); `n_ios` = I/O pairs it holds (sizes the Z / SCALARS taps)."""
        return _ShardView(self, self._shard_handle(index), n_ios)


class _ServerBase:
    """What the batch servers of both schemes share (include/avrf.h, "Batch server"): tickets, waits and the lifetime
    of borrowed arrays.  The arrays of a submitted batch (and the decode flags a wire-format submit allocates) are kept
    alive, and must not be modified, until its `wait` returns."""

    def _start(self, new, suite, fmt, workers: int, hashers: int, own_hash_workers: int) -> None:
        self._lib = _lib.load()
        self.suite, self.fmt, self.workers, self.hashers = Suite(suite), Format(fmt), int(workers), int(hashers)
        self._h = new(int(self.suite), int(self.fmt), self.workers, self.hashers, int(own_hash_workers))
        if not self._h:
            msg = self._lib.avrf_last_error()
            raise _lib.AvrfError(msg.decode() if msg else "batch server: creation failed")
        self._live = {}
        self._dec_ok = {}                    # ticket -> decode flags of a wire-format job

    def _submit(self, fn, arrays, n: int, wire: bool) -> int:
        ok = np.zeros(max(n, 1), dtype=np.uint8) if wire else None
        t = int(fn(self._h, n, *[ptr(a) for a in arrays], *((ptr(ok), None) if wire else ())))
        if t < 0:
            _lib.check(t)
        self._live[t] = (arrays, ok)
        if wire:
            self._dec_ok[t] = ok[:n]
        return t

    def wait(self, ticket: int) -> int:
        st = C.c_int32(-1)
        try:
            _lib.check(self._lib.avrf_server_wait(self._h, ticket, C.byref(st)))
        finally:
            self._live.pop(ticket, None)
        return st.value

    def wait_compressed(self, ticket: int) -> Tuple[int, np.ndarray]:
        """`wait` for a wire-format job: (status, per-proof decode flags).  When a flag is False the job's proofs did
        not all decode, nothing was verified and the status is InvalidData."""
        if ticket in self._live and ticket not in self._dec_ok:
            raise ValueError(f"ticket {ticket} is not a wire-format job")
        ok = self._dec_ok.pop(ticket, None)
        status = self.wait(ticket)
        return status, ok.astype(bool)

    def verify(self, ticket: int) -> None:
        """`wait`, mapped onto the reference's `Result<(), Error>`."""
        _raise_for_status(self.wait(ticket))

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.avrf_server_free(self._h)       # finishes queued batches first
            self._h = None
            self._live.clear()
            self._dec_ok.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchServer(_ServerBase):
    """Throughput mode: a native pool of worker threads, one `BatchVerifier` handle each (include/avrf.h,
    "Batch server").  `submit` enqueues a whole batch and returns a ticket; `wait` returns its status code.
    The arrays of a submitted batch are kept alive (and must not be modified) until its `wait` returns."""

    def __init__(self, suite: Union[Suite, int], fmt: Union[Format, int] = Format.CANONICAL, workers: int = 4,
                 hashers: int = 0, own_hash_workers: int = 0):
        """`hashers` > 0: that many shared multi-buffer SHA-512 threads (eight batches' hash chains per thread)
        instead of one hashing core per worker - for boxes with fewer free cores than batches in flight.
        `own_hash_workers`: that many of the workers keep hashing on their own thread (mixed pool)."""
        self._start(_lib.load().avrf_server_new_mixed, suite, fmt, workers, hashers, own_hash_workers)

    def submit(self, pk, ios, io_offsets, ad_blob, ad_offsets, r, s) -> int:
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        return self._submit(self._lib.avrf_server_submit, (pk, ios, io_offsets, ad_blob, ad_offsets, r, s), n, False)

    def submit_compressed(self, pk32, ios32, io_offsets, ad_blob, ad_offsets, r32, s) -> int:
        """A job of proofs in wire format, arguments as `BatchVerifier.push_compressed`; `wait_compressed` returns its
        status and decode flags."""
        n = len(io_offsets) - 1
        assert len(ad_offsets) == n + 1
        return self._submit(self._lib.avrf_server_submit_compressed, (pk32, ios32, io_offsets, ad_blob, ad_offsets, r32, s),
                            n, True)


def seed_of_stream(suite: Union[Suite, int], cs_stream) -> bytes:
    """SHA512(SUITE_ID || 0x50 || stream) (src/thin.rs:274-279)."""
    lib = _lib.load()
    out = (C.c_uint8 * 64)()
    n = (cs_stream.nbytes if isinstance(cs_stream, np.ndarray) else len(cs_stream)) // 64
    _lib.check(lib.avrf_thin_seed(int(suite), ptr(cs_stream), n, out))
    return bytes(out)


def seed_of_tree(suite: Union[Suite, int], n_total: int, leaves: np.ndarray) -> bytes:
    lib = _lib.load()
    out = (C.c_uint8 * 64)()
    leaves = np.ascontiguousarray(leaves, dtype=np.uint8)
    _lib.check(lib.avrf_thin_seed_tree(int(suite), n_total, ptr(leaves), leaves.size // 64, out))
    return bytes(out)


def seed_of_device_stream(suite: Union[Suite, int], dev_ptr: int, n_items: int) -> bytes:
    lib = _lib.load()
    out = (C.c_uint8 * 64)()
    _lib.check(lib.avrf_thin_seed_dev(int(suite), dev_ptr, n_items, out))
    return bytes(out)


def combine_partials(suite: Union[Suite, int], partials: bytes) -> int:
    lib = _lib.load()
    st = C.c_int32(-1)
    _lib.check(lib.avrf_thin_combine_partials(int(suite), partials, len(partials) // 128, C.byref(st)))
    return st.value


class Public:
    """`Public<S>` with `thin::Verifier::verify` (src/thin.rs:131-165)."""

    def __init__(self, suite: Union[Suite, int], point, fmt: Union[Format, int] = Format.CANONICAL):
        self.suite, self.fmt, self.point = Suite(suite), Format(fmt), _bytes_of(point, 64)

    def verify(self, ios, ad, proof: Proof) -> None:
        lib = _lib.load()
        iob, k = _ios_bytes(ios)
        st = C.c_int32(-1)
        _lib.check(lib.avrf_thin_verify_one(int(self.suite), int(self.fmt), self.point, iob if k else None, k,
                                            bytes(ad) if ad else None, len(ad), _bytes_of(proof.r, 64),
                                            _bytes_of(proof.s, 32), C.byref(st)))
        _raise_for_status(st.value)
