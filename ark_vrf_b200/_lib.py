"""ctypes binding of libavrf_gpu.so (include/avrf.h).

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  Loading
fails loudly when it is missing; computing fails loudly when there is no CUDA device - there
is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libavrf_gpu.so")

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)


class ShardedTimings(C.Structure):
    _fields_ = [("hash_wait_ms", C.c_float), ("host_hash_ms", C.c_float), ("issue_ms", C.c_float),
                ("device_wait_ms", C.c_float), ("total_ms", C.c_float), ("shard_msm_ms_max", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Timings(C.Structure):
    _fields_ = [
        ("h2d_ms", C.c_float), ("prepare_ms", C.c_float), ("d2h_ms", C.c_float), ("host_hash_ms", C.c_float),
        ("scalars_ms", C.c_float), ("sort_ms", C.c_float), ("accumulate_ms", C.c_float), ("reduce_ms", C.c_float),
        ("total_ms", C.c_float),
        ("n_points", C.c_uint64), ("n_entries", C.c_uint64), ("n_tasks", C.c_uint64), ("kernel_launches", C.c_uint64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# name -> (restype, argtypes); every symbol include/avrf.h declares
SIGNATURES = {
    "avrf_init": (C.c_int, [C.c_int]),
    "avrf_init_multi": (C.c_int, [C.c_int, C.POINTER(C.c_int)]),
    "avrf_device_count": (C.c_int, []),
    "avrf_shutdown": (C.c_int, []),
    "avrf_last_error": (C.c_char_p, []),
    "avrf_version": (C.c_char_p, []),
    "avrf_thin_batch_new": (C.c_void_p, [C.c_uint32, C.c_uint32]),
    "avrf_thin_batch_new_on": (C.c_void_p, [C.c_int, C.c_uint32, C.c_uint32]),
    "avrf_thin_batch_device": (C.c_int, [C.c_void_p]),
    "avrf_thin_batch_reserve": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]),
    "avrf_thin_batch_free": (None, [C.c_void_p]),
    "avrf_thin_batch_clear": (C.c_int, [C.c_void_p]),
    "avrf_thin_batch_len": (C.c_int64, [C.c_void_p]),
    "avrf_thin_batch_invalidate": (C.c_int, [C.c_void_p]),
    "avrf_thin_batch_set_eager": (C.c_int, [C.c_void_p, C.c_int]),
    "avrf_thin_batch_set_blocking": (C.c_int, [C.c_void_p, C.c_int]),
    "avrf_hash_pool_new": (C.c_void_p, [C.c_uint32]),
    "avrf_hash_pool_free": (None, [C.c_void_p]),
    "avrf_thin_batch_set_hash_pool": (C.c_int, [C.c_void_p, C.c_void_p]),
    "avrf_stream": (C.c_void_p, []),
    "avrf_thin_batch_stream": (C.c_void_p, [C.c_void_p]),
    "avrf_thin_batch_set_weights_mode": (C.c_int, [C.c_void_p, C.c_uint32]),
    "avrf_thin_batch_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_void_p]),
    "avrf_thin_batch_push_compressed": (C.c_int, [C.c_void_p, C.c_uint64] + [C.c_void_p] * 9),
    "avrf_thin_batch_push_many": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "avrf_thin_batch_verify": (C.c_int, [C.c_void_p, i32p]),
    "avrf_thin_batch_verify_async": (C.c_int, [C.c_void_p]),
    "avrf_thin_batch_verify_wait": (C.c_int, [C.c_void_p, i32p]),
    "avrf_thin_verify_one": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                       C.c_uint32, C.c_void_p, C.c_void_p, i32p]),
    "avrf_thin_batch_prepare": (C.c_int, [C.c_void_p, i32p]),
    "avrf_thin_batch_cs_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "avrf_thin_seed": (C.c_int, [C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_thin_batch_cs_dev": (C.c_void_p, [C.c_void_p]),
    "avrf_thin_seed_dev": (C.c_int, [C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_thin_batch_tree_leaves": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]),
    "avrf_thin_seed_tree": (C.c_int, [C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_thin_batch_partial": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_thin_combine_partials": (C.c_int, [C.c_uint32, C.c_void_p, C.c_uint32, i32p]),
    "avrf_thin_batch_tap": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t]),
    "avrf_thin_sharded_new": (C.c_void_p, [C.c_uint32, C.c_uint32]),
    "avrf_thin_sharded_free": (None, [C.c_void_p]),
    "avrf_thin_sharded_devices": (C.c_int, [C.c_void_p]),
    "avrf_thin_sharded_len": (C.c_int64, [C.c_void_p]),
    "avrf_thin_sharded_clear": (C.c_int, [C.c_void_p]),
    "avrf_thin_sharded_push_many": (C.c_int, [C.c_void_p, C.c_uint64] + [C.c_void_p] * 7),
    "avrf_thin_sharded_verify": (C.c_int, [C.c_void_p, i32p]),
    "avrf_thin_sharded_seed": (C.c_int, [C.c_void_p, C.c_void_p]),
    "avrf_thin_sharded_timings": (C.c_int, [C.c_void_p, C.POINTER(ShardedTimings)]),
    "avrf_thin_sharded_shard": (C.c_void_p, [C.c_void_p, C.c_int]),
    "avrf_pedersen_batch_new": (C.c_void_p, [C.c_uint32, C.c_uint32]),
    "avrf_pedersen_batch_push_many": (C.c_int, [C.c_void_p, C.c_uint64] + [C.c_void_p] * 9),
    "avrf_pedersen_batch_push_compressed": (C.c_int, [C.c_void_p, C.c_uint64] + [C.c_void_p] * 7),
    "avrf_pedersen_batch_verify": (C.c_int, [C.c_void_p, i32p]),
    "avrf_pedersen_batch_verify_each": (C.c_int, [C.c_void_p, C.c_void_p]),
    "avrf_pedersen_verify_one": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, i32p]),
    "avrf_pedersen_prove_many": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint64] + [C.c_void_p] * 12),
    "avrf_hash_to_curve": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "avrf_vrf_output": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_vrf_io_many": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "avrf_public_keys": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_thin_prove_many": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "avrf_points_deserialize": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "avrf_thin_batch_verify_each": (C.c_int, [C.c_void_p, C.c_void_p]),
    "avrf_point_compress": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_point_to_hash": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "avrf_thin_batch_timings": (C.c_int, [C.c_void_p, C.POINTER(Timings)]),
    "avrf_server_new": (C.c_void_p, [C.c_uint32, C.c_uint32, C.c_uint32]),
    "avrf_server_new_mixed": (C.c_void_p, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "avrf_server_new_ex": (C.c_void_p, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "avrf_server_free": (None, [C.c_void_p]),
    "avrf_server_submit": (C.c_int64, [C.c_void_p, C.c_uint64] + [C.c_void_p] * 7),
    "avrf_server_wait": (C.c_int, [C.c_void_p, C.c_int64, i32p]),
    "avrf_mb_sha512": (C.c_int, [C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, i32p]),
    "avrf_microbench": (C.c_int, [C.c_uint32, C.c_uint32, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
}

_lib = None


class AvrfError(RuntimeError):
    """System-level failure (CUDA, memory, bad argument) - never a verification verdict."""


def load() -> C.CDLL:
    """Load libavrf_gpu.so and declare every prototype.  Raises if the extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AvrfError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  ark_vrf_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().avrf_last_error()
        raise AvrfError(f"libavrf_gpu error {rc}: {msg.decode() if msg else ''}")
