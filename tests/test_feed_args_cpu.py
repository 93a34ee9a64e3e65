"""The handle-less entry points (hash-to-curve, outputs, public keys, vrf_io_many, the provers, compression,
deserialisation, point-to-hash, combine_partials, the microbenchmarks) refuse every malformed argument with
AVRF_ERR_ARG and the same avrf_last_error() text, before they look for a device; a well-formed call without a
device fails with a system error, never 0."""
import ctypes as C

import pytest

AVRF_ERR_ARG, AVRF_ERR_NO_DEVICE = -2, -4


def _u32(*v):
    return (C.c_uint32 * len(v))(*v)


def _out(n):
    return C.create_string_buffer(n)


def _valid_calls():
    """name -> (positional arguments of a well-formed one-item call, names of those arguments)"""
    offs, sk, pt = _u32(0, 3), bytes(32), bytes(64)
    io_off, ad_off = _u32(0, 1), _u32(0, 0)
    return {
        "avrf_hash_to_curve": ((0, 1, b"abc", offs, 1, _out(64), _out(32), _out(1)),
                               "suite fmt msgs offsets n out_affine out_compressed ok"),
        "avrf_vrf_output": ((0, 1, sk, 32, pt, 1, _out(64)), "suite fmt sk sk_stride inputs n outputs"),
        "avrf_public_keys": ((0, 1, sk, 1, _out(64)), "suite fmt sk n pk"),
        "avrf_vrf_io_many": ((0, 1, b"abc", offs, 1, sk, 32, _out(64), _out(64), _out(32), _out(1)),
                             "suite fmt msgs offsets n sk sk_stride out_inputs out_outputs out_hashes ok"),
        "avrf_thin_prove_many": ((0, 1, 1, sk, pt, bytes(128), io_off, None, ad_off, _out(64), _out(32)),
                                 "suite fmt n sk pk ios io_offsets ad_blob ad_offsets r s"),
        "avrf_pedersen_prove_many": ((0, 1, 1, sk, pt, bytes(128), io_off, None, ad_off, _out(64), _out(64), _out(64),
                                      _out(32), _out(32), _out(32)),
                                     "suite fmt n sk pk ios io_offsets ad_blob ad_offsets pk_com r ok s sb blinding"),
        "avrf_point_compress": ((0, 1, pt, 1, _out(32)), "suite fmt points n out32"),
        "avrf_point_to_hash": ((0, 1, pt, 1, _out(32)), "suite fmt points n out32"),
        "avrf_points_deserialize": ((0, 1, 1, sk, 1, _out(64), _out(1)), "suite fmt kind in32 n out64 ok"),
        "avrf_thin_combine_partials": ((0, bytes(128), 1, C.byref(C.c_int32(-7))), "suite partials n status"),
        "avrf_microbench": ((0, 1, C.byref(C.c_double()), C.byref(C.c_float())), "kind iters per_second ms"),
    }


# (entry point, {argument: value}, avrf_last_error() text): every kind of argument each entry point refuses
_BAD = "bad argument"
REJECTED = (
    [("avrf_hash_to_curve", {a: v}, _BAD) for a, v in [("suite", 3), ("fmt", 2), ("offsets", None), ("msgs", None)]]
    + [("avrf_vrf_output", {"inputs": None}, "null inputs")]
    + [("avrf_vrf_output", {a: v}, _BAD) for a, v in [("suite", 3), ("fmt", 2), ("sk", None), ("outputs", None),
                                                        ("sk_stride", 4), ("sk_stride", 64)]]
    + [("avrf_public_keys", {a: v}, _BAD) for a, v in [("suite", 3), ("fmt", 2), ("sk", None), ("pk", None)]]
    + [("avrf_vrf_io_many", {a: v}, _BAD) for a, v in [("suite", 3), ("fmt", 2), ("offsets", None), ("sk", None),
                                                         ("msgs", None), ("sk_stride", 16)]]
    + [("avrf_thin_prove_many", {a: v}, _BAD) for a, v in [("suite", 3), ("fmt", 2), ("sk", None), ("pk", None),
                                                             ("io_offsets", None), ("ad_offsets", None), ("r", None),
                                                             ("s", None)]]
    + [("avrf_pedersen_prove_many", {a: v}, _BAD)
       for a, v in [("suite", 3), ("fmt", 2), ("sk", None), ("pk", None), ("io_offsets", None), ("ad_offsets", None),
                    ("pk_com", None), ("r", None), ("ok", None), ("s", None), ("sb", None)]]
    + [(f, {a: v}, _BAD) for f in ("avrf_point_compress", "avrf_point_to_hash")
       for a, v in [("suite", 3), ("fmt", 2), ("points", None), ("out32", None)]]
    + [("avrf_points_deserialize", {a: v}, _BAD) for a, v in [("suite", 3), ("fmt", 2), ("kind", 2), ("in32", None),
                                                                ("out64", None), ("ok", None)]]
    + [("avrf_thin_combine_partials", {a: v}, _BAD) for a, v in [("suite", 3), ("partials", None), ("n", 0),
                                                                   ("status", None)]]
    + [("avrf_microbench", {a: v}, _BAD) for a, v in [("per_second", None), ("iters", 0)]]
)


def _call(name, **change):
    from ark_vrf_b200 import _lib
    lib = _lib.load()
    args, names = _valid_calls()[name]
    args = list(args)
    for k, v in change.items():
        args[names.split().index(k)] = v
    return getattr(lib, name)(*args), lib.avrf_last_error().decode()


@pytest.mark.parametrize("name,change,msg", REJECTED,
                         ids=[f"{n}-{'-'.join(f'{k}={v}' for k, v in c.items())}" for n, c, _ in REJECTED])
def test_rejects_bad_argument(name, change, msg):
    rc, err = _call(name, **change)
    assert (rc, err) == (AVRF_ERR_ARG, msg)


@pytest.mark.parametrize("name", sorted(_valid_calls()))
def test_valid_call_needs_a_device(name):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    rc, _ = _call(name)
    assert rc == AVRF_ERR_NO_DEVICE


@pytest.mark.gpu
def test_checks_after_device_lookup():
    """Refusals that come after the device is bound: too many proofs (before io_offsets[n] is read: the offsets
    array here has two entries), a missing I/O blob that the offsets say is not empty, an unknown microbench kind."""
    big = 1 << 32
    for name, change, msg in [("avrf_thin_prove_many", {"n": big}, "too many proofs for one call"),
                              ("avrf_pedersen_prove_many", {"n": big}, "too many proofs for one call"),
                              ("avrf_public_keys", {"n": big}, "too many items for one call"),
                              ("avrf_thin_prove_many", {"ios": None}, "null argument"),
                              ("avrf_pedersen_prove_many", {"ios": None}, "null argument"),
                              ("avrf_microbench", {"kind": 5}, "unknown microbench kind")]:
        assert _call(name, **change) == (AVRF_ERR_ARG, msg), (name, change)
