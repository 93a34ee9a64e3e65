"""CPU, world_size 2, gloo: `dist.sharded_verify` with Pedersen shards - 96-byte batch-seed records gathered in global
order, (t_j, u_j) squeezed two proofs per block at the global index, each rank's share of the G and B terms, the
InvalidData gate, the refused tree mode - with an oracle-backed stand-in for the per-GPU engine (the real engine is
exercised by tests/test_gpu_pedersen_sharded.py).  Also: the new C entry points refuse bad arguments, and those that
need a device fail without one."""
import ctypes as C
import dataclasses
import hashlib
import os
import socket

import numpy as np
import pytest

from oracle import pyref as o

R = 1 << 256
N = 45                                      # shard_bounds(45, 2, .): 32 and 13 proofs


class OraclePedersenShard:
    """The sharded API of ark_vrf_b200.pedersen.BatchVerifier, computed by the oracle."""

    cs_stride = 96

    def __init__(self, S, cases):
        self.S = S
        self.items = [o.pedersen_batch_prepare(S, ios, ad, pf) for ios, ad, pf in cases]

    def __len__(self):
        return len(self.items)

    def prepare_device(self):
        return any(e.pf.pk_com == o.IDENTITY or e.io_identity for e in self.items)

    def cs_stream(self):
        b = b"".join(o.enc_scalar(e.c) + o.enc_scalar(e.pf.s) + o.enc_scalar(e.pf.sb) for e in self.items)
        return np.frombuffer(b, dtype=np.uint8).reshape(-1, 96).copy()

    def partial(self, seed, first):
        S, r = self.S, self.S.r
        acc = o.EXT_ID
        g = bb = 0
        for q, e in enumerate(self.items):
            j = first + q
            blk = hashlib.sha512(seed + (j // 2).to_bytes(8, "little")).digest()
            t = int.from_bytes(blk[32 * (j % 2):32 * (j % 2) + 16], "little")
            u = int.from_bytes(blk[32 * (j % 2) + 16:32 * (j % 2) + 32], "little")
            terms = [(e.output, t * e.c % r), (e.pf.ok, t), (e.input, (-t * e.pf.s) % r), (e.pf.pk_com, u * e.c % r),
                     (e.pf.r, u)]
            g = (g + u * e.pf.s) % r
            bb = (bb + u * e.pf.sb) % r
            for P, k in terms:
                acc = o.ext_add(S, acc, o.ext_mul(S, o.to_ext(P), k))
        acc = o.ext_add(S, acc, o.ext_mul(S, o.to_ext(S.G), (-g) % r))
        acc = o.ext_add(S, acc, o.ext_mul(S, o.to_ext(S.B), (-bb) % r))
        return b"".join((c * R % S.p).to_bytes(32, "little") for c in acc)


def _combine_fn(S):
    def f(suite, blob):
        acc = o.EXT_ID
        ri = pow(R, -1, S.p)
        for k in range(len(blob) // 128):
            pt = tuple(int.from_bytes(blob[128 * k + 32 * i:128 * k + 32 * i + 32], "little") * ri % S.p for i in range(4))
            acc = o.ext_add(S, acc, pt)
        return 0 if o.ext_is_identity(S, acc) else 1
    return f


def _proofs(S, n, signers=5):
    """n Pedersen proofs of one I/O pair each: signer j % signers, input data_to_point(LE64(j) || LE32(0))."""
    sks = [o.secret_from_seed(S, o.synth_seed(k)) for k in range(signers)]
    out = []
    for j in range(n):
        inp = o.data_to_point(S, o.synth_msg(j, 0))
        ios = [(inp, o.pt_mul(S, inp, sks[j % signers]))]
        ad = b"ad-%d" % j
        out.append((ios, ad, o.pedersen_prove(S, sks[j % signers], ios, ad)[0]))
    return out


_CASES = {}


def _case(name):
    """(proof list, expected verdict) of a named case; proofs are made once per module."""
    S = o.BANDERSNATCH
    if "base" not in _CASES:
        _CASES["base"] = _proofs(S, N)
    cases = [(list(ios), ad, dataclasses.replace(pf)) for ios, ad, pf in _CASES["base"]]

    def bump(j, field):
        setattr(cases[j][2], field, (getattr(cases[j][2], field) + 1) % S.r)
    if name == "bad_s_last":
        bump(N - 1, "s")
    elif name == "bad_sb_rank0_first":
        bump(0, "sb")
    elif name == "identity_pk_com_rank1":
        cases[40][2].pk_com = o.IDENTITY
        bump(3, "s")
    elif name == "identity_input":
        ios, ad, pf = cases[20]
        cases[20] = ([(o.IDENTITY, ios[0][1])], ad, pf)
    elif name == "empty":
        cases = []
    items = [o.pedersen_batch_prepare(S, ios, ad, pf) for ios, ad, pf in cases]
    return cases, o.pedersen_batch_verify(S, items), o.pedersen_batch_seed(S, items)


def _worker(rank, world, port, cases, weights, q):
    import torch.distributed as dist
    from ark_vrf_b200 import dist as avdist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    S = o.BANDERSNATCH
    lo, hi = avdist.shard_bounds(len(cases), world, rank)
    shard = OraclePedersenShard(S, cases[lo:hi])
    seeds = []

    def seed_fn(suite, stream):
        assert stream.size == 96 * len(cases)
        seeds.append(hashlib.sha512(S.suite_id + b"\x50" + bytes(stream)).digest())
        return seeds[-1]
    try:
        st = avdist.sharded_verify(shard, 0, lo, seed_fn=seed_fn, combine_fn=_combine_fn(S), weights=weights)
    except ValueError as e:
        st = "ValueError: %s" % e
    q.put((rank, (lo, hi), st, seeds[0] if seeds else None))
    dist.barrier()
    dist.destroy_process_group()


def _run(cases, weights="reference"):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, cases, weights, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


@pytest.mark.parametrize("case,expect", [("valid", 0), ("bad_s_last", 1), ("bad_sb_rank0_first", 1),
                                         ("identity_pk_com_rank1", 2), ("identity_input", 2), ("empty", 0)])
def test_pedersen_sharded_verify_gloo_world2(case, expect):
    cases, want, seed = _case(case)
    assert want == expect
    res = _run(cases)
    if cases:
        assert [b for _, b, _, _ in res] == [(0, 32), (32, N)]           # both ranks hold proofs
    for rank, _, st, got_seed in res:
        assert st == expect, (rank, st)
        assert got_seed == seed, rank                                    # the seed both ranks agree on


def test_pedersen_tree_weights_refused_on_every_rank():
    cases, _, _ = _case("valid")
    res = _run(cases, weights="tree")
    assert len(res) == 2
    for rank, _, st, got_seed in res:
        assert isinstance(st, str) and st.startswith("ValueError") and got_seed is None, (rank, st)


# ---- C entry points without a device ------------------------------------------------------------------------------
AVRF_ERR_ARG, AVRF_ERR_NO_DEVICE = -2, -4


def _lib():
    from ark_vrf_b200 import _lib as L
    return L.load()


def _no_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")


def _err(lib):
    return lib.avrf_last_error().decode()


def test_pedersen_entry_points_refuse_bad_arguments():
    lib = _lib()
    seed = C.create_string_buffer(64)
    for suite, fmt in [(3, 0), (0, 2)]:
        assert lib.avrf_pedersen_batch_new_on(-1, suite, fmt) is None and _err(lib) == "bad suite/fmt"
        assert lib.avrf_pedersen_sharded_new(suite, fmt) is None and _err(lib) == "bad suite/fmt"
    off = (C.c_uint32 * 2)(0, 1)
    args = [bytes(128), off, None, (C.c_uint32 * 2)(0, 0)] + [bytes(64), bytes(64), bytes(64), bytes(32), bytes(32)]
    assert lib.avrf_pedersen_sharded_push_many(None, 1, *args) == AVRF_ERR_ARG and _err(lib) == "null handle"
    assert lib.avrf_pedersen_sharded_push_many(None, 0, *[None] * 9) == AVRF_ERR_ARG
    for fn in (lib.avrf_pedersen_seed, lib.avrf_pedersen_seed_dev):
        for a in [(3, bytes(96), 1, seed), (0, None, 1, seed), (0, bytes(96), 1, None)]:
            assert fn(*a) == AVRF_ERR_ARG and _err(lib) == "bad argument", (fn, a)


def test_pedersen_seed_is_a_host_hash():
    """avrf_pedersen_seed needs no device: SHA512(SUITE_ID || 0x50 || 96-byte records), for every suite."""
    from ark_vrf_b200 import pedersen as ped
    lib = _lib()
    rec = bytes(range(96)) * 3
    for sid, S in o.SUITES.items():
        out = C.create_string_buffer(64)
        assert lib.avrf_pedersen_seed(sid, rec, 3, out) == 0
        want = hashlib.sha512(S.suite_id + b"\x50" + rec).digest()
        assert out.raw == want
        assert ped.seed_of_stream(sid, np.frombuffer(rec, dtype=np.uint8).reshape(3, 96)) == want
        assert lib.avrf_pedersen_seed(sid, None, 0, out) == 0 and out.raw == hashlib.sha512(S.suite_id + b"\x50").digest()
    # the Thin seed keeps its 64-byte records
    out = C.create_string_buffer(64)
    assert lib.avrf_thin_seed(0, rec, 3, out) == 0
    assert out.raw == hashlib.sha512(o.BANDERSNATCH.suite_id + b"\x50" + rec[:192]).digest()


def test_pedersen_entry_points_need_a_device():
    _no_gpu()
    lib = _lib()
    assert lib.avrf_pedersen_batch_new_on(-1, 0, 1) is None and _err(lib).startswith("no CUDA device")
    assert lib.avrf_pedersen_sharded_new(0, 1) is None and _err(lib).startswith("no CUDA device")
    seed = C.create_string_buffer(64)
    assert lib.avrf_pedersen_seed_dev(0, None, 0, seed) == AVRF_ERR_NO_DEVICE
    from ark_vrf_b200 import _lib as L, pedersen as ped
    for make in (lambda: ped.BatchVerifier(0), lambda: ped.BatchVerifier(0, eager_seed=False, device=0),
                 lambda: ped.ShardedBatchVerifier(0)):
        with pytest.raises(L.AvrfError, match="no CUDA device"):
            make()


def test_python_record_sizes():
    """The per-class record size the sharded helpers use: Thin 64, Pedersen 96; a shard without one counts as Thin."""
    from ark_vrf_b200 import dist as avdist, pedersen as ped, thin
    assert thin.BatchVerifier.cs_stride == 64 and ped.BatchVerifier.cs_stride == 96
    assert avdist._seed_fns(64) == (thin.seed_of_stream, thin.seed_of_device_stream)
    assert avdist._seed_fns(96) == (ped.seed_of_stream, ped.seed_of_device_stream)
