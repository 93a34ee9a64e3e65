"""GPU: one Pedersen VRF batch over several GPUs (pedersen.rs:255-427).  The per-handle building blocks of a batch spread
over processes (prepare, 96-byte batch-seed stream, partial at a global first index, combine) against one handle and the
oracle; the in-library multi-GPU path (avrf_pedersen_sharded_*) against one handle (nd = 1 on a one-GPU box, N under a
multi-GPU run); a 2^20-proof batch; NCCL across two processes; the C++ mirror."""
import hashlib
import os
import socket
import struct
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import pyref as o
from helpers import pt_bytes, pt_from_bytes, sc_bytes

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
RINV = {sid: pow(1 << 256, -1, S.p) for sid, S in o.SUITES.items()}


@pytest.fixture(scope="module")
def av():
    import ark_vrf_b200 as a
    a.load().avrf_init(0)
    return a


def _args(b):
    return (b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.pk_com, b.r, b.ok, b.s, b.sb)


def _slice(b, lo, hi, **change):
    """push_many arguments of proofs [lo, hi) of a synthetic Pedersen batch (canonical), columns replaced by `change`."""
    cols = {k: change.get(k, getattr(b, k)) for k in ("pk_com", "r", "ok", "s", "sb")}
    io0, io1 = int(b.io_offsets[lo]), int(b.io_offsets[hi])
    ad0, ad1 = int(b.ad_offsets[lo]), int(b.ad_offsets[hi])
    return (np.ascontiguousarray(np.concatenate([b.ios[io0:io1], np.zeros((1, 128), np.uint8)])),
            (b.io_offsets[lo:hi + 1] - io0).astype(np.uint32),
            np.concatenate([b.ad_blob[ad0:ad1], np.zeros(16, np.uint8)]), (b.ad_offsets[lo:hi + 1] - ad0).astype(np.uint32),
            *[np.ascontiguousarray(cols[k][lo:hi]) for k in ("pk_com", "r", "ok", "s", "sb")])


def _bumped(S, arr, *rows):
    """A copy of a (n, 32) scalar column with scalar + 1 (mod r) at `rows`: still a field element, in either format."""
    out = arr.copy()
    for j in rows:
        v = (int.from_bytes(out[j].tobytes(), "little") + 1) % S.r
        out[j] = np.frombuffer(v.to_bytes(32, "little"), dtype=np.uint8)
    return out


def _ext(sid, part):
    """A 128-byte partial (Montgomery extended X, Y, Z, T) as oracle extended coordinates."""
    part = bytes(part)
    return tuple(int.from_bytes(part[32 * i:32 * i + 32], "little") * RINV[sid] % o.SUITES[sid].p for i in range(4))


def _same(S, P, Q):
    return o.ext_is_identity(S, o.ext_add(S, P, o.ext_neg(S, Q)))


def _oracle_items(S, b, s, sb):
    items = []
    for j in range(b.n):
        ios = [(pt_from_bytes(b.ios[k][:64]), pt_from_bytes(b.ios[k][64:]))
               for k in range(int(b.io_offsets[j]), int(b.io_offsets[j + 1]))]
        ad = bytes(b.ad_blob[int(b.ad_offsets[j]):int(b.ad_offsets[j + 1])])
        pf = o.PedersenProof(pt_from_bytes(b.pk_com[j]), pt_from_bytes(b.r[j]), pt_from_bytes(b.ok[j]),
                             int.from_bytes(s[j].tobytes(), "little"), int.from_bytes(sb[j].tobytes(), "little"))
        items.append(o.pedersen_batch_prepare(S, ios, ad, pf))
    return items


def _oracle_cut_msm(S, items, seed, lo, hi):
    """The cut [lo, hi)'s share of the 5N+2-point MSM of pedersen.rs:373-418 under the whole batch's weights."""
    bases, scalars, g, bb, r = [], [], 0, 0, S.r
    for j in range(lo, hi):
        e = items[j]
        blk = hashlib.sha512(seed + (j // 2).to_bytes(8, "little")).digest()
        t = int.from_bytes(blk[32 * (j % 2):32 * (j % 2) + 16], "little")
        u = int.from_bytes(blk[32 * (j % 2) + 16:32 * (j % 2) + 32], "little")
        bases += [e.output, e.pf.ok, e.input, e.pf.pk_com, e.pf.r]
        scalars += [t * e.c % r, t, (-(t * e.pf.s)) % r, u * e.c % r, u]
        g, bb = (g + u * e.pf.s) % r, (bb + u * e.pf.sb) % r
    return o.msm(S, bases + [S.G, S.B], scalars + [(-g) % r, (-bb) % r])


# ---- 1. building blocks on one GPU -------------------------------------------------------------------------------
@pytest.mark.parametrize("sid", [0, 1, 2])
@pytest.mark.parametrize("m", [0, 1, 3])
def test_building_blocks_at_uneven_cuts(av, sid, m):
    """Cuts at 13 (odd: splits the two-proof weight block of proofs 12 and 13) and 38 (not a multiple of 32), each in its
    own eager_seed=False handle: the concatenated 96-byte streams hash (host and device) to the whole handle's seed and
    the oracle's; each cut's partial at its global first index is the oracle's MSM of its terms; its SCALARS are the
    whole batch's at the global positions; the partials add up to the whole handle's PARTIAL and combine to its verdict."""
    import torch
    from ark_vrf_b200 import pedersen as ped, synth, thin
    S, F, n = o.SUITES[sid], av.Format.CANONICAL, 70
    cuts = [0, 13, 38, n]
    b = synth.make_pedersen_batch(sid, n, m, signers=5, fmt=F)
    for variant, want in (("valid", 0), ("bad_sb", 1)):
        sb = _bumped(S, b.sb, 20) if variant == "bad_sb" else b.sb
        whole = ped.BatchVerifier(sid, F)
        whole.push_many(*_slice(b, 0, n, sb=sb))
        assert whole.verify_status() == want
        seed = bytes(whole.tap(av.Tap.SEED))
        scal = whole.tap(av.Tap.SCALARS).reshape(-1, 32)
        whole_partial = _ext(sid, whole.tap(av.Tap.PARTIAL))
        w_all = whole.tap(av.Tap.W).reshape(-1, 32)
        items = _oracle_items(S, b, b.s, sb)
        assert seed == o.pedersen_batch_seed(S, items)
        parts, streams = [], []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            h = ped.BatchVerifier(sid, F, eager_seed=False)
            h.push_many(*_slice(b, lo, hi, sb=sb))
            assert h.prepare_device() is False
            cs = h.cs_stream()
            assert cs.shape == (hi - lo, 96)
            streams.append(cs)
            parts.append((h, lo, hi))
        stream = np.ascontiguousarray(np.concatenate(streams))
        assert ped.seed_of_stream(sid, stream) == seed
        dev = torch.from_numpy(stream.reshape(-1)).cuda(0)
        torch.cuda.synchronize(0)
        assert ped.seed_of_device_stream(sid, dev.data_ptr(), n) == seed
        acc, blobs = o.EXT_ID, []
        for h, lo, hi in parts:
            p = h.partial(seed, lo)
            blobs.append(p)
            P = _ext(sid, p)
            assert _same(S, P, _oracle_cut_msm(S, items, seed, lo, hi)), (variant, lo)
            acc = o.ext_add(S, acc, P)
            cs = h.tap(av.Tap.SCALARS).reshape(-1, 32)
            assert cs.shape[0] == 5 * (hi - lo) + 2
            assert (cs[:5 * (hi - lo)] == scal[5 * lo:5 * hi]).all(), (variant, lo)
            assert (h.tap(av.Tap.W).reshape(-1, 32) == w_all[lo:hi]).all()
        assert _same(S, acc, whole_partial)
        assert thin.combine_partials(sid, b"".join(blobs)) == want


# ---- 2. the in-library multi-GPU path ----------------------------------------------------------------------------
@pytest.mark.parametrize("sid,m,n", [(0, 1, 5001), (2, 3, 701), (1, 0, 301)])
def test_sharded_in_library(av, sid, m, n):
    import torch
    from ark_vrf_b200 import pedersen as ped, synth
    S, F = o.SUITES[sid], av.Format.CANONICAL
    nd = av.init_multi(torch.cuda.device_count())
    assert nd == torch.cuda.device_count()
    b = synth.make_pedersen_batch(sid, n, m, signers=16, fmt=F)
    one = ped.BatchVerifier(sid, F)
    one.push_many(*_args(b))
    assert one.verify_status() == 0
    seed = bytes(one.tap(av.Tap.SEED))
    w_all = one.tap(av.Tap.W).reshape(n, 32)
    sh = ped.ShardedBatchVerifier(sid, F)
    assert sh.devices == nd
    sh.push_many(*_args(b))
    assert len(sh) == n
    assert sh.verify_status() == 0
    assert sh.seed() == seed == hashlib.sha512(S.suite_id + b"\x50" + one.cs_stream().tobytes()).digest()
    per = ((n + nd - 1) // nd + 31) // 32 * 32
    bounds = [(min(n, d * per), min(n, d * per + per)) for d in range(nd)]
    for d, (lo, hi) in enumerate(bounds):
        if hi > lo:
            v = sh.shard(d)
            assert len(v) == hi - lo
            assert (v.tap(av.Tap.W).reshape(-1, 32) == w_all[lo:hi]).all()
    assert sh.verify_status() == 0                # repeatable
    assert sh.timings()["total_ms"] > 0
    # faults in s and in sb at the first and last proof of every shard
    edges = sorted({x for lo, hi in bounds if hi > lo for x in (lo, hi - 1)})
    for col in ("s", "sb"):
        for pos in edges:
            sh.clear()
            sh.push_many(*_slice(b, 0, n, **{col: _bumped(S, getattr(b, col), pos)}))
            assert sh.verify_status() == 1, (col, pos)
    # the faulty proof named by its device's verify_each, at its local index
    pos = edges[-1]
    for d, (lo, hi) in enumerate(bounds):
        if hi > lo:
            st = sh.shard(d).verify_each()
            assert list(np.nonzero(st)[0]) == ([pos - lo] if lo <= pos < hi else []), d
    # InvalidData takes precedence over a bad response
    pk2 = b.pk_com.copy()
    pk2[n - 1] = synth.identity_point(sid, F)
    sh.clear()
    sh.push_many(*_slice(b, 0, n, pk_com=pk2, s=_bumped(S, b.s, 0)))
    assert sh.verify_status() == 2
    # the same batch in three pushes of odd sizes: several runs of global indices per device, odd run starts
    c1 = (n // 3) | 1
    cuts = [0, c1, c1 + 17, n]
    assert all((hi - lo) % 2 == 1 for lo, hi in zip(cuts[:-1], cuts[1:]))
    for s_col, want in ((b.s, 0), (_bumped(S, b.s, c1 + 5), 1)):
        sh.clear()
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            sh.push_many(*_slice(b, lo, hi, s=s_col))
        assert len(sh) == n
        assert sh.verify_status() == want
        if want == 0:
            assert sh.seed() == seed
    # empty batch, clear
    sh.clear()
    assert len(sh) == 0 and sh.verify_status() == 0
    # scheme mismatches are refused and leave the handle's proofs and seed as they were
    lib = av.load()
    sh.push_many(*_args(b))
    assert sh.verify_status() == 0
    tb = synth.make_batch(sid, 64, 1, signers=4, fmt=F)
    targs = (tb.pk, tb.ios, tb.io_offsets, tb.ad_blob, tb.ad_offsets, tb.r, tb.s)
    from ark_vrf_b200.thin import ptr
    rc = lib.avrf_thin_sharded_push_many(sh._h, 64, *[ptr(x) for x in targs])
    assert rc == -2 and b"not a Thin-VRF sharded batch" == lib.avrf_last_error()
    assert len(sh) == n and sh.seed() == seed
    th = av.ShardedBatchVerifier(sid, F)
    th.push_many(*targs)
    assert th.verify_status() == 0
    tseed = th.seed()
    rc = lib.avrf_pedersen_sharded_push_many(th._h, n, *[ptr(x) for x in _args(b)])
    assert rc == -2 and b"not a Pedersen sharded batch" == lib.avrf_last_error()
    assert len(th) == 64 and th.seed() == tseed
    assert th.verify_status() == 0 and sh.verify_status() == 0
    th.close()
    sh.close()


# ---- 3. full size ------------------------------------------------------------------------------------------------
def test_sharded_full_size(av):
    """2^20 Bandersnatch proofs (M = 1, 4096 signers): the large sort path on every device."""
    import torch
    from ark_vrf_b200 import pedersen as ped, synth
    S, F, n = o.BANDERSNATCH, av.Format.CANONICAL, 1 << 20
    av.init_multi(torch.cuda.device_count())
    b = synth.make_pedersen_batch(0, n, 1, signers=4096, fmt=F)
    sh = ped.ShardedBatchVerifier(0, F)
    sh.push_many(*_args(b))
    assert sh.verify_status() == 0
    sh.clear()
    sh.push_many(*_slice(b, 0, n, s=_bumped(S, b.s, n - 1)))
    assert sh.verify_status() == 1
    sh.close()


# ---- 4. NCCL: one process per GPU --------------------------------------------------------------------------------
def _nccl_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import ark_vrf_b200 as a
    from ark_vrf_b200 import dist as avdist, pedersen as ped, synth
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    a._lib.check(a.load().avrf_init(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    S, F, n = o.BANDERSNATCH, a.Format.MONTGOMERY, 4096 + 64
    lo, hi = avdist.shard_bounds(n, world, rank)
    b = synth.make_pedersen_batch(0, hi - lo, 1, fmt=F, first=lo)
    res = {}
    for case in ("valid", "bad_s_last_rank", "identity_pk_com_rank0"):
        s, pk = b.s, b.pk_com.copy()
        if case == "bad_s_last_rank" and rank == world - 1:
            s = _bumped(S, b.s, hi - lo - 1)
        if case == "identity_pk_com_rank0" and rank == 0:
            pk[0] = synth.identity_point(0, F)
        bv = ped.BatchVerifier(0, F, eager_seed=False)
        bv.push_many(b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, pk, b.r, b.ok, s, b.sb)
        res[case] = avdist.sharded_verify(bv, 0, lo, device=dev)
    try:
        avdist.sharded_verify(bv, 0, lo, device=dev, weights="tree")
        res["tree"] = "no error"
    except ValueError:
        res["tree"] = "ValueError"
    q.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_verify_nccl():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [q.get(timeout=600) for _ in range(2)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, res in out:
        assert res == {"valid": 0, "bad_s_last_rank": 1, "identity_pk_com_rank0": 2, "tree": "ValueError"}, (rank, res)


# ---- 5. C++ ------------------------------------------------------------------------------------------------------
def test_cpp_pedersen_sharded_driver(av):
    """include/avrf.hpp's ark_vrf::pedersen::ShardedBatchVerifier through a compiled driver, on every GPU of the box."""
    import torch
    S = o.BANDERSNATCH
    sks = [o.secret_from_seed(S, o.synth_seed(k)) for k in range(3)]
    blob = b""
    count = 0
    for j, m in enumerate([1, 1, 0, 2, 1, 3]):
        ios = []
        for i in range(m):
            inp = o.data_to_point(S, o.synth_msg(j, i))
            ios.append((inp, o.pt_mul(S, inp, sks[j % 3])))
        ad = b"cpp-%d" % j
        pf, _ = o.pedersen_prove(S, sks[j % 3], ios, ad)
        blob += struct.pack("<I", len(ios)) + b"".join(pt_bytes(a) + pt_bytes(x) for a, x in ios)
        blob += struct.pack("<I", len(ad)) + ad
        blob += pt_bytes(pf.pk_com) + pt_bytes(pf.r) + pt_bytes(pf.ok) + sc_bytes(pf.s) + sc_bytes(pf.sb)
        count += 1
    blob = struct.pack("<I", count) + blob
    root = os.path.dirname(HERE)
    with tempfile.TemporaryDirectory() as d:
        exe, data = os.path.join(d, "pedersen_sharded_driver"), os.path.join(d, "proofs.bin")
        open(data, "wb").write(blob)
        lib = os.path.join(root, "ark_vrf_b200")
        subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"),
                               os.path.join(HERE, "cpp", "pedersen_sharded_driver.cpp"), "-o", exe,
                               "-L", lib, "-l:libavrf_gpu.so", "-Wl,-rpath," + lib])
        out = subprocess.run([exe, data], capture_output=True, text=True, timeout=600)
        print(out.stdout, out.stderr)
        assert out.returncode == 0 and "ALL OK" in out.stdout
        assert "devices: %d" % torch.cuda.device_count() in out.stdout
