"""Pedersen VRF on one GPU next to the Thin VRF, on the same synthetic workload (2^20 Bandersnatch proofs, one I/O pair
each, 4096 signers; every proof distinct).  Prints one JSON line with the device name and power limit read in the same
run.  Legs (best of --reps after a warm-up, except the latency leg):
  prove_many        avrf_pedersen_prove_many, proofs/s
  batch             push of the 2^20 proofs from pinned memory + verify, wall time, with avrf_thin_batch_timings
  sharded           the same push + verify through pedersen.ShardedBatchVerifier over every GPU of the run
                    (avrf_init_multi), wall time, with avrf_thin_sharded_timings (hash_wait_ms, host_hash_ms,
                    shard_msm_ms_max), the device count and every card's name and power limit; beside the batch leg
  drop_in           the reference's call sequence: pedersen::BatchVerifier::push once per proof through the C++ mirror
                    (tools/push_loop.cpp, heap items, Montgomery format) + verify, wall time of the push loop and of
                    verify; beside it, at 2^14 proofs (a 2^20 loop of it takes too long to repeat), the same loop with
                    each proof pushed as a one-proof push_many - what BatchVerifier::push did before single pushes were
                    staged - reported per proof
  wire              the same batch serialised once (pedersen.serialize_proofs: 160-byte records, compressed I/O pairs),
                    pushed from pinned memory through push_compressed (decoded and validated on the GPU) + verify, wall
                    time; then one more push + verify under torch.profiler for the device time of the decode kernels
  verify_each       avrf_pedersen_batch_verify_each over the batch, proofs/s
  verify_one        median latency of 200 avrf_pedersen_verify_one calls
  thin_prove_many / thin_verify_each   the same two legs of the Thin VRF on its batch of the same size
Usage: python tools/bench_pedersen.py [--log2n 20] [--reps 5]"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def device_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    name, power = (x.strip() for x in out.stdout.strip().split(",")) if out.returncode == 0 else ("unknown", "unknown")
    return name, power


def cards():
    """(name, power limit) of every GPU of the run, read now."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True)
    if out.returncode != 0:
        return []
    return [[x.strip() for x in line.split(",")] for line in out.stdout.strip().splitlines()]


def best(fn, reps):
    fn()                                   # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts)


DECODE_KERNELS = ("k_ped_wire_unpack", "k_dec_prep", "k_batch_inv", "k_dec_finish", "k_ped_proof_ok", "k_scalars_to_mont")


def decode_kernel_ms(fn):
    """Device time (ms) of the wire decode kernels during one call of fn, from torch.profiler's CUDA activity records,
    per kernel and in total."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            k = next((k for k in DECODE_KERNELS if k in ev.name), None)
            if k:
                per[k] = per.get(k, 0.0) + ev.device_time_total / 1e3
    out = {k: round(v, 3) for k, v in per.items()}
    out["total"] = round(sum(per.values()), 3)
    return out


def drop_in(b, n, reps):
    """The `drop_in` leg: best of `reps` push loops + verify after a warm-up, and the one-proof push_many loop."""
    import numpy as np
    from ark_vrf_b200 import Format, synth
    pl = ctypes.CDLL(os.path.join(ROOT, "tools", "libavrf_pushloop.so"))
    pl.avrf_pushloop_ped_new.restype = ctypes.c_void_p
    pl.avrf_pushloop_ped_new.argtypes = [ctypes.c_uint64] + [ctypes.c_void_p] * 9
    pl.avrf_pushloop_ped_step.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int,
                                          ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    pl.avrf_pushloop_ped_free.argtypes = [ctypes.c_void_p]
    # the batch leg's statements, proven again with the points and scalars as arkworks values lie in memory
    mb = synth.make_pedersen_batch(b.suite, n, 1, 4096, Format.MONTGOMERY)
    arrs = [np.ascontiguousarray(x) for x in (mb.ios, mb.io_offsets, mb.ad_blob, mb.ad_offsets, mb.pk_com, mb.r, mb.ok,
                                              mb.s, mb.sb)]
    h = pl.avrf_pushloop_ped_new(n, *[x.ctypes.data for x in arrs])
    assert h
    pm, vm = ctypes.c_double(0), ctypes.c_double(0)

    def step(n_items, one_by_one_many):
        assert pl.avrf_pushloop_ped_step(h, n_items, one_by_one_many, ctypes.byref(pm), ctypes.byref(vm)) == 0
        return pm.value, vm.value
    try:
        runs = [step(0, 0) for _ in range(reps + 1)][1:]
        push_ms, verify_ms = min(runs, key=sum)
        n_old = min(n, 1 << 14)
        old = [step(n_old, 1) for _ in range(3)][1:]
        new = [step(n_old, 0) for _ in range(3)][1:]
    finally:
        pl.avrf_pushloop_ped_free(h)
    return {"n": n, "push_loop_ms": round(push_ms, 2), "verify_ms": round(verify_ms, 2),
            "total_ms": round(push_ms + verify_ms, 2), "proofs_per_s": round(n / ((push_ms + verify_ms) * 1e-3)),
            "one_proof_push_many": {"n": n_old, "push_us_per_proof": round(1e3 * min(p for p, _ in old) / n_old, 2),
                                    "staged_push_us_per_proof": round(1e3 * min(p for p, _ in new) / n_old, 3)}}


def sharded(arrs, n, reps, batch_ms):
    """The `sharded` leg: best of `reps` clear + push_many + verify of the batch over every GPU after a warm-up, and the
    sharded timings of that best run."""
    import torch
    import ark_vrf_b200 as av
    from ark_vrf_b200 import pedersen as ped
    nd = av.init_multi(torch.cuda.device_count())
    sh = ped.ShardedBatchVerifier(0, av.Format.CANONICAL)
    status, runs = [], []

    def run():
        t0 = time.perf_counter()
        sh.clear()
        sh.push_many(*arrs)
        status.append(sh.verify_status())
        runs.append((time.perf_counter() - t0, sh.timings()))
    run()                                  # warm-up
    runs.clear()
    for _ in range(reps):
        run()
    assert set(status) == {0}, status
    t, tm = min(runs, key=lambda x: x[0])
    sh.close()
    return {"devices": nd, "cards": cards(), "n": n, "push_verify_ms": round(1e3 * t, 2), "proofs_per_s": round(n / t),
            "hash_wait_ms": round(tm["hash_wait_ms"], 2), "host_hash_ms": round(tm["host_hash_ms"], 2),
            "shard_msm_ms_max": round(tm["shard_msm_ms_max"], 3), "batch_push_verify_ms": batch_ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import numpy as np
    import torch
    import ark_vrf_b200 as av
    from ark_vrf_b200 import _lib, ops, pedersen as ped, synth
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU only")
    lib = av.load()
    _lib.check(lib.avrf_init(0))
    n, F, sid = 1 << a.log2n, av.Format.CANONICAL, 0
    name, power = device_info()
    res = {"device": name, "power_limit": power, "n": n, "m": 1, "signers": 4096, "suite": "bandersnatch"}

    b = synth.make_pedersen_batch(sid, n, 1, 4096, F)
    t = best(lambda: ops.pedersen_prove_many(sid, b.sk, b.pk, b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, F), a.reps)
    res["prove_many_proofs_per_s"] = round(n / t)

    def pin(x):
        p = torch.empty(x.shape, dtype=torch.uint8, pin_memory=True) if x.dtype == np.uint8 else \
            torch.empty(x.shape, dtype=torch.int32, pin_memory=True)
        p.numpy()[...] = x.view(np.uint8) if x.dtype == np.uint8 else x.view(np.int32)
        return p
    arrs = [pin(x) for x in (b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.pk_com, b.r, b.ok, b.s, b.sb)]
    bv = ped.BatchVerifier(sid, F)
    status = []

    def batch():
        bv.clear()
        bv.push_many(*arrs)
        status.append(bv.verify_status())
    t = best(batch, a.reps)
    assert set(status) == {0}, status
    tm = _lib.Timings()
    _lib.check(lib.avrf_thin_batch_timings(bv._h, ctypes.byref(tm)))
    res["batch_push_verify_ms"] = round(1e3 * t, 2)
    res["batch_proofs_per_s"] = round(n / t)
    res["batch_timings"] = {k: (round(v, 3) if isinstance(v, float) else v) for k, v in tm.as_dict().items()}
    res["sharded"] = sharded(arrs, n, a.reps, res["batch_push_verify_ms"])
    res["drop_in"] = drop_in(b, n, a.reps)

    # wire format: what callers hold before Proof::deserialize_compressed
    nio = int(b.io_offsets[n])
    ios32 = np.concatenate([ops.point_compress(sid, b.ios[:nio].reshape(-1, 64), F).reshape(-1), np.zeros(64, np.uint8)])
    recs = ped.serialize_proofs(sid, b.pk_com, b.r, b.ok, b.s, b.sb, F)
    warrs = [pin(x) for x in (ios32, b.io_offsets, b.ad_blob, b.ad_offsets, recs)]
    wv = ped.BatchVerifier(sid, F)
    wstatus = []

    def wire():
        wv.clear()
        assert wv.push_compressed(*warrs).all()
        wstatus.append(wv.verify_status())
    t = best(wire, a.reps)
    assert set(wstatus) == {0}, wstatus
    res["wire_push_verify_ms"] = round(1e3 * t, 2)
    res["wire_proofs_per_s"] = round(n / t)
    res["wire_bytes_per_proof"] = int((recs.nbytes + 64 * nio) // n)
    res["wire_decode_kernels_ms"] = decode_kernel_ms(wire)

    each = []
    t = best(lambda: each.append(bv.verify_each()), a.reps)
    assert all((e == 0).all() for e in each)
    res["verify_each_proofs_per_s"] = round(n / t)

    pf = ped.Proof(bytes(b.pk_com[0]), bytes(b.r[0]), bytes(b.ok[0]), bytes(b.s[0]), bytes(b.sb[0]))
    ios, ad = bytes(b.ios[0]), bytes(b.ad_blob[b.ad_offsets[0]:b.ad_offsets[1]])
    lat = []
    for i in range(201):
        t0 = time.perf_counter()
        ped.verify(sid, ios, ad, pf, F)
        if i:
            lat.append(time.perf_counter() - t0)
    res["verify_one_median_us"] = round(1e6 * statistics.median(lat), 1)

    tb = synth.make_batch(sid, n, 1, 4096, F)
    t = best(lambda: ops.thin_prove_many(sid, tb.sk, tb.pk, tb.ios, tb.io_offsets, tb.ad_blob, tb.ad_offsets, F), a.reps)
    res["thin_prove_many_proofs_per_s"] = round(n / t)
    tv = av.BatchVerifier(sid, F)
    tv.push_many(tb.pk, tb.ios, tb.io_offsets, tb.ad_blob, tb.ad_offsets, tb.r, tb.s)
    t = best(lambda: tv.verify_each(), a.reps)
    res["thin_verify_each_proofs_per_s"] = round(n / t)
    res["prove_ratio_pedersen_over_thin"] = round(res["thin_prove_many_proofs_per_s"] / res["prove_many_proofs_per_s"], 2)
    res["verify_each_ratio_pedersen_over_thin"] = round(res["thin_verify_each_proofs_per_s"] /
                                                        res["verify_each_proofs_per_s"], 2)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
