#!/usr/bin/env python3
"""bench.py - Bandersnatch thin-VRF batch-verified proofs/sec on B200 (BASELINE.json metric).

A step = one pass of the hot path (BatchVerifier push/prepare + verify, reference src/thin.rs:209-325) over ONE
batch of 2^20 synthetic proofs (SURVEY.md 8d, BASELINE.json configs[1]).  The reference seeds every batch with one
serial SHA-512 over all its (c_j, s_j) (thin.rs:273-279): ~82 ms on one host core per 2^20-proof batch, against
~12 ms of GPU work.  A verifier that serves traffic therefore keeps several batches in flight - each batch's hash
on its own core (bit-identical weights), the kernels of all batches sharing the GPU - and that is what the headline
measures; the one-batch-at-a-time figures are reported beside it (`single_batch`).

  value  : proofs/s, K steps over T batch handles whose inputs are resident in HBM (every step redoes prepare +
           seed + MSM), T host threads
  e2e    : proofs/s, K steps through the library's batch server (avrf_server_*) from pinned HOST buffers: H2D of
           every batch and D2H of its (c,s) stream / verdict inside the timed region
  single_batch : one handle, one batch at a time: resident, e2e (push_many) and the drop-in shape of the
           reference's own bench (benches/thin.rs:76-88: BatchVerifier::push per proof through the C++ mirror)
  roofline     : the dominant kernel (k_accumulate) against the integer-multiply peak measured live
  configs      : BASELINE.json configs[2..4] at their stated sizes
  cpu_baseline : the C port of the reference algorithm on the box's host cores, bounded sample

Every leg above that is timed per batch runs K = --steps steps, one batch each (configs[2..3] too); configs[4] is one
pass over its 2^24 inputs and `verify_one_us` the mean of 30 single-proof calls.

--dump-outputs DIR : after the timed steps of `value`, what its last step computed goes to DIR/<name>.npy (float32 /
                   float64; rank 0's batch): the verdict, the batch seed, and the challenges c_j and delinearization
                   scalars z_j of a fixed sample of 2^16 proofs.  The inputs are fixed by the arguments, so two builds
                   can be compared output for output.
--impl reference : that CPU port timed alone on the same config (the reference is Rust on un-vendored crates and
                   cannot be built in this image; DESIGN.md section 2).
--gpus N (torchrun): every rank serves whole batches on its own GPU (independent batches: no data-path
                   collective), scaling "weak"; one batch sharded over the N GPUs is reported as `sharded`.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree it runs from as it found it (it may be read-only)

import numpy as np  # noqa: E402

# canonical algorithmic work (SURVEY.md 8d): wide MACs (32x32->64 multiply-accumulate)
MM_MACS = 136                      # one 8x32-limb Montgomery multiplication
CANON_MM_PER_ADD = 7
METRIC = "bandersnatch_thin_vrf_batch_verified_proofs_per_sec"


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


def workload_name(log2n):
    return "Bandersnatch thin-VRF batch verify, 2^%d synthetic proofs (M=1, 4096 signers), BASELINE.json configs[1]" % log2n


DUMP_SAMPLE = 1 << 16


def dump_outputs(out_dir, h, status):
    """What the step `h` last ran computed, as DIR/<name>.npy: the verdict `BatchVerifier.verify` reports, the batch
    seed, and for a fixed sample of proofs the challenges c_j and delinearization scalars z_j (the C and Z taps; one row
    of bytes per proof).  Bytes are stored as float32, under 9 MB in all."""
    from ark_vrf_b200 import Tap
    os.makedirs(out_dir, exist_ok=True)
    n = len(h)
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    arrays = {
        "verdict": np.array([status], dtype=np.float64),
        "seed": h.tap(Tap.SEED).astype(np.float32),
        "sample_index": idx.astype(np.float64),
        "challenge_c": h.tap(Tap.C).reshape(n, 16)[idx].astype(np.float32),
        "delinearization_z": h.tap(Tap.Z).reshape(n, -1)[idx].astype(np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[bench] outputs of the last timed step -> {out_dir}: " + ", ".join(f"{k} {a.shape}" for k, a in arrays.items()))


def cpu_reference_arm(args, rank):
    """--impl reference: the CPU port of thin::BatchVerifier (oracle/avrf_oracle.c) on all host threads, the SAME
    config as the GPU arm: every step prepares and verifies one whole 2^log2n-proof batch."""
    if rank != 0:
        return
    from oracle import corc
    T = host_threads()
    n = 1 << args.log2n
    t0 = time.perf_counter()
    arrs = corc.synth_batch(0, n, 1, signers=4096, nthreads=T)
    gen_s = time.perf_counter() - t0
    log(f"[reference] generated 2^{args.log2n} proofs with the CPU port in {gen_s:.1f}s on {T} threads")
    for _ in range(args.warmup):
        st, _, _ = corc.thin_batch_verify(0, *arrs, nthreads=T)
        assert st == 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st, _, _ = corc.thin_batch_verify(0, *arrs, nthreads=T)
        assert st == 0
    dt = (time.perf_counter() - t0) / args.steps
    v = n / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v,
        "unit": "proofs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(args.log2n), "suite": "Bandersnatch-SHA512-ELL2-v1", "batch": n, "io_pairs": 1},
        "cpu_baseline": {"value": v, "unit": "proofs/s", "cores": T, "kind": "port",
                         "sample": f"whole 2^{args.log2n}-proof batch per step, prepare+verify, {T} threads"},
        "e2e": {"value": v, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--cpu-sample-log2n", type=int, default=18)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[2..4] block")
    ap.add_argument("--concurrency", type=int, default=0, help="batches in flight per GPU (0: from the host cores)")
    ap.add_argument("--stagger-ms", type=float, default=-1.0,
                    help="resident leg: handle i starts its first step i x this many ms after the burst begins (-1: automatic)")
    ap.add_argument("--e2e-own", type=int, default=-1, help="experiment: own-thread workers of the e2e server")
    ap.add_argument("--e2e-hashers", type=int, default=-1, help="experiment: shared multi-buffer threads of the e2e server")
    ap.add_argument("--hashers", type=int, default=-1,
                    help="shared multi-buffer SHA-512 threads per GPU for the e2e leg (0: one hashing core per worker; "
                         "-1: 0 when the rank has a core per worker, else up to 3 with 8 workers each)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        cpu_reference_arm(args, rank)
        return

    import torch
    import ark_vrf_b200 as av
    from ark_vrf_b200 import dist as avdist, ops, synth
    lib = av.load()
    av._lib.check(lib.avrf_init(local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    n = 1 << args.log2n
    cores = max(1, host_threads() // world)
    # ---- synthetic workload: every rank owns a whole batch (proofs rank*n ...), generated on its GPU ----------
    t0 = time.perf_counter()
    b = synth.make_batch(0, n, 1, signers=4096, fmt=av.Format.MONTGOMERY, first=rank * n)
    gen_s = time.perf_counter() - t0

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    host = [pin(x) for x in (b.pk, b.ios, b.io_offsets, b.ad_blob, b.ad_offsets, b.r, b.s)]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host)

    # ---- integer-multiply peak, measured live (roofline denominator) ---------------------------
    peak_wide = max(ops.microbench(0, 4096)[0] for _ in range(3))
    peak_carry = max(ops.microbench(3, 4096)[0] for _ in range(3))

    bv = av.BatchVerifier(0, av.Format.MONTGOMERY)
    bv.push_many(*host)
    stream = torch.cuda.ExternalStream(bv.stream, device=dev)     # the stream this handle's kernels run on

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, others=()):
        """`steps` steps bracketed by CUDA events on the first handle's stream, barrier + synchronize on both sides,
        max over ranks; `others`: further handles whose streams the closing event must wait for."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = fn()
        for h in others:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.ExternalStream(h.stream, device=dev))
            stream.wait_event(ev)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, out

    # ---- reject legs, before any timing: the verifier must say no at full size, on every rank count ----------
    s_bad = host[6].clone()
    s_bad[n - 1, 0] ^= 1
    pk_id = host[0].clone()
    pk_id[0] = torch.from_numpy(synth.identity_point(0, av.Format.MONTGOMERY))
    rej = av.BatchVerifier(0, av.Format.MONTGOMERY)
    rej.push_many(host[0], host[1], host[2], host[3], host[4], host[5], s_bad)
    st_bad = rej.verify_status()
    rej.clear()
    rej.push_many(pk_id, host[1], host[2], host[3], host[4], host[5], s_bad)     # identity pk AND a bad response
    st_id = rej.verify_status()
    assert (st_bad, st_id) == (1, 2), (st_bad, st_id)
    rejects = {"bad_s_last_proof": st_bad, "identity_pk_and_bad_s": st_id}
    sharded = None
    if world > 1:
        # one 2^log2n batch sharded over the ranks (contiguous shards; NCCL all-gather of (c,s) + 130-byte partials)
        lo, hi = avdist.shard_bounds(n, world, rank)
        shv = av.BatchVerifier(0, av.Format.MONTGOMERY, eager_seed=False)
        # the sharded batch is proofs 0 .. n-1 of the synthetic set: every rank generates its own shard on its GPU
        bs = synth.make_batch(0, hi - lo, 1, signers=4096, fmt=av.Format.MONTGOMERY, first=lo)

        def shard_of(pk_arr, s_arr):
            return (pk_arr, bs.ios, bs.io_offsets, bs.ad_blob, bs.ad_offsets, bs.r, s_arr)
        s_bad2 = bs.s.copy()
        if rank == world - 1:
            s_bad2[hi - lo - 1, 0] ^= 1                   # the last rank's last proof
        pk_id2 = bs.pk.copy()
        if rank == 0:
            pk_id2[0] = synth.identity_point(0, av.Format.MONTGOMERY)      # rank 0's first proof
        res = []
        for pk_arr, s_arr in ((bs.pk, bs.s), (bs.pk, s_bad2), (pk_id2, s_bad2)):
            shv.clear()
            shv.push_many(*shard_of(pk_arr, s_arr))
            res.append(avdist.sharded_verify(shv, 0, lo, device=dev))
        assert res == [0, 1, 2], res
        rejects["sharded_%d_gpus" % world] = {"valid": res[0], "bad_s_last_rank_last_proof": res[1], "identity_pk_rank0": res[2]}
        shv.clear()
        shv.push_many(*shard_of(bs.pk, bs.s))
        sh_t = []

        def step_sharded():
            shv.invalidate()
            td = {}
            assert avdist.sharded_verify(shv, 0, lo, device=dev, timings=td) == 0
            sh_t.append(td)
        for _ in range(2):
            step_sharded()
        k_sh = args.steps
        ms_sh, _ = timed(lambda: [step_sharded() for _ in range(k_sh)], k_sh, others=[shv])
        sharded = {"ms_per_batch": round(ms_sh, 3), "proofs_per_s": n / (ms_sh * 1e-3), "scaling": "strong",
                   "phases_ms": {k.replace("_s", ""): round(1e3 * float(np.mean([t[k] for t in sh_t[-k_sh:]])), 3)
                                 for k in ("prepare_s", "gather_s", "hash_s", "partial_s", "gather2_s", "combine_s")},
                   "note": "ONE batch over %d GPUs; bound by the serial SHA-512 of thin.rs:273-279" % world}
        shv.close()
    rej.close()
    log("[bench] reject legs ok:", json.dumps(rejects))

    # ---- single batch at a time (one handle): resident, e2e, roofline inputs -----------------------------------
    def step_resident():
        bv.invalidate()                      # redo prepare too: the whole path, inputs resident in HBM
        assert bv.verify_status() == 0
        return bv.timings()

    def step_e2e():
        bv.clear()
        bv.push_many(*host)                  # H2D from pinned host memory
        assert bv.verify_status() == 0
    k1 = args.steps
    for _ in range(3):
        step_resident()
    ms_one, tms = timed(lambda: [step_resident() for _ in range(k1)], k1)
    for _ in range(2):
        step_e2e()
    ms_one_e2e, _ = timed(lambda: [step_e2e() for _ in range(k1)], k1)

    # thin::Verifier::verify of ONE proof (the exact equation; latency-bound on a GPU)
    p0 = [bytes(host[0][0].numpy()), bytes(host[1][0].numpy()), bytes(host[3][:int(host[4][1])].numpy()), bytes(host[5][0].numpy()),
          bytes(host[6][0].numpy())]
    st1 = ctypes.c_int32(-1)
    for _ in range(5):
        av._lib.check(lib.avrf_thin_verify_one(0, 0, p0[0], p0[1], 1, p0[2], len(p0[2]), p0[3], p0[4], ctypes.byref(st1)))
    assert st1.value == 0
    t0 = time.perf_counter()
    for _ in range(30):
        lib.avrf_thin_verify_one(0, 0, p0[0], p0[1], 1, p0[2], len(p0[2]), p0[3], p0[4], ctypes.byref(st1))
    verify_one_us = (time.perf_counter() - t0) / 30 * 1e6

    # drop-in shape: BatchVerifier::push per proof through the C++ mirror (benches/thin.rs:76-88)
    drop_in = None
    try:
        pl = ctypes.CDLL(os.path.join(ROOT, "tools", "libavrf_pushloop.so"))
        pl.avrf_pushloop_new.restype = ctypes.c_void_p
        pl.avrf_pushloop_new.argtypes = [ctypes.c_uint64] + [ctypes.c_void_p] * 7
        pl.avrf_pushloop_step.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        pl.avrf_pushloop_free.argtypes = [ctypes.c_void_p]
        hpl = pl.avrf_pushloop_new(n, *[t.data_ptr() for t in host])
        pm, vm = ctypes.c_double(0), ctypes.c_double(0)
        for _ in range(2):
            assert pl.avrf_pushloop_step(hpl, 1, ctypes.byref(pm), ctypes.byref(vm)) == 0
        kd = args.steps
        acc = []

        def step_drop():
            assert pl.avrf_pushloop_step(hpl, 1, ctypes.byref(pm), ctypes.byref(vm)) == 0
            acc.append((pm.value, vm.value))
        t0 = time.perf_counter()
        barrier()
        for _ in range(kd):
            step_drop()
        barrier()
        ms_drop = (time.perf_counter() - t0) * 1e3 / kd
        drop_in = {"ms_per_batch": round(ms_drop, 3), "proofs_per_s": n / (ms_drop * 1e-3),
                   "push_loop_ms": round(float(np.mean([a for a, _ in acc])), 3), "verify_ms": round(float(np.mean([v for _, v in acc])), 3),
                   "note": "2^%d x BatchVerifier::push (C++ mirror, heap items) + verify" % args.log2n}
        pl.avrf_pushloop_free(hpl)
    except OSError as e:
        drop_in = {"unavailable": str(e)[:60]}

    # wire-format shape: the same batch as compressed encodings (what a caller holds before deserialisation), decoded and
    # validated on the device by avrf_thin_batch_push_compressed, then verified
    wire = None
    try:
        bc = synth.make_batch(0, n, 1, signers=4096, fmt=av.Format.CANONICAL, first=rank * n)
        wpk = pin(ops.point_compress(0, bc.pk, fmt=av.Format.CANONICAL))
        wr = pin(ops.point_compress(0, bc.r, fmt=av.Format.CANONICAL))
        wio = pin(np.concatenate([ops.point_compress(0, bc.ios[:128 * n].reshape(-1, 64), fmt=av.Format.CANONICAL).reshape(-1),
                                  np.zeros(64, np.uint8)]))
        wargs = (wpk, wio, host[2], host[3], host[4], wr, pin(bc.s))
        del bc
        wv = av.BatchVerifier(0, av.Format.MONTGOMERY)

        def step_wire():
            wv.clear()
            assert wv.push_compressed(*wargs).all()
            assert wv.verify_status() == 0
        for _ in range(2):
            step_wire()
        kw = args.steps
        barrier()
        t0 = time.perf_counter()
        for _ in range(kw):
            step_wire()
        barrier()
        ms_wire = (time.perf_counter() - t0) * 1e3 / kw
        wire = {"ms_per_batch": round(ms_wire, 3), "proofs_per_s": n / (ms_wire * 1e-3),
                "h2d_bytes_per_step": int(sum(t.numel() for t in wargs)), "points_decoded": 4 * n,
                "note": "avrf_thin_batch_push_compressed (GPU decode + subgroup check) + verify"}
        wv.close()
        del wargs, wpk, wr, wio
    except Exception as e:          # noqa: BLE001
        wire = {"unavailable": repr(e)[:80]}

    # ---- headline: T batches in flight -----------------------------------------------------------------------------
    # batches in flight.  With a core per batch in flight every batch's SHA-512 runs on its own core (K timed steps are
    # best served by two waves of K/2: the hashes of the second wave run under the MSMs of the first).  With fewer cores
    # (8 GPUs on a 32-core host: 4 per rank) the hashes go to shared multi-buffer threads, eight chains per core.
    # A burst of K batches is served fastest with all of them in flight: K hashes start at once and the GPU works through
    # the MSMs in the order the hashes finish.  A hash on a thread of its own has the lowest latency (82 ms on a free core);
    # hashes in the lanes of a shared multi-buffer thread cost an eighth of a core each but take ~190 ms.  Measured on the
    # 16-core box with taskset (ms per step, resident / end to end): all own-thread - 16 cores 14.1 / 14.5, 12 cores 14.0 /
    # 14.7, 8 cores 17.5 / 15.1; own-thread as far as the cores reach, the rest in lanes - 16 cores 14.0 / 15.8, 12 cores
    # 15.4 / 15.9, 8 cores 16.8 / 16.9; 4 cores (8 GPUs on a 32-core host), all in lanes 17.8 / 18.1, own-thread 27.3 / 27.9.
    # (End to end the pushes are staggered by their host-to-device copies, so fewer hashes run at the same time.)
    def split(T, mixed):
        if not mixed:
            return T, 0
        own = min(T, cores - 1)
        nh = 0
        if own < T:
            nh = -(-(T - own) // 7)
            own = max(1, min(T, cores - 1 - nh))
            nh = max(nh, -(-(T - own) // 8))
        return own, nh
    if args.concurrency or args.hashers >= 0:
        T = args.concurrency or max(1, min(16, cores, max(4, (args.steps + 1) // 2)))
        n_hash = max(0, args.hashers)
        n_own = T if n_hash == 0 else 0
        n_own_e2e, n_hash_e2e = n_own, n_hash
    elif cores < 6:
        n_hash = max(1, min(3, cores - 1))
        T = min(8 * n_hash, max(args.steps, 8))
        n_own = 0
        n_own_e2e, n_hash_e2e = n_own, n_hash
    else:
        T = max(4, min(args.steps, 24))
        n_own, n_hash = split(T, mixed=cores < 10)
        n_own_e2e, n_hash_e2e = T, 0
    if args.e2e_own >= 0 and args.e2e_hashers >= 0:
        n_own_e2e, n_hash_e2e = args.e2e_own, args.e2e_hashers
    handles = [bv]
    for _ in range(T - 1):
        h = av.BatchVerifier(0, av.Format.MONTGOMERY)
        h.push_many(*host)
        assert h.verify_status() == 0
        handles.append(h)
    pool = av.HashPool(n_hash) if n_hash else None
    for i, h in enumerate(handles):
        h.set_blocking(True)              # waiting threads sleep: the cores belong to the hashes of the other batches
        if pool is not None and i >= n_own:
            h.set_hash_pool(pool)
    launches = [0]
    # own-thread hashes: handle i starts i x 4 ms into the burst, so fewer hashes compete for the cores at the same time
    # and the first seeds are ready sooner (measured, K = 20, 16 cores: 0 / 4 / 6 / 8 / 10 ms -> 13.2 / 12.8 / 13.4 / 13.7 /
    # 14.1 ms per step); the GPU needs a new batch only every ~8 ms
    stagger_s = (args.stagger_ms if args.stagger_ms >= 0 else (4.0 if (n_hash == 0 and T > 8) else 0.0)) * 1e-3

    def run_steps(k):
        """k steps shared by the T handles: each host thread takes the next step until k are done.  Returns the handle
        that ran the k-th step and its verdict."""
        lock = threading.Lock()
        left = [k]
        errs = []
        last = [None, None]
        trace = [] if os.environ.get("AVRF_BENCH_TRACE") else None
        t_run0 = time.perf_counter()

        def work(h, idx=0):
            try:
                if stagger_s > 0 and idx:
                    time.sleep(idx * stagger_s)       # release the batches at the rate the GPU consumes them
                while True:
                    with lock:
                        if left[0] == 0:
                            return
                        left[0] -= 1
                        is_last = left[0] == 0
                    t_a = time.perf_counter()
                    h.invalidate()
                    st = h.verify_status()
                    if st != 0:
                        errs.append("verdict")
                    if is_last:
                        last[:] = [h, st]
                    tm = h.timings()
                    with lock:
                        launches[0] += tm["kernel_launches"]
                        if trace is not None:
                            trace.append((round((t_a - t_run0) * 1e3, 1), round((time.perf_counter() - t_run0) * 1e3, 1),
                                          round(tm["host_hash_ms"], 1), round(tm["prepare_ms"], 1)))
            except Exception as e:          # noqa: BLE001
                errs.append(repr(e))
        ths = [threading.Thread(target=work, args=(h, i)) for i, h in enumerate(handles)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        assert not errs, errs
        if trace:
            log("[trace] (start_ms, end_ms, host_hash_ms, prepare_ms) per step:", sorted(trace))
        return last

    t_e2e = T

    def run_e2e(k):
        tickets = [srv.submit(*host) for _ in range(k)]
        for t in tickets:
            assert srv.wait(t) == 0

    with ClockSampler(local_rank) as clk:          # nvidia-smi takes ~1 s to start: begin before warm-up
        run_steps(max(args.warmup, T))             # warm-up: every handle has run at least once
        clk.rows.clear()
        launches[0] = 0
        ms_step, (h_last, st_last) = timed(lambda: run_steps(args.steps), args.steps, others=handles[1:])
        n_launch = launches[0]
        clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, h_last, st_last)
    for h in handles[1:]:
        h.close()
    bv.set_blocking(False)
    if pool is not None:
        bv.set_hash_pool(None)
        pool.close()
    srv = av.BatchServer(0, av.Format.MONTGOMERY, workers=t_e2e, hashers=n_hash_e2e, own_hash_workers=n_own_e2e)     # native worker pool (avrf_server_*)
    run_e2e(max(args.warmup, t_e2e))
    ms_e2e, _ = timed(lambda: run_e2e(args.steps), args.steps)
    srv.close()

    # opt-in tree-hashed weights (not the reference's transcript bytes; reported beside, never as `value`)
    bv.set_weights_mode(1)

    def step_tree():
        bv.invalidate()
        assert bv.verify_status() == 0
    for _ in range(2):
        step_tree()
    ms_tree, _ = timed(lambda: [step_tree() for _ in range(k1)], k1)
    bv.set_weights_mode(0)

    # ---- per-kernel figures (CUDA events on the launch stream, single-batch leg: the kernel timed alone) --
    def avg(key):
        return float(np.mean([t[key] for t in tms]))
    acc_ms = avg("accumulate_ms")
    entries = float(np.mean([t["n_entries"] for t in tms]))
    canon_macs = entries * CANON_MM_PER_ADD * MM_MACS          # per launch
    achieved = canon_macs / (acc_ms * 1e-3) / 1e12
    executed = entries * (8 * 64 + 7 * 48) / (acc_ms * 1e-3) / 1e12     # 8 products, 7 reductions (lazy), BLS12-381 Fr shortcut
    phases = {k: round(avg(k), 3) for k in ("prepare_ms", "host_hash_ms", "scalars_ms", "sort_ms", "accumulate_ms", "reduce_ms")}
    npts = float(np.mean([t["n_points"] for t in tms]))
    sort_bytes = entries * 4 + npts * (32 + 64) + 4 * (1 << 19) * 6        # entries written, digits+ranks read, bin arrays
    peaks, traffic = {}, None
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    try:      # dram bytes of ONE launch from the committed `ncu --set full` capture of this workload, per addition
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["k_accumulate"]
        traffic = tr["dram_bytes_per_launch"] * entries / tr["additions_per_launch"]
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)

    # ---- BASELINE.json configs[2..4] at their stated sizes ---------------------------------------------------------
    configs = None
    if not args.no_configs:
        configs = {}
        bv.clear()

        def run_cfg(sid, m, lg, steps):
            bb = synth.make_batch(sid, 1 << lg, m, signers=4096, fmt=av.Format.MONTGOMERY)
            hh = av.BatchVerifier(sid, av.Format.MONTGOMERY)
            hh.push_many(bb.pk, bb.ios, bb.io_offsets, bb.ad_blob, bb.ad_offsets, bb.r, bb.s)
            hs = torch.cuda.ExternalStream(hh.stream, device=dev)
            tt = []

            def st():
                hh.invalidate()
                assert hh.verify_status() == 0
                tt.append(hh.timings())
            st()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(hs)
            for _ in range(steps):
                st()
            e1.record(hs)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            s2 = bb.s.copy()
            s2[(1 << lg) - 1, 0] ^= 1
            hh.clear()
            hh.push_many(bb.pk, bb.ios, bb.io_offsets, bb.ad_blob, bb.ad_offsets, bb.r, s2)
            rej_st = hh.verify_status()
            assert rej_st == 1
            a_ms = float(np.mean([t["accumulate_ms"] for t in tt[1:]]))
            ent = float(np.mean([t["n_entries"] for t in tt[1:]]))
            hh.close()
            return {"proofs_per_s": (1 << lg) / (ms * 1e-3), "ms_per_batch": round(ms, 2), "batch": 1 << lg, "io_pairs": m,
                    "host_hash_ms": round(float(np.mean([t["host_hash_ms"] for t in tt[1:]])), 2), "accumulate_ms": round(a_ms, 3),
                    "roofline_frac": round(ent * CANON_MM_PER_ADD * MM_MACS / (a_ms * 1e-3) / peak_wide, 4), "reject_ok": True}
        configs["C2_ed25519_2p20"] = run_cfg(1, 1, 20, args.steps)
        configs["C3_babyjubjub_2p22_m4"] = run_cfg(2, 4, 22, args.steps)
        # C4: bulk Elligator2 hash-to-curve + VRF output, 2^24 inputs over the ranks (no collective), host buffers
        n4 = (1 << 24) // world
        chunk = 1 << 21
        sk = synth.secret_from_seed(0, bytes(32))
        skb = np.frombuffer(sk.to_bytes(32, "little"), dtype=np.uint8).copy()
        off = (np.arange(chunk + 1, dtype=np.uint64) * 8).astype(np.uint32)
        outp = {"inputs": torch.empty((chunk, 64), dtype=torch.uint8).pin_memory(),
                "outputs": torch.empty((chunk, 64), dtype=torch.uint8).pin_memory(),
                "ok": torch.empty(chunk, dtype=torch.uint8).pin_memory()}
        blob = torch.empty(8 * chunk + 16, dtype=torch.uint8).pin_memory()
        ops.vrf_io_many(0, blob, off, skb, av.Format.MONTGOMERY, out=outp)      # warm-up (allocations)
        barrier()
        t0 = time.perf_counter()
        for first in range(rank * n4, rank * n4 + n4, chunk):
            blob[:8 * chunk] = torch.from_numpy(np.arange(first, first + chunk, dtype=np.uint64).view(np.uint8))
            ops.vrf_io_many(0, blob, off, skb, av.Format.MONTGOMERY, out=outp)  # Input::new + Secret::output, one call
            assert bool(outp["ok"].all())
        digest = int(np.bitwise_xor.reduce(outp["outputs"].numpy().view(np.uint64).reshape(-1)))     # last chunk
        barrier()
        dt4 = time.perf_counter() - t0
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([dt4], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt4 = float(t.item())
        configs["C4_h2c_output_2p24"] = {"inputs_per_s": (1 << 24) / dt4, "seconds": round(dt4, 3), "inputs": 1 << 24,
                                         "per_gpu": n4, "api": "avrf_vrf_io_many, pinned host buffers, chunks of 2^21", "xor64": "%016x" % digest}

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import corc
        Tc = host_threads()
        ns = min(n, 1 << args.cpu_sample_log2n)
        bc = synth.make_batch(0, ns, 1, signers=4096, fmt=av.Format.CANONICAL)      # the oracle takes canonical integers
        st, tm, _ = corc.thin_batch_verify(0, bc.pk, bc.ios, bc.io_offsets, bc.ad_blob, bc.ad_offsets, bc.r, bc.s, nthreads=Tc)
        assert st == 0
        small = {}
        for k in (256, 1024):               # configs[0] and the reference's largest published size, one thread
            best = 1e9
            for _ in range(3):
                st1, tm1, _ = corc.thin_batch_verify(0, bc.pk[:k], bc.ios[:k], bc.io_offsets[:k + 1], bc.ad_blob,
                                                     bc.ad_offsets[:k + 1], bc.r[:k], bc.s[:k], nthreads=1)
                assert st1 == 0
                best = min(best, sum(tm1))
            small["n%d_1thread_ms" % k] = round(best * 1e3, 2)
        cpu_baseline = {"value": ns / sum(tm), "unit": "proofs/s", "cores": Tc, "kind": "port",
                        "sample": f"first 2^{int(np.log2(ns))} proofs, prepare+verify ({tm[0]:.2f}s+{tm[1]:.2f}s), {Tc} threads",
                        **small, "published_n256_1thread_ms": 14.8}

    if rank == 0:
        value = world * n / (ms_step * 1e-3)
        e2e = world * n / (ms_e2e * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "proofs/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
            "data": "synthetic",
            "config": {"workload": workload_name(args.log2n),
                       "suite": "Bandersnatch-SHA512-ELL2-v1", "batch": n, "io_pairs": 1, "weights": "reference (serial SHA-512 per batch)",
                       "concurrency": T, "host_cores_per_gpu": cores, "own_thread_hashes": n_own, "mb_sha512_threads": n_hash,
                       "release_stagger_ms": round(stagger_s * 1e3, 1),
                       "step": "one whole 2^%d-proof batch per step; T batches in flight per GPU" % args.log2n,
                       "l2": "working set ~1.5 GB per batch exceeds the 126 MB L2; no flush",
                       "sharding": "every rank serves whole batches (no collective)" if world > 1 else "single GPU"},
            "e2e": {"value": e2e, "unit": "proofs/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": int(64 * n + 16), "workers": t_e2e, "own_thread_hashes": n_own_e2e, "mb_sha512_threads": n_hash_e2e,
                    "api": "avrf_server_submit/_wait, pinned host buffers"},
            "single_batch": {"resident_ms": round(ms_one, 3), "resident_proofs_per_s": n / (ms_one * 1e-3),
                             "e2e_ms": round(ms_one_e2e, 3), "e2e_proofs_per_s": n / (ms_one_e2e * 1e-3),
                             "phases_ms": phases, "drop_in": drop_in, "wire_push": wire, "verify_one_us": round(verify_one_us, 1),
                             "gpu_ms": round(sum(phases[k] for k in ("prepare_ms", "scalars_ms", "sort_ms", "accumulate_ms", "reduce_ms")), 3)},
            "sharded": sharded,
            "rejects": rejects,
            "gpu_launches": int(n_launch),
            "roofline": {"bound": "imad", "kernel": "k_accumulate", "achieved": achieved, "peak": peak_wide / 1e12,
                         "unit": "T wide-MAC/s", "frac": achieved / (peak_wide / 1e12), "traffic": traffic,
                         "executed": executed, "peak_carry_chain": peak_carry / 1e12,
                         "additions_per_launch": entries, "kernel_ms": acc_ms,
                         "hbm_sort": {"bound": "hbm", "kernels": "k_scan_*+k_scatter", "achieved": sort_bytes / (avg("sort_ms") * 1e-3) / 1e9,
                                      "peak": hbm_peak, "unit": "GB/s", "frac": sort_bytes / (avg("sort_ms") * 1e-3) / 1e9 / hbm_peak}},
            "alt_tree_weights": {"proofs_per_s": n / (ms_tree * 1e-3), "ms_per_batch": round(ms_tree, 3), "note": "opt-in, one batch at a time"},
            "configs": configs,
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "workload_generation_s": round(gen_s, 2),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
