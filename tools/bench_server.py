"""The batch server (avrf_server_*) on one GPU for both proof schemes and both input forms, on the synthetic workload of
bench.py: bursts of K batches of 2^20 Bandersnatch proofs (one I/O pair each, 4096 signers), submitted from pinned host
memory and waited for in order.  Each burst leg reports the best of --reps bursts after a warm-up burst.  Prints one
JSON line with the device name and power limit read in the same run.  Legs:
  thin_decoded       avrf_server_submit (what bench.py's `e2e` leg runs)
  thin_wire          avrf_server_submit_compressed: 32-byte points, decoded and validated on the GPU
  pedersen_decoded   avrf_pedersen_server_submit
  pedersen_wire      avrf_pedersen_server_submit_compressed: 160-byte records (pedersen.serialize_proofs)
  pedersen_one       one Pedersen batch at a time: pedersen.BatchVerifier push_many + verify (the baseline of the ratios)
Workers: one per batch of the burst.  With 10 or more host cores every worker hashes its batch seed on its own thread;
with fewer, the workers share ceil(K / 8) multi-buffer SHA-512 threads and as many keep a core of their own as remain.
Usage: python tools/bench_server.py [--log2n 20] [--burst 20] [--reps 3]"""
import argparse
import json
import os
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


def best(fn, reps):
    fn()                                   # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--burst", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import numpy as np
    import torch
    import ark_vrf_b200 as av
    from ark_vrf_b200 import _lib, ops, pedersen as ped, synth
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU only")
    lib = av.load()
    _lib.check(lib.avrf_init(0))
    n, K, sid = 1 << a.log2n, a.burst, 0
    cores = len(os.sched_getaffinity(0))
    hashers = 0 if cores >= 10 else -(-K // 8)
    own = K if hashers == 0 else max(1, min(K, cores - 1 - hashers))
    name, power = device_info()
    res = {"device": name, "power_limit": power, "n": n, "m": 1, "signers": 4096, "suite": "bandersnatch", "burst": K,
           "reps": a.reps, "host_cores": cores, "workers": K, "own_thread_hashes": own, "mb_sha512_threads": hashers}

    def pin(x):
        x = np.ascontiguousarray(x)
        return torch.from_numpy(x.view(np.int32) if x.dtype == np.uint32 else x).pin_memory()

    def leg(key, srv, submit, arrays, wire):
        args = [pin(x) for x in arrays]
        bad = []

        def burst():
            tickets = [submit(*args) for _ in range(K)]
            for t in tickets:
                st = srv.wait_compressed(t)[0] if wire else srv.wait(t)
                if st != 0:
                    bad.append(st)
        t = best(burst, a.reps)
        srv.close()
        assert not bad, (key, bad)
        res[key] = {"proofs_per_s": round(K * n / t), "ms_per_batch": round(1e3 * t / K, 2)}

    F = av.Format.MONTGOMERY
    tb = synth.make_batch(sid, n, 1, 4096, F)
    srv = av.BatchServer(sid, F, workers=K, hashers=hashers, own_hash_workers=own)
    leg("thin_decoded", srv, srv.submit, (tb.pk, tb.ios, tb.io_offsets, tb.ad_blob, tb.ad_offsets, tb.r, tb.s), False)
    C = av.Format.CANONICAL                 # wire format: canonical scalars; the point encodings are format-free
    tc = synth.make_batch(sid, n, 1, 4096, C)
    ios32 = ops.point_compress(sid, tc.ios.reshape(-1, 64), C).reshape(-1)
    srv = av.BatchServer(sid, F, workers=K, hashers=hashers, own_hash_workers=own)
    leg("thin_wire", srv, srv.submit_compressed, (ops.point_compress(sid, tc.pk, C), ios32, tc.io_offsets, tc.ad_blob,
                                                   tc.ad_offsets, ops.point_compress(sid, tc.r, C), tc.s), True)
    del tb, tc

    pb = synth.make_pedersen_batch(sid, n, 1, 4096, F)
    dec = (pb.ios, pb.io_offsets, pb.ad_blob, pb.ad_offsets, pb.pk_com, pb.r, pb.ok, pb.s, pb.sb)
    srv = ped.BatchServer(sid, F, workers=K, hashers=hashers, own_hash_workers=own)
    leg("pedersen_decoded", srv, srv.submit, dec, False)
    ios32 = ops.point_compress(sid, pb.ios.reshape(-1, 64), F).reshape(-1)
    recs = ped.serialize_proofs(sid, pb.pk_com, pb.r, pb.ok, pb.s, pb.sb, F)
    srv = ped.BatchServer(sid, F, workers=K, hashers=hashers, own_hash_workers=own)
    leg("pedersen_wire", srv, srv.submit_compressed, (ios32, pb.io_offsets, pb.ad_blob, pb.ad_offsets, recs), True)

    args = [pin(x) for x in dec]
    bv = ped.BatchVerifier(sid, F)
    status = []

    def one():
        bv.clear()
        bv.push_many(*args)
        status.append(bv.verify_status())
    t = best(one, a.reps)
    assert set(status) == {0}, status
    res["pedersen_one"] = {"proofs_per_s": round(n / t), "ms_per_batch": round(1e3 * t, 2)}
    base = res["pedersen_one"]["proofs_per_s"]
    res["ratio_over_pedersen_one"] = {k: round(res[k]["proofs_per_s"] / base, 2)
                                      for k in ("thin_decoded", "thin_wire", "pedersen_decoded", "pedersen_wire")}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
