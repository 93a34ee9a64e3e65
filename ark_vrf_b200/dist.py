"""One batch sharded over the GPUs of a box: one process per GPU, `torch.distributed` plumbing.

The reference has no distributed code; this is the multi-GPU form of
`thin::BatchVerifier::verify` (src/thin.rs:257-325) described in SURVEY.md section 8(e):

  1. every rank runs the per-proof transcripts of its contiguous shard on its GPU
     (BatchVerifier::prepare, thin.rs:209-226) and the identity gate (thin.rs:266-271);
  2. the (c_j, s_j) byte streams are all-gathered in global proof order and every rank
     computes the batch seed - one serial SHA-512 over all proofs (thin.rs:273-279), the
     only step that cannot shard;
  3. every rank squeezes its own weights by counter index (thin.rs:289) and reduces its
     shard of the MSM (thin.rs:282-319) to ONE partial point;
  4. the 128-byte partials (+ the InvalidData flag) meet in a single all-gather (NCCL over
     NVLink on GPUs; gloo in the CPU tests) and every rank adds them and tests for the
     identity (thin.rs:320-324).

The verdict is identical on every rank.  Shard boundaries need no alignment (weights are
addressed by global index).  A `pedersen.BatchVerifier` shard runs the same steps for
`pedersen::BatchVerifier::verify` (src/pedersen.rs:341-426): 96-byte (c_j, s_j, sb_j) records in
step 2, five MSM terms per proof and the shard's share of G and B in step 3.
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence

import numpy as np

STATUS_OK, STATUS_VERIFICATION_FAILURE, STATUS_INVALID_DATA = 0, 1, 2


def shard_bounds(n: int, world: int, rank: int):
    """Contiguous shards, multiples of 32 proofs (one tree leaf = 32 proofs, one weight block = 4)."""
    per = ((n + world - 1) // world + 31) // 32 * 32
    lo = min(n, rank * per)
    hi = min(n, lo + per)
    return lo, hi


def _all_gather_bytes(local: np.ndarray, group, device) -> list:
    """all_gather of variable-length uint8 arrays; returns the per-rank arrays in rank order."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    n_local = torch.tensor([local.size], dtype=torch.int64, device=device)
    sizes = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(sizes, n_local, group=group)
    sizes = [int(s.item()) for s in sizes]
    cap = max(max(sizes), 1)
    buf = torch.zeros(cap, dtype=torch.uint8, device=device)
    if local.size:
        buf[:local.size] = torch.from_numpy(np.ascontiguousarray(local).reshape(-1)).to(device)
    out = torch.empty(world * cap, dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(out, buf, group=group)
    host = out.cpu().numpy().reshape(world, cap)
    return [host[r, :sizes[r]] for r in range(world)]


class _DevView:
    """Zero-copy view of a device buffer for torch (``__cuda_array_interface__``)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


_gather_buf = {}


def _seed_fns(stride: int):
    """(host, device) seed functions of the scheme whose batch-seed records are `stride` bytes."""
    from . import pedersen, thin
    if stride == pedersen.BatchVerifier.cs_stride:
        return pedersen.seed_of_stream, pedersen.seed_of_device_stream
    return thin.seed_of_stream, thin.seed_of_device_stream


def _device_seed(shard, suite: int, group, device, stride: int = 64):
    """NCCL fast path: all-gather the batch-seed streams (`stride` bytes per proof) device-to-device (equal
    shard sizes), then hash the gathered stream with the chunked D2H overlapped with the host SHA-512.
    Returns (seed, n_total) or None when shard sizes differ (caller falls back to the generic path)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    nl = len(shard)
    sizes = torch.tensor([nl], dtype=torch.int64, device=device)
    all_sizes = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(all_sizes, sizes, group=group)
    all_sizes = [int(x.item()) for x in all_sizes]
    if len(set(all_sizes)) != 1 or nl == 0:
        return None
    ptr, nbytes = shard.cs_stream_dev()
    local = torch.as_tensor(_DevView(ptr, nbytes), device=device)
    key = (str(device), world * nbytes)
    out = _gather_buf.get(key)
    if out is None:
        out = torch.empty(world * nbytes, dtype=torch.uint8, device=device)
        _gather_buf.clear()
        _gather_buf[key] = out
    dist.all_gather_into_tensor(out, local, group=group)
    torch.cuda.current_stream(device).synchronize()
    return _seed_fns(stride)[1](suite, out.data_ptr(), world * nl), world * nl


def sharded_verify(shard, suite: int, first_index: int, group=None, device=None,
                   seed_fn: Optional[Callable] = None, combine_fn: Optional[Callable] = None,
                   timings: Optional[dict] = None, weights: str = "reference") -> int:
    """Verify one batch whose proofs [first_index, first_index + len(shard)) live in `shard`
    (a `thin.BatchVerifier` or `pedersen.BatchVerifier` holding this rank's proofs).  Returns the status
    code (same on all ranks).

    `seed_fn(suite, stream_bytes)` / `combine_fn(suite, partials_bytes)` default to the library's
    (avrf_thin_seed or avrf_pedersen_seed, by the shard's `cs_stride`; avrf_thin_combine_partials);
    tests inject oracle-backed ones to exercise the rank plumbing on CPU.  `weights="tree"` is
    defined for Thin shards only: a Pedersen shard raises ValueError, on every rank, before any
    collective."""
    import time
    from . import thin
    stride = int(getattr(shard, "cs_stride", 64))
    default_seed, _ = _seed_fns(stride)
    if weights == "tree" and default_seed is not thin.seed_of_stream:
        raise ValueError("weights='tree' is defined for Thin-VRF batches only")
    seed_fn = seed_fn or default_seed
    combine_fn = combine_fn or thin.combine_partials
    dev = device if device is not None else "cpu"
    t0 = time.perf_counter()
    invalid = bool(shard.prepare_device())
    fast = None
    if weights == "tree":
        # opt-in tree seed: every rank hashes only its own shard on its GPU, the 64-byte leaf digests
        # (one per 32 proofs) are all-gathered and the root is a 2 MiB host hash
        t1 = time.perf_counter()
        leaves = np.ascontiguousarray(shard.tree_leaves(first_index)).reshape(-1)
        meta = np.frombuffer(int(len(shard)).to_bytes(8, "little"), dtype=np.uint8)
        got = _all_gather_bytes(np.concatenate([meta, leaves]), group, dev)
        n_total = sum(int.from_bytes(bytes(g[:8]), "little") for g in got)
        all_leaves = np.concatenate([g[8:] for g in got])
        fast = (thin.seed_of_tree(suite, n_total, all_leaves), n_total)
    elif dev != "cpu" and hasattr(shard, "cs_stream_dev") and seed_fn is default_seed:
        t1 = time.perf_counter()
        fast = _device_seed(shard, suite, group, dev, stride)
    if fast is not None:
        seed, total = fast
        t2 = t3 = time.perf_counter()
    else:
        cs_local = np.ascontiguousarray(shard.cs_stream(), dtype=np.uint8).reshape(-1)
        t1 = time.perf_counter()
        streams = _all_gather_bytes(cs_local, group, dev)
        stream = np.concatenate(streams) if len(streams) > 1 else streams[0]
        t2 = time.perf_counter()
        seed = seed_fn(suite, np.ascontiguousarray(stream))
        t3 = time.perf_counter()
        total = stream.size // stride
    if total == 0:
        return STATUS_OK                                       # thin.rs:262-264
    partial = shard.partial(seed, first_index) if len(shard) else None
    t4 = time.perf_counter()
    msg = np.zeros(130, dtype=np.uint8)
    if partial is not None:
        msg[:128] = np.frombuffer(partial, dtype=np.uint8)
        msg[128] = 1
    msg[129] = 1 if invalid else 0
    parts = _all_gather_bytes(msg, group, dev)
    t5 = time.perf_counter()
    if any(int(p[129]) for p in parts):
        status = STATUS_INVALID_DATA                           # thin.rs:266-271
    else:
        blob = b"".join(bytes(p[:128]) for p in parts if int(p[128]))
        status = combine_fn(suite, blob)
    t6 = time.perf_counter()
    if timings is not None:
        timings.update(prepare_s=t1 - t0, gather_s=t2 - t1, hash_s=t3 - t2, partial_s=t4 - t3,
                       gather2_s=t5 - t4, combine_s=t6 - t5)
    return status


def sharded_inputs_outputs(suite: int, n_total: int, sk, fmt: int = 0, group=None, device=None,
                           h2c_fn: Optional[Callable] = None, out_fn: Optional[Callable] = None,
                           compress_fn: Optional[Callable] = None):
    """BASELINE.json configs[4]: `Input::new` (lib.rs:500-502) + `Secret::output` (lib.rs:391-393) for the
    messages LE64(j), j < n_total, sharded over the ranks - no data-path collective (SURVEY.md 8e: "C4 is
    embarrassingly parallel").  Returns (lo, hi, inputs, outputs, digest): this rank's slice as (hi-lo, 64)
    arrays and a 64-bit checksum of ALL compressed outputs (XOR of per-point words, all-reduced by summing the
    per-rank XORs' bit-planes modulo 2) that is the same on every rank and independent of the sharding.

    `h2c_fn(suite, blob, offsets, fmt)`, `out_fn(suite, sk, inputs, fmt)`, `compress_fn(suite, points, fmt)`
    default to ark_vrf_b200.ops; the CPU tests inject oracle-backed ones."""
    import torch
    import torch.distributed as dist
    from . import ops
    h2c_fn = h2c_fn or (lambda su, blob, off, f: ops.hash_to_curve(su, blob, off, f)[0])
    out_fn = out_fn or ops.vrf_output
    compress_fn = compress_fn or ops.point_compress
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    lo, hi = shard_bounds(n_total, world, rank)
    k = hi - lo
    msgs = np.arange(lo, hi, dtype=np.uint64).view(np.uint8).reshape(k, 8)
    off = (np.arange(k + 1, dtype=np.uint64) * 8).astype(np.uint32)
    blob = np.concatenate([msgs.reshape(-1), np.zeros(16, dtype=np.uint8)])
    if k:
        inputs = h2c_fn(suite, blob, off, fmt)
        sks = np.ascontiguousarray(np.broadcast_to(np.asarray(sk, dtype=np.uint8).reshape(1, 32), (k, 32)))
        outputs = out_fn(suite, sks, inputs, fmt)
        enc = np.ascontiguousarray(compress_fn(suite, outputs, fmt)).view(np.uint64)
        x = int(np.bitwise_xor.reduce(enc.reshape(-1)))
    else:
        inputs = outputs = np.zeros((0, 64), dtype=np.uint8)
        x = 0
    digest = x
    if world > 1:
        dev = device if device is not None else "cpu"
        planes = torch.tensor([(x >> i) & 1 for i in range(64)], dtype=torch.int64, device=dev)
        dist.all_reduce(planes, group=group)                   # XOR of the ranks = bit-plane sums mod 2
        digest = sum((int(v) & 1) << i for i, v in enumerate(planes.cpu().tolist()))
    return lo, hi, inputs, outputs, digest
