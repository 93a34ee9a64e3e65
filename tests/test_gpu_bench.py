"""GPU: `bench.py --dump-outputs` writes what the last timed step of the headline computed, and on the synthetic batch it
equals the C oracle's verdict, seed, challenges and delinearization scalars."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs(tmp_path):
    from oracle import corc
    log2n = 12
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--log2n", str(log2n),
                          "--no-configs", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    d = {f[:-len(".npy")]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert set(d) == {"verdict", "seed", "sample_index", "challenge_c", "delinearization_z"}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    # the bench's workload, generated independently by the oracle's prover
    st, _, taps = corc.thin_batch_verify(0, *corc.synth_batch(0, 1 << log2n, 1, signers=4096, nthreads=8), nthreads=8, taps=True)
    idx = d["sample_index"].astype(np.int64)
    assert d["verdict"].tolist() == [st] == [0]
    assert (d["seed"] == taps["seed"]).all()
    assert (d["challenge_c"] == taps["c"][idx]).all()
    assert (d["delinearization_z"] == taps["z"][idx]).all()
