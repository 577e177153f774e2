"""bench.py on the GPU: --steps sets the number of timed steps, and --dump-outputs writes what the last of them returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_ids_of_the_last_timed_step(tmp_path):
    """TinyLlama batch 1 (the persistent decode kernel), 5 timed steps: the JSON line reports 5 steps, and next_token_ids.npy holds
    the ids the 5th step emitted -- the ids this process gets from the same seeded weights, synthetic KV cache and first token."""
    import bench
    from fastllm_b200 import models, presets
    K, W = 5, 3
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tinyllama_b1", "--steps", str(K), "--warmup", str(W),
                        "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == K
    got = np.load(tmp_path / "next_token_ids.npy")
    _, batch, ctx, _ = bench.WORKLOADS["tinyllama_b1"]
    cls, cf = presets.PRESETS["tinyllama"]
    model, _ = cls.initialize_model(cf, None, "bf16", 0, random_seed=0, std=0.02)
    cache = models.DeviceCache(model.dev, batch, ctx + max(K, W, 16) + 8)
    cache.fill_synthetic(batch, ctx)
    ids, _ = cache.decode_greedy_loop(np.full((batch,), 5, dtype=np.uint32), ctx, K)
    assert got.dtype == np.float64 and got.shape == (batch,) and np.array_equal(got, ids[-1])
