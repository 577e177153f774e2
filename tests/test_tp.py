"""Tensor parallelism: world_size-2 gloo test of the sharding scheme on CPU, and (when 2+ GPUs are visible) TP-2 through
the library with real NCCL against the TP-1 result."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(mode, nproc, out, port):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "tp_worker.py"), mode, out]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return json.load(open(out))


def test_tp_sharding_scheme_gloo_world2(tmp_path):
    """Column-parallel gate/up + row-parallel down with an all-reduce, vocab-parallel head with an all-gather, q/k/v split by
    head (incl. replicated kv head + padded query heads), and the Mixtral expert-parallel dispatch / combine data flow with
    data-parallel rows: same numbers as the unsharded oracle (numpy over gloo, 2 processes)."""
    assert _run("cpu", 2, str(tmp_path / "cpu.json"), 29631)["ok"]


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_ngpu() < 2, reason="needs 2 GPUs")
def test_tp2_matches_tp1(tmp_path):
    r1 = _run("gpu", 1, str(tmp_path / "tp1.json"), 29641)
    r2 = _run("gpu", 2, str(tmp_path / "tp2.json"), 29642)
    # expert parallelism (Mixtral): EP-2 == EP-1 == golden greedy ids
    assert r1["mixtral"]["ids"] == r2["mixtral"]["ids"] == r1["mixtral"]["golden_ids"]
    assert np.abs(np.array(r1["mixtral"]["logits"]) - np.array(r2["mixtral"]["logits"])).max() < 3e-3
    # expert parallelism with data-parallel attention + dispatch/combine all-to-all: same logits as one GPU running all 4 sequences
    assert np.abs(np.array(r1["mixtral_dp"]) - np.array(r2["mixtral_dp"])).max() < 3e-3
    # persistent decode kernel with the in-kernel NVLink all-reduce (TP-2) against the single-GPU persistent kernel
    assert r1["wide"]["ids"] == r2["wide"]["ids"] and r1["wide"]["loop_ids"] == r2["wide"]["loop_ids"]
    assert np.abs(np.array(r1["wide"]["logits"]) - np.array(r2["wide"]["logits"])).max() < 6e-3
    # Qwen2 with more ranks than kv heads: replicated kv head + zero-padded query heads
    assert r1["qwen2"]["ids"] == r2["qwen2"]["ids"] == r1["qwen2"]["golden_ids"]
    for k in ("logits", "synth_logits", "batch3"):
        assert np.abs(np.array(r1["qwen2"][k]) - np.array(r2["qwen2"][k])).max() < 3e-3, k
    one, two = r1["mistral"], r2["mistral"]
    assert one["ids"] == two["ids"]
    assert np.abs(np.array(one["logits"]) - np.array(two["logits"])).max() < 3e-3
    assert np.abs(np.array(one["synth_logits"]) - np.array(two["synth_logits"])).max() < 3e-3
    assert np.abs(np.array(one["batch3"]) - np.array(two["batch3"])).max() < 3e-3


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 4, 8])
def test_tpN_matches_tp1_at_true_widths(n, tmp_path):
    """N ranks against ONE rank on the same synthetic weights, through real NCCL / NVLink peer memory: Mistral-7B and Qwen2.5-7B
    shapes (2 layers; Qwen with its real 28 q / 4 kv heads -- padded and replicated at 8 ranks -- and its 152064-row vocabulary),
    batch 1 in the persistent kernel (in-kernel all-reduce) and batch 8 on the dense path, plus expert-parallel Mixtral-8x7B shapes
    (1 layer, 8 experts).  Teacher-forced with fixed tokens; logits within the true-width kernel tolerance (the split changes the
    summation order), arg-max identical wherever the single-GPU top-2 gap exceeds that noise."""
    if _ngpu() < n:
        pytest.skip(f"needs {n} GPUs")
    r1 = _run("gpu_wide", 1, str(tmp_path / "w1.json"), 29651)
    rn = _run("gpu_wide", n, str(tmp_path / f"w{n}.json"), 29652 + n)
    for tag in ("mistral7b", "qwen25_7b"):
        a, b = r1[tag], rn[tag]
        e1 = float(np.abs(np.array(a["logits"]) - np.array(b["logits"])).max())
        e8 = float(np.abs(np.array(a["b8_logits"]) - np.array(b["b8_logits"])).max())
        print(f"{tag}: tp{n} vs tp1 max-abs logits diff, batch 1 (persistent) {e1:.2e}, batch 8 (dense) {e8:.2e}")
        assert e1 < 6e-3 and e8 < 6e-3, tag
        # arg-max identical wherever the single-GPU top-2 gap is not inside the summation-order noise
        for (i1, g1), (i2, _) in zip(a["top"] + [t for l in a["b8_top"] for t in l], b["top"] + [t for l in b["b8_top"] for t in l]):
            assert i1 == i2 or g1 <= 2 * max(e1, e8), tag
        # the device-resident loop on N ranks emits the (near-)arg-max of its own step-by-step logits
        assert max(b["loop_slack"]) <= 2 * 6e-3 and max(a["loop_slack"]) <= 2 * 6e-3, tag
    em = float(np.abs(np.array(r1["mixtral"]["logits"]) - np.array(rn["mixtral"]["logits"])).max())
    print(f"mixtral 8 experts: ep{n} vs 1 GPU max-abs logits diff {em:.2e}")
    assert em < 6e-3


def test_head_layout_more_ranks_than_kv_heads():
    """tp.head_layout (the Python statement of build_weights in csrc/fl_lib.cu): Qwen2.5-7B (28 q / 4 kv heads) at TP-8 replicates each
    kv head on two ranks and deals its 7 query heads 4 + 3 (+1 zero head); every q head is owned exactly once; Mistral-7B at TP-8
    is the plain split."""
    from fastllm_b200 import tp
    owned = []
    for r in range(8):
        q0, qn, nhl, k0, kn = tp.head_layout(28, 4, r, 8)
        assert (nhl, kn, k0) == (4, 1, r // 2) and qn == (4 if r % 2 == 0 else 3)
        assert all(h // 7 == k0 for h in range(q0, q0 + qn))          # a rank's q heads belong to its kv head's group
        owned += list(range(q0, q0 + qn))
    assert sorted(owned) == list(range(28))
    assert [tp.head_layout(32, 8, r, 8) for r in range(8)] == [(4 * r, 4, 4, r, 1) for r in range(8)]
    w = {"model.layers.0.self_attn.q_proj.weight": np.zeros((28 * 128, 64), np.float32),
         "model.layers.0.self_attn.k_proj.weight": np.zeros((4 * 128, 64), np.float32),
         "model.layers.0.self_attn.o_proj.weight": np.zeros((64, 28 * 128), np.float32)}
    sh = tp.shard_weights(w, 28, 4, 3, 8)      # rank 3: kv head 1, q heads 11..13
    assert sh["model.layers.0.self_attn.q_proj.weight"].shape == (3 * 128, 64)
    assert sh["model.layers.0.self_attn.k_proj.weight"].shape == (128, 64)
    assert sh["model.layers.0.self_attn.o_proj.weight"].shape == (64, 3 * 128)
