"""Attention inside the persistent batch-1 decode kernel, where each item's cached K/V pages reach shared memory as stages of
the weight ring and only the row appended in the current step is read from L2 afterwards.

At true width (2 layers) for TinyLlama (head_dim 64), Mistral-7B and Qwen2.5-7B (7 query heads per kv head: every item is
streamed twice), decode steps of the persistent kernel are compared with the multi-kernel path (FL_NO_PERSISTENT=1) on the
same synthetic KV: the decoded slot at page offsets 0, 1 and 63, an 8k context whose items span more pages than the ring has
stages, a context shorter than the number of splits (empty items), and one greedy-loop launch whose steps cross a page and an
item boundary against one launch per step."""
from dataclasses import replace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KERNEL_TOL_WIDE = 6e-3      # persistent vs multi-kernel path at true width (tests/test_parity_gpu.py)


def _model(arch):
    from fastllm_b200 import presets
    cls, cf = presets.PRESETS[arch]
    model, _ = cls.initialize_model(replace(cf, num_hidden_layers=2, max_position_embeddings=16384), None, "bf16", 0, random_seed=1, std=0.02)
    return model


def _steps(model, ctx, n, cap):
    """n decode steps from a synthetic ctx-token KV, one launch per step -> (ids, logits) per step."""
    from fastllm_b200 import models
    c = models.DeviceCache(model.dev, 1, cap)
    c.fill_synthetic(1, ctx)
    tok, ids, logits = np.array([[5]], dtype=np.uint32), [], []
    for s in range(n):
        lg = c.forward(tok, ctx + s)[0]
        logits.append(lg)
        tok = np.array([[models.sample_argmax(lg)]], dtype=np.uint32)
        ids.append(int(tok[0, 0]))
    return ids, np.stack(logits)


@pytest.mark.parametrize("arch", ["tinyllama", "mistral7b", "qwen25_7b"])
def test_persistent_attention_matches_multikernel_path(arch, monkeypatch):
    from fastllm_b200 import models
    model = _model(arch)
    # (context, steps): slot at page offsets 0 / 1 / 63, 8 pages per item, fewer pages than splits
    cases = [(2048, 1), (2049, 1), (2111, 2), (8191, 1), (100, 2)]
    got = {k: _steps(model, *k, 8256) for k in cases}
    monkeypatch.setenv("FL_NO_PERSISTENT", "1")
    for k in cases:
        ids, want = _steps(model, *k, 8256)
        err = float(np.abs(got[k][1] - want).max())
        print(f"{arch} ctx {k[0]}: persistent vs multi-kernel max-abs logits diff {err:.3e}")
        assert got[k][0] == ids and err <= KERNEL_TOL_WIDE, (arch, k, err)


@pytest.mark.parametrize("arch", ["tinyllama", "mistral7b", "qwen25_7b"])
def test_greedy_loop_across_page_and_item_boundaries(arch):
    """Steps 2040 .. 2059 in ONE launch: the slot leaves page 31 for page 32, which is also the first page of the next item."""
    from fastllm_b200 import models
    model = _model(arch)
    c = models.DeviceCache(model.dev, 1, 2200)
    c.fill_synthetic(1, 2040)
    loop_ids, _ = c.decode_greedy_loop(np.array([5], dtype=np.uint32), 2040, 20)
    step_ids, _ = _steps(model, 2040, 20, 2200)
    assert list(loop_ids[:, 0]) == step_ids
