"""fl_forward_logprobs on the device: per-position log-probs of given targets and the arg-max, in one forward.

Tolerances (max-abs): against the oracle with the same bf16 KV rounding, a log-prob is z[target] - lse(z), and each of the two
terms is within KERNEL_TOL of the oracle's, so the bar is 2 x KERNEL_TOL; against fl_forward on the same cache state both take the
dense path with the same hidden states and only the lm_head's summation order differs (1e-4)."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from oracle import causal_lm as ocl
from oracle import synth

from helpers import GOLDEN, TINY, golden_weights, product_model
from logprobs_ref import log_softmax64, logits_all, top2_gap

KERNEL_TOL = 3e-3
KERNEL_TOL_WIDE = 6e-3
LOGIT_TOL_FULL = 6e-2
LP_TOL = 2 * KERNEL_TOL


def _targets(seed, V, shape):
    """random targets with 0, V - 1 and ids of the last (partial) 256-wide vocab tile among them"""
    tg = synth.token_ids(seed, V, shape).copy()
    flat = tg.reshape(-1)
    last_tile = (V - 1) // 256 * 256
    flat[0], flat[1], flat[-1] = 0, V - 1, last_tile
    flat[len(flat) // 2] = (last_tile + V - 1) // 2
    return tg


def _check_against(lp, am, z, targets, tol, what):
    want = np.take_along_axis(log_softmax64(z), targets[..., None].astype(np.int64), axis=-1)[..., 0]
    err = float(np.abs(lp - want).max())
    gap = top2_gap(z)
    sure = gap > tol
    wrong = int(((am != np.argmax(z, axis=-1)) & sure).sum())
    print(f"{what}: max-abs log-prob err {err:.3e} (tol {tol:.0e}); arg-max differs at {wrong} of {int(sure.sum())} positions "
          f"with a top-2 gap > {tol:.0e} ({int((~sure).sum())} closer)")
    assert np.isfinite(lp).all()
    assert err <= tol and wrong == 0
    return err


def _shapes(name):
    # R = b * t below one 128-row tile, exactly one, and above two (a partial last M tile); the Llama fixtures' RoPE tables hold 128
    # positions, so their third shape takes a third sequence instead of 150 tokens
    big = (3, 100) if TINY[name].max_position_embeddings < 150 else (2, 150)
    return [(2, 40), (2, 64), big]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(TINY))
def test_logprobs_match_the_oracle(name):
    from fastllm_b200 import models
    cfg, w, _ = golden_weights(name)
    model, _ = product_model(cfg, w)
    for b, t in _shapes(name):
        ids = synth.token_ids(40 + t, cfg.vocab_size, (b, t))
        tg = _targets(41 + t, cfg.vocab_size, (b, t))
        c = models.DeviceCache(model.dev, b, 256)
        lp, am = c.forward_logprobs(ids, tg, 0)
        assert lp.shape == (b, t) and am.shape == (b, t) and c.kv_len() == t
        z = logits_all(ocl.CausalLM(cfg, w, kv_dtype="bf16"), ids, 0)
        _check_against(lp, am, z, tg, LP_TOL, f"{name} b={b} t={t} R={b * t}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["llama", "mistral", "qwen2"])
def test_logprobs_agree_with_fl_forward(name):
    from fastllm_b200 import models
    cfg, w, _ = golden_weights(name)
    model, _ = product_model(cfg, w)
    b, t = 2, 9
    ids = synth.token_ids(77, cfg.vocab_size, (b, t))
    tg = _targets(78, cfg.vocab_size, (b, t))
    lp, am = models.DeviceCache(model.dev, b, 64).forward_logprobs(ids, tg, 0)
    # the last position: the same dense forward, only the lm_head's summation order differs
    z = models.DeviceCache(model.dev, b, 64).forward(ids, 0)
    greedy = models.DeviceCache(model.dev, b, 64).forward_greedy(ids, 0)
    assert np.array_equal(greedy, np.array([models.sample_argmax(r) for r in z], dtype=np.uint32))
    want = log_softmax64(z)[np.arange(b), tg[:, -1]]
    err = float(np.abs(lp[:, -1] - want).max())
    sure = top2_gap(z) > 1e-4
    print(f"{name}: last position vs fl_forward logits {err:.3e}")
    assert err <= 1e-4
    assert np.array_equal(am[:, -1][sure], greedy[sure])
    # earlier positions: the last position of a shorter call on a fresh cache
    for j in (0, 3, 6):
        zj = models.DeviceCache(model.dev, b, 64).forward(np.ascontiguousarray(ids[:, :j + 1]), 0)
        e = float(np.abs(lp[:, j] - log_softmax64(zj)[np.arange(b), tg[:, j]]).max())
        print(f"{name}: position {j} vs fl_forward of ids[:, :{j + 1}] {e:.3e}")
        assert e <= LP_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mistral", "qwen2", "mistral_sw"])
def test_scoring_on_a_non_empty_cache(name):
    """Prefill a context with fl_forward, then score the continuation at RoPE offset t0.  A multi-token call on a non-empty cache
    sees every cached key (candle's mask puts zeros over the past), so with a 5-token window (mistral_sw) it is NOT one call over
    context + continuation; the oracle fed the same two calls is the reference, and the one-call comparison holds where the window
    does not bite."""
    from fastllm_b200 import models
    cfg, w, _ = golden_weights(name)
    model, _ = product_model(cfg, w)
    b, t0, t1 = 2, 20, 13
    ids = synth.token_ids(90, cfg.vocab_size, (b, t0 + t1))
    tg = _targets(91, cfg.vocab_size, (b, t0 + t1))
    c = models.DeviceCache(model.dev, b, 128)
    c.forward(np.ascontiguousarray(ids[:, :t0]), 0)
    lp, am = c.forward_logprobs(np.ascontiguousarray(ids[:, t0:]), np.ascontiguousarray(tg[:, t0:]), t0)
    assert c.kv_len() == t0 + t1
    o = ocl.CausalLM(cfg, w, kv_dtype="bf16")
    o.forward(ids[:, :t0], 0)
    z = logits_all(o, ids[:, t0:], t0)
    _check_against(lp, am, z, tg[:, t0:], LP_TOL, f"{name}: prefill {t0} + score {t1} vs the oracle")
    if cfg.sliding_window >= t0 + t1:
        one, _ = models.DeviceCache(model.dev, b, 128).forward_logprobs(ids, tg, 0)
        err = float(np.abs(lp - one[:, t0:]).max())
        print(f"{name}: prefill {t0} + score {t1} vs one scoring call over {t0 + t1}: {err:.3e}")
        assert err <= LP_TOL
    # the cache holds what a forward would have left: the next decode step matches the oracle
    nxt = synth.token_ids(92, cfg.vocab_size, (b, 1))
    got = c.forward(nxt, t0 + t1)
    kerr = float(np.abs(got - o.forward(nxt, t0 + t1)).max())
    print(f"{name}: decode step after scoring vs oracle {kerr:.3e}")
    assert kerr <= KERNEL_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("name,b", [("llama", 3), ("qwen2", 2)])
def test_scoring_is_deterministic_and_rows_are_independent(name, b):
    from fastllm_b200 import models
    cfg, w, _ = golden_weights(name)
    model, _ = product_model(cfg, w)
    ids = synth.token_ids(21, cfg.vocab_size, (b, 9))
    tg = _targets(22, cfg.vocab_size, (b, 9))
    lp1, am1 = models.DeviceCache(model.dev, b, 64).forward_logprobs(ids, tg, 0)
    lp2, am2 = models.DeviceCache(model.dev, b, 64).forward_logprobs(ids, tg, 0)
    assert np.array_equal(lp1, lp2) and np.array_equal(am1, am2)
    for s in range(b):
        lps, ams = models.DeviceCache(model.dev, 1, 64).forward_logprobs(ids[s:s + 1], tg[s:s + 1], 0)
        assert np.array_equal(lps[0], lp1[s]) and np.array_equal(ams[0], am1[s])
    # one token of one sequence (fl_forward would run it in the persistent / GEMV path)
    lp, am = models.DeviceCache(model.dev, 1, 64).forward_logprobs(ids[:1, :1], tg[:1, :1], 0)
    z = logits_all(ocl.CausalLM(cfg, w, kv_dtype="bf16"), ids[:1, :1], 0)
    _check_against(lp, am, z, tg[:1, :1], LP_TOL, f"{name} b=1 t=1")


@pytest.mark.gpu
def test_scoring_errors():
    from fastllm_b200 import _lib, models
    cfg, w, _ = golden_weights("mistral")
    model, _ = product_model(cfg, w)
    lib = model.dev.lib
    c = models.DeviceCache(model.dev, 2, 64)
    ids = synth.token_ids(5, cfg.vocab_size, (2, 6))
    c.forward(ids, 0)
    bad = ids.copy()
    bad[1, 3] = cfg.vocab_size
    with pytest.raises(_lib.FastllmError) as e:
        c.forward_logprobs(ids, bad, 6)
    assert e.value.code == -1 and c.kv_len() == 6
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    lp = np.empty((2, 6), dtype=np.float32)
    assert lib.fl_forward_logprobs(model.dev.h, c.h, ptr(ids), None, 2, 6, 6, ptr(lp), None) == -1
    assert lib.fl_forward_logprobs(model.dev.h, c.h, ptr(ids), ptr(ids), 2, 6, 6, None, None) == -1
    assert c.kv_len() == 6
    # argmax_ids = NULL: the same log-probs
    want, _ = models.DeviceCache(model.dev, 2, 64).forward_logprobs(ids, ids, 0)
    c2 = models.DeviceCache(model.dev, 2, 64)
    assert lib.fl_forward_logprobs(model.dev.h, c2.h, ptr(ids), ptr(ids), 2, 6, 0, ptr(lp), None) == 0
    assert np.array_equal(lp, want) and c2.kv_len() == 6
    # a cache driven by sequence slots
    c3 = models.DeviceCache(model.dev, 2, 64)
    c3.forward_slots([0], ids[:1], [0])
    with pytest.raises(_lib.FastllmError) as e:
        c3.forward_logprobs(ids, ids, 0)
    assert e.value.code == -3


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["qwen2", "llama"])
def test_adapter_scoring_leaves_the_generate_cache_alone(name):
    """_CausalBase.logprobs scores on a cache of its own: a generation with scoring calls between its steps is bit-identical to one
    without them, for the position-per-call (Mistral / Qwen2) and the caller-position (Llama) adapters."""
    from fastllm_b200 import models
    cfg, w, _ = golden_weights(name)
    ids = synth.token_ids(3, cfg.vocab_size, (1, 7))

    def run(score):
        m, _ = product_model(cfg, w)
        cache = m.initialize_cache()
        out, scores = [np.asarray(m.forward(ids, 0, cache)).reshape(-1)], []
        for s in range(3):
            if score:
                scores.append(m.logprobs(ids, ids)[0])
            tok = np.array([[models.sample_argmax(out[-1])]], dtype=np.uint32)
            out.append(np.asarray(m.forward(tok, 7 + s, cache)).reshape(-1))
        return out, scores

    want, _ = run(False)
    got, scores = run(True)
    assert all(np.array_equal(a, b) for a, b in zip(want, got))
    assert all(np.array_equal(scores[0], x) for x in scores[1:])      # reset before every call: the same scores each time
    m, c = product_model(cfg, w)
    total, greedy = models.Model(m, c).loglikelihood(ids[0, :3], ids[0, 3:])
    assert np.isfinite(total) and total < 0 and isinstance(greedy, bool)


@pytest.mark.gpu
def test_tinyllama_full_depth_scores_the_golden_continuation():
    """TinyLlama-1.1B (22 layers, synthetic seed 0) scores prompt + golden ids[:63] in ONE 191-token call: position 127 + s predicts
    golden id s; its arg-max is that id wherever the golden margin allows, and its log-prob matches the committed f32 logits."""
    from fastllm_b200 import models, presets
    g = json.load(open(os.path.join(GOLDEN, "fulldepth_tinyllama.json")))
    z = np.load(os.path.join(GOLDEN, "fulldepth_tinyllama_logits.npz"))
    prompt = synth.token_ids(int(g["prompt_seed"]), ocl.TINYLLAMA.vocab_size, (128,))
    assert np.array_equal(prompt, z["prompt"])
    gids = np.asarray(g["ids"], dtype=np.uint32)
    ids = np.concatenate([prompt, gids[:63]])[None]
    tg = np.concatenate([prompt[1:], gids])[None]
    cls, cf = presets.PRESETS["tinyllama"]
    model, _ = cls.initialize_model(cf, None, "bf16", 0, random_seed=0, std=0.02)
    lp, am = model.logprobs(ids, tg)
    steps = np.arange(64)
    sure = np.asarray(g["margins"]) > 2 * LOGIT_TOL_FULL
    wrong = [int(s) for s in steps[sure] if am[0, 127 + s] != gids[s]]
    errs = {s: abs(float(lp[0, 127 + s]) - float(log_softmax64(z[f"logits_{s}"])[gids[s]])) for s in (0, 31, 63)}
    print(f"TinyLlama 22L, one 191-token scoring call: arg-max == golden id at {int(sure.sum()) - len(wrong)} of {int(sure.sum())} "
          f"steps with margin > {2 * LOGIT_TOL_FULL}; log-prob err vs golden logits {errs}")
    assert not wrong and max(errs.values()) <= 2 * LOGIT_TOL_FULL


@pytest.mark.gpu
def test_true_width_real_vocab_qwen():
    """Qwen2.5-7B per-layer shapes, 2 layers, the real 152064-token vocabulary (594 vocab tiles, the last one partial), t = 300."""
    from dataclasses import replace
    from fastllm_b200 import models
    cfg = replace(ocl.QWEN25_7B, num_hidden_layers=2, max_position_embeddings=512)
    w = ocl.synth_weights(cfg, 0, 0.02)
    model, _ = product_model(cfg, w)
    ids = synth.token_ids(1, cfg.vocab_size, (1, 300))
    tg = _targets(2, cfg.vocab_size, (1, 300))
    lp, am = models.DeviceCache(model.dev, 1, 512).forward_logprobs(ids, tg, 0)
    z = logits_all(ocl.CausalLM(cfg, w, kv_dtype="bf16"), ids, 0, per_position=False)
    _check_against(lp, am, z, tg, 2 * KERNEL_TOL_WIDE, "qwen25_7b 2L real vocab t=300")


@pytest.mark.gpu
def test_cpp_mirror_loglikelihood_equals_the_python_mirror(tmp_path):
    from fastllm_b200 import models
    from test_host_cpp_gpu import EXE, _write_inputs
    cfg, w, _ = golden_weights("llama_gqa8")
    _write_inputs(str(tmp_path), cfg, w)
    ctx = [int(x) for x in synth.token_ids(7, cfg.vocab_size, (17,))]
    cont = [int(x) for x in synth.token_ids(8, cfg.vocab_size, (6,))]
    out = subprocess.run([EXE, str(tmp_path / "manifest.txt"), str(tmp_path / "weights.bin"), "0", "--loglikelihood"]
                         + [str(t) for t in ctx] + ["/"] + [str(t) for t in cont], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    got = json.loads(out.stdout.strip().splitlines()[0])
    model, cache = product_model(cfg, w)
    want = models.Model(model, cache).loglikelihood(ctx, cont)
    print(f"loglikelihood: C++ {got}, Python {want}")
    assert got[0] == want[0] and got[1] == want[1]
