"""KV page pools and slot forks on the device (fl_cache_create_pool, fl_cache_slot_fork).

Every kernel reads and writes K/V through the page table; with a pool smaller than max_batch * pages_per_seq the test slots hold
scrambled, non-home pages next to live "garbage" sequences, and every call must return the logits of the same call on a default
cache bit for bit.  Also: exhaustion of every entry point, forks (page cost, bitwise continuation, untouched shared pages, every
error code), a prefix continuation against the oracle, Mistral-7B at 256 slots x 32 768 tokens on a 65 536-token pool, and the
Python and C++ PackedBatcher with a pool and a shared prefix."""
import json
import os
import subprocess
import tempfile
from dataclasses import replace

import numpy as np
import pytest

from oracle import causal_lm as ocl
from oracle import synth

from helpers import TINY, golden_weights, product_model

pytestmark = pytest.mark.gpu

KERNEL_TOL = 3e-3       # a call's rows against the oracle (tests/test_parity_gpu.py)
FL_ERR_INVALID, FL_ERR_STATE = -1, -3

CASES = {
    "llama": replace(TINY["llama"], max_position_embeddings=512),
    "mistral_sw": replace(TINY["mistral_sw"], max_position_embeddings=512),
    "qwen2": TINY["qwen2"],
    "mixtral": TINY["mixtral"],
    # head_dim 64 (a 100-token window) and 128: fresh prompts of more than a page run on the tcgen05 prefill kernel
    "d64_window": ocl.CausalLMConfig("mistral", 256, 352, 384, 2, 4, 2, 1e-5, 1e4, 1024, 100),
    "d128_gqa4": ocl.CausalLMConfig("qwen2", 512, 704, 384, 2, 4, 1, 1e-6, 1e6, 1024, 4096, qkv_bias=True),
}


def _model(cfg, seed=31):
    w = ocl.synth_weights(cfg, seed, 0.08)
    model, _ = product_model(cfg, w)
    return model, w


def _ids(seed, cfg, n):
    return synth.token_ids(seed, cfg.vocab_size, (n,))


def _code(fn):
    from fastllm_b200._lib import FastllmError
    with pytest.raises(FastllmError) as e:
        fn()
    return e.value.code


def _garbage(cache, cfg):
    """Admit, decode and reset sequences in slots 4-7.  On the 20-page pool (home pages for slots 0-4 only) slots 5 / 6 / 7 take pages
    [0, 4] / [1, 5] / [2, 3]; resetting slot 6 leaves pages 1 and 5 free between live ones, so the first test prompt (slot 0, 130
    tokens, three pages: a tcgen05 prefill at head_dim 64 / 128) lands on pages 1, 5, 6 -- neither its home pages nor contiguous."""
    cache.forward_packed([5, 6, 7], [_ids(900, cfg, 64), _ids(901, cfg, 64), _ids(902, cfg, 100)], [0, 0, 0])
    cache.forward_packed([5, 6, 7], [_ids(903, cfg, 1), _ids(904, cfg, 1), _ids(905, cfg, 1)], [1, 1, 1])
    cache.slot_reset(6)
    cache.forward_packed([4], [_ids(906, cfg, 65)], [0])


@pytest.mark.parametrize("name", list(CASES))
def test_scrambled_pages_are_bitwise_equal_to_the_default_cache(name):
    """Slot and packed calls on scattered pages: fresh prompts of one to three pages (mma.sync / tcgen05 prefill), mixed packed calls,
    stream-K decode steps, dense-path slot calls and, on Mistral / Qwen2, continuations of non-empty slots."""
    from fastllm_b200 import models
    cfg = CASES[name]
    model, _ = _model(cfg)
    ref = models.DeviceCache(model.dev, 8, 256)
    pool = models.DeviceCache(model.dev, 8, 256, pool_tokens=20 * 64)
    assert pool.pool_pages() == (20, 20) and ref.pool_pages() == (32, 32)
    calls = [("packed", [0, 1, 2], [_ids(10, cfg, 130), _ids(11, cfg, 5), _ids(12, cfg, 70)], [0, 0, 0])]
    for k in range(3):
        calls.append(("slots", [0, 1, 2], [_ids(20 + k, cfg, 1) for _ in range(3)], [130 + k, 5 + k, 70 + k]))
    calls.append(("packed", [3, 0, 2], [_ids(30, cfg, 90), _ids(31, cfg, 1), _ids(32, cfg, 1)], [0, 133, 73]))
    if cfg.arch != "llama":
        calls.append(("packed", [1, 0], [_ids(40, cfg, 7), _ids(41, cfg, 1)], [8, 134]))
        calls.append(("slots", [1], [_ids(42, cfg, 9)], [15]))
    for k in range(60):      # decode across page boundaries: slot 1 from 24 to 84 tokens, slot 3 from 90 to 150
        calls.append(("slots", [0, 1, 2, 3], [_ids(50 + k, cfg, 1) for _ in range(4)], [140 + k, 30 + k, 80 + k, 90 + k]))
    for c in (ref, pool):
        _garbage(c, cfg)
    assert pool.pool_pages()[0] == 20 - 6
    for kind, slots, parts, ropes in calls:
        got = []
        for c in (ref, pool):
            if kind == "packed":
                got.append(c.forward_packed(slots, parts, ropes))
            else:
                got.append(c.forward_slots(slots, np.stack(parts), ropes))
        assert np.array_equal(got[0], got[1], equal_nan=True), (name, kind, slots)
        assert np.isfinite(got[1]).all()
    lens = [ref.slot_len(s) for s in range(8)]
    assert [pool.slot_len(s) for s in range(8)] == lens
    used = sum(-(-n // 64) for n in lens)
    assert pool.pool_pages() == (20 - used, 20)
    for s in range(8):
        pool.slot_reset(s)
    assert pool.pool_pages() == (20, 20)


@pytest.mark.parametrize("name", ["llama", "mistral_sw", "qwen2", "mixtral"])
def test_uniform_calls_on_non_home_pages(name):
    """Uniform calls: 2 rows (GEMV path) on a pool of one slot's pages, so slot 1 has no home page and the two slots' pages
    interleave; 3 rows (dense path) on a pool without slot 2's home pages.  Prompt, then decode steps across page boundaries."""
    from fastllm_b200 import models
    cfg = CASES[name]
    model, _ = _model(cfg)
    for b, pool_pages in ((2, 4), (3, 6)):
        ref = models.DeviceCache(model.dev, 4, 256)
        pool = models.DeviceCache(model.dev, 4, 256, pool_tokens=pool_pages * 64)
        steps = [(np.stack([_ids(60 + i, cfg, 40) for i in range(b)]), 0)]
        steps += [(np.stack([_ids(100 + 10 * k + i, cfg, 1) for i in range(b)]), 40 + k) for k in range(60)]
        for ids, ro in steps:
            a, p = ref.forward(ids, ro), pool.forward(ids, ro)
            assert np.array_equal(a, p, equal_nan=True), (name, b, ro)
        assert pool.pool_pages() == (pool_pages - 2 * b, pool_pages)
        pool.reset()
        assert pool.pool_pages() == (pool_pages, pool_pages)


def test_fill_and_slot_reset_keep_pages_and_lengths_consistent():
    """fl_cache_fill_synthetic turns a slot-driven cache into a uniform one (slot lengths 0, its slots' pages only); fl_cache_slot_reset
    on a cache of uniform calls keeps the row's pages, which the common length still covers."""
    from fastllm_b200 import models
    cfg = CASES["mistral_sw"]
    model, _ = _model(cfg)
    c = models.DeviceCache(model.dev, 4, 256, pool_tokens=6 * 64)
    c.forward_slots([1], _ids(97, cfg, 100)[None], [0])
    c.fill_synthetic(2, 70)
    assert [c.slot_len(s) for s in range(4)] == [0] * 4 and c.kv_len() == 70 and c.pool_pages() == (2, 6)
    c.forward(np.stack([_ids(98, cfg, 1)] * 2), 70)           # a uniform call is accepted after the fill
    c.slot_reset(1)
    assert c.pool_pages() == (2, 6)
    assert np.isfinite(c.forward(np.stack([_ids(99, cfg, 1)] * 2), 71)).all()
    c.reset()
    assert c.pool_pages() == (6, 6)


def test_exhaustion_of_every_entry_point_changes_nothing():
    from fastllm_b200 import models
    cfg = CASES["mistral_sw"]
    model, _ = _model(cfg)
    pool, twin = (models.DeviceCache(model.dev, 4, 256, pool_tokens=128) for _ in range(2))
    big = np.stack([_ids(1, cfg, 65), _ids(2, cfg, 65)])                   # 2 x 2 pages > 2
    lp = models.LogitsProcessor(0, 0.7)
    uniform = [lambda: pool.forward(big, 0), lambda: pool.forward_greedy(big, 0), lambda: pool.forward_logprobs(big, big, 0),
               lambda: pool.forward_sample(big, 0, lp), lambda: pool.forward_sample_device(big, 0, lp),
               lambda: pool.decode_greedy_loop(np.array([3], dtype=np.uint32), 0, 129), lambda: pool.fill_synthetic(3, 64)]
    for fn in uniform:
        assert _code(fn) == FL_ERR_STATE
        assert pool.pool_pages() == (2, 2) and pool.kv_len() == 0
    ids = np.stack([_ids(3, cfg, 10), _ids(4, cfg, 10)])
    assert np.array_equal(pool.forward(ids, 0), twin.forward(ids, 0))
    assert pool.pool_pages() == (0, 2) and pool.kv_len() == 10
    pool.reset(), twin.reset()
    assert pool.pool_pages() == (2, 2)
    assert _code(lambda: pool.forward_slots([0, 1, 2], np.stack([_ids(5 + i, cfg, 50) for i in range(3)]), [0, 0, 0])) == FL_ERR_STATE
    assert _code(lambda: pool.forward_packed([0, 1], [_ids(8, cfg, 100), _ids(9, cfg, 50)], [0, 0])) == FL_ERR_STATE
    assert pool.pool_pages() == (2, 2) and [pool.slot_len(s) for s in range(4)] == [0] * 4
    parts = [_ids(10, cfg, 60), _ids(11, cfg, 10)]
    assert np.array_equal(pool.forward_packed([0, 1], parts, [0, 0]), twin.forward_packed([0, 1], parts, [0, 0]))
    assert pool.pool_pages() == (0, 2)
    assert _code(lambda: pool.forward_slots([0, 1], np.stack([_ids(12, cfg, 5)] * 2), [1, 1])) == FL_ERR_STATE   # slot 0 needs a page
    pool.slot_reset(1), twin.slot_reset(1)
    assert pool.pool_pages() == (1, 2)
    step = np.stack([_ids(13, cfg, 5)])
    assert np.array_equal(pool.forward_slots([0], step, [1]), twin.forward_slots([0], step, [1]))
    assert pool.pool_pages() == (0, 2)


@pytest.mark.parametrize("src_len", [100, 128])
def test_fork(src_len):
    """fork costs one page for a partial last page, none at a multiple of 64; the fork continues as its source would, bit for bit;
    the shared pages are never written (the source still equals an unforked control after both decode), and resetting the source
    leaves the fork's results unchanged."""
    from fastllm_b200 import models
    cfg = CASES["mistral_sw"]
    model, _ = _model(cfg)
    a = models.DeviceCache(model.dev, 4, 256, pool_tokens=16 * 64)
    twin, control = models.DeviceCache(model.dev, 4, 256), models.DeviceCache(model.dev, 4, 256)
    prompt = _ids(70, cfg, src_len)
    for c in (a, twin, control):
        c.forward_slots([0], prompt[None], [0])
    free = a.pool_pages()[0]
    a.slot_fork(0, 1)
    assert a.pool_pages()[0] == free - (1 if src_len % 64 else 0)
    assert a.slot_len(1) == src_len
    tok = _ids(71, cfg, 1)[None]
    assert np.array_equal(a.forward_slots([1], tok, [1]), twin.forward_slots([0], tok, [1]))      # the fork = its source
    for k in range(70):                      # both decode across a page boundary; the source on its own, like the control
        s_tok, d_tok = _ids(200 + k, cfg, 1)[None], _ids(300 + k, cfg, 1)[None]
        assert np.array_equal(a.forward_slots([0], s_tok, [1 + k]), control.forward_slots([0], s_tok, [1 + k]))
        assert np.array_equal(a.forward_slots([1], d_tok, [2 + k]), twin.forward_slots([0], d_tok, [2 + k]))
    a.slot_reset(0)
    a.forward_packed([0, 2], [_ids(80, cfg, 90), _ids(81, cfg, 30)], [0, 0])      # new sequences take the freed pages
    for k in range(5):
        d_tok = _ids(400 + k, cfg, 1)[None]
        assert np.array_equal(a.forward_slots([1], d_tok, [72 + k]), twin.forward_slots([0], d_tok, [72 + k]))


def test_fork_errors_leave_the_cache_unchanged():
    from fastllm_b200 import models
    cfg = CASES["mistral_sw"]
    model, _ = _model(cfg)
    c = models.DeviceCache(model.dev, 4, 256, pool_tokens=3 * 64)
    c.forward_slots([0], _ids(90, cfg, 100)[None], [0])
    c.forward_slots([2], _ids(91, cfg, 10)[None], [0])
    state = lambda: (c.pool_pages(), [c.slot_len(s) for s in range(4)])
    before = state()
    assert before == ((0, 3), [100, 0, 10, 0])
    for src, dst in ((0, 0), (-1, 1), (0, 4), (1, 3)):              # same slot, out of range, empty source
        assert _code(lambda: c.slot_fork(src, dst)) == FL_ERR_INVALID
        assert state() == before
    assert _code(lambda: c.slot_fork(0, 2)) == FL_ERR_STATE           # destination not empty
    assert _code(lambda: c.slot_fork(0, 1)) == FL_ERR_STATE           # no free page for the partial last page
    assert state() == before
    u = models.DeviceCache(model.dev, 2, 128, pool_tokens=256)
    u.forward(np.stack([_ids(92, cfg, 5)]), 0)
    assert _code(lambda: u.slot_fork(0, 1)) == FL_ERR_STATE           # tokens of uniform calls
    assert u.pool_pages() == (3, 4) and u.kv_len() == 5
    assert _code(lambda: u.slot_fork(1, 0)) == FL_ERR_STATE


@pytest.mark.parametrize("name", ["mistral", "qwen2"])
@pytest.mark.parametrize("plen", [64, 70])
def test_prefix_continuation_matches_the_one_call_prompt(name, plen):
    """A prompt fed as a forked prefix (a whole page, and a page and a bit) plus its suffix at RoPE offset len(prefix) against the
    bf16-KV oracle of the one-call prompt."""
    from fastllm_b200 import models
    cfg = TINY[name]
    model, w = _model(cfg)
    c = models.DeviceCache(model.dev, 4, 256, pool_tokens=8 * 64)
    prompt = _ids(95, cfg, plen + 20)
    c.forward_slots([0], prompt[None, :plen], [0])
    c.slot_fork(0, 2)
    got = c.forward_slots([2], prompt[None, plen:], [plen])[0]
    want = ocl.CausalLM(cfg, w, kv_dtype="bf16").forward(prompt[None], 0)[0]
    assert float(np.abs(got - want).max()) <= KERNEL_TOL


def test_mistral_7b_256_slots_on_a_65536_token_pool():
    """256 slots of 32 768 tokens would take 1.1 TB of KV at a static layout; a 65 536-token pool (8.6 GB) serves a packed step."""
    from fastllm_b200 import models, presets
    cls, cf = presets.PRESETS["mistral7b"]
    model, _ = cls.initialize_model(cf, None, "bf16", 0, random_seed=0)
    c = models.DeviceCache(model.dev, 256, 32768, pool_tokens=65536)
    assert c.pool_pages() == (1024, 1024)
    V = cf.vocab_size
    slots = [0, 100, 255]
    c.forward_packed(slots, [synth.token_ids(1400 + s, V, (n,)) for s, n in zip(slots, (300, 17, 1000))], [0, 0, 0])
    got = c.forward_packed(slots + [7], [synth.token_ids(1500 + s, V, (1,)) for s in slots] + [synth.token_ids(1600, V, (50,))],
                           [1, 1, 1, 0])
    assert np.isfinite(got).all()
    assert c.pool_pages() == (1024 - (5 + 1 + 16 + 1), 1024)


def test_packed_batcher_with_a_pool_and_a_shared_prefix():
    """PackedBatcher on a pool smaller than max_batch x capacity, with a shared prefix: every emitted token is the arg-max of the
    lone request's logits up to twice the kernel tolerance (the check of test_packed_batcher_tokens_are_the_per_request_argmax); the
    prefix is prefilled once; and the C++ mirror emits the same ids."""
    from fastllm_b200 import models
    from test_host_cpp_gpu import EXE, _write_inputs
    cfg, w, g = golden_weights("mistral")
    model, _ = product_model(cfg, w)
    prefix = list(map(int, _ids(150, cfg, 70)))
    prompts = [prefix + list(map(int, _ids(160 + i, cfg, n))) for i, n in enumerate([9, 3, 40, 17])]
    prompts += [list(map(int, _ids(170, cfg, 12))), prefix[:30]]           # no prefix / shorter than it: the normal path
    # 3 pages: the prefix holds 2, so one request runs at a time although a second slot is free
    pb = models.PackedBatcher(model, max_batch=3, eos_token_id=None, pool_tokens=3 * 64)
    outs = pb.generate(prompts, 6, shared_prefix=prefix)
    assert [len(t) for t in outs] == [6] * len(prompts)
    assert pb.prefill_tokens == 70 + 9 + 3 + 40 + 17 + 12 + 30
    assert pb.peak_pages == 3 and pb.cache.pool_pages() == (3, 3)
    for p, toks in zip(prompts, outs):
        c = model.initialize_cache()
        logits = np.asarray(model.forward(np.asarray([p], dtype=np.uint32), 0, c))[0].reshape(-1)
        for tok in toks:
            assert logits[tok] >= logits.max() - 2 * KERNEL_TOL
            logits = np.asarray(model.forward(np.array([[tok]], dtype=np.uint32), 0, c))[0].reshape(-1)
    with tempfile.TemporaryDirectory() as tmp:
        _write_inputs(tmp, cfg, w)
        args = []
        for i, p in enumerate(prompts):
            args += (["/"] if i else []) + [str(t) for t in p]
        out = subprocess.run([EXE, os.path.join(tmp, "manifest.txt"), os.path.join(tmp, "weights.bin"), "6", "--packed-pool", "3",
                              str(3 * 64), "70"] + args, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert json.loads(out.stdout.strip().splitlines()[0]) == outs
