"""fl_forward_packed on the device: new prompts and decode steps of running requests, of different lengths, in ONE forward.

Every row is checked against a per-sequence oracle with the cache's bf16 K/V rounding, and later steps show that the K/V pages went
to the right slots.  Also: the tcgen05 prefill work items (head_dim 64 / 128), independence of the caller's order, equal lengths
being fl_forward_slots bit for bit, slot bookkeeping, every error code, Mistral-7B at its true width, and the Python and C++
PackedBatcher."""
import ctypes as C
import json
import subprocess
from dataclasses import replace

import numpy as np
import pytest

from oracle import causal_lm as ocl
from oracle import synth

from helpers import TINY, golden_weights, product_model

pytestmark = pytest.mark.gpu

KERNEL_TOL = 3e-3       # a call's rows against the oracle (tests/test_parity_gpu.py)
LONG_TOL = 1e-2         # long dense-path decode against the oracle (tests/test_zz_widening_gpu.py)
FL_ERR_INVALID, FL_ERR_STATE, FL_ERR_UNSUPPORTED = -1, -3, -5

# the shapes of tests/test_attn_streamk_gpu.py: head_dim 64 (GQA 2, and a 100-token window) and head_dim 128 (GQA 4)
TC_CASES = {
    "d64_gqa2": ocl.CausalLMConfig("llama", 256, 352, 384, 2, 4, 2, 1e-5, 1e4, 1024),
    "d64_window": ocl.CausalLMConfig("mistral", 256, 352, 384, 2, 4, 2, 1e-5, 1e4, 1024, 100),
    "d128_gqa4": ocl.CausalLMConfig("qwen2", 512, 704, 384, 2, 4, 1, 1e-6, 1e6, 1024, 4096, qkv_bias=True),
}


class _Seq:
    """One request: its slot, its oracle (bf16 K/V like the cache) and the adapter's RoPE rule."""

    def __init__(self, cfg, w, slot):
        self.slot, self.oracle, self.pos = slot, ocl.CausalLM(cfg, w, kv_dtype="bf16"), 0
        self.per_call = cfg.arch != "llama"          # Mistral / Qwen2 adapters: RoPE offset + 1 per call

    def feed(self, ids):
        """-> RoPE offset of this call; the oracle's logits of its last position in self.want"""
        ro = self.pos
        self.want = self.oracle.forward(np.asarray(ids, dtype=np.uint32)[None], ro)[0]
        self.pos += 1 if self.per_call else len(ids)
        return ro


def _packed(cache, seqs, parts):
    """One packed call: parts[i] fed to seqs[i]; -> per-row max-abs error against the oracles"""
    ropes = [s.feed(p) for s, p in zip(seqs, parts)]
    got = cache.forward_packed([s.slot for s in seqs], parts, ropes)
    return [float(np.abs(got[i] - s.want).max()) for i, s in enumerate(seqs)], got


def _mixed_call_then_steps(cfg, w, cache, first, fresh, cont=None, steps=6):
    """Prefill `first` (slot -> prompt length) with lone forward_slots calls, then ONE packed call: a decode row for each of them,
    the `fresh` prompts (slot -> length) and, optionally, `cont` = (slot of `first`, length): a multi-token sequence on a non-empty
    slot.  Then `steps` decode steps alternating forward_packed / forward_slots.  -> (packed-call errors, later errors)"""
    from fastllm_b200 import models
    seqs = {}
    for slot, n in first.items():
        s = _Seq(cfg, w, slot)
        prompt = synth.token_ids(500 + slot, cfg.vocab_size, (n,))
        got = cache.forward_slots([slot], prompt[None], [s.feed(prompt)])[0]
        s.tok = models.sample_argmax(got)
        seqs[slot] = s
    rows, parts = [], []
    for slot, s in seqs.items():
        rows.append(s)
        if cont is not None and cont[0] == slot:
            parts.append(synth.token_ids(600 + slot, cfg.vocab_size, (cont[1],)))
        else:
            parts.append(np.array([s.tok], dtype=np.uint32))
    for slot, n in fresh.items():
        s = _Seq(cfg, w, slot)
        seqs[slot] = s
        rows.append(s)
        parts.append(synth.token_ids(700 + slot, cfg.vocab_size, (n,)))
    perm = np.random.RandomState(len(rows)).permutation(len(rows))      # the caller's order is not the internal one
    rows, parts = [rows[i] for i in perm], [parts[i] for i in perm]
    errs, got = _packed(cache, rows, parts)
    for i, s in enumerate(rows):
        s.tok = models.sample_argmax(got[i])
    later = []
    for k in range(steps):
        order = sorted(seqs)
        ids = [np.array([seqs[s].tok], dtype=np.uint32) for s in order]
        ropes = [seqs[s].feed(ids[i]) for i, s in enumerate(order)]
        if k % 2 == 0:
            got = cache.forward_packed(order, ids, ropes)
        else:
            got = cache.forward_slots(order, np.stack(ids), ropes)
        for i, s in enumerate(order):
            later.append(float(np.abs(got[i] - seqs[s].want).max()))
            seqs[s].tok = models.sample_argmax(got[i])
    return errs, later, seqs


@pytest.mark.parametrize("name", ["llama_gqa8", "mistral", "mistral_sw", "qwen2", "mixtral"])
def test_mixed_call_against_the_oracle(name):
    """Two decode rows on non-empty slots, fresh prompts of 5, 70 and 130 tokens (one, two and three pages) and, on Mistral / Qwen2,
    a 7-token continuation of a non-empty slot, in one call; then six more steps, which read the K/V pages the call wrote."""
    from fastllm_b200 import models
    cfg = replace(TINY[name], max_position_embeddings=512)
    w = ocl.synth_weights(cfg, 31, 0.08)
    model, _ = product_model(cfg, w)
    cache = models.DeviceCache(model.dev, 8, 256)
    first = {1: 9, 6: 12}
    cont = None
    if cfg.arch != "llama":
        first[2] = 6
        cont = (2, 7)
    errs, later, seqs = _mixed_call_then_steps(cfg, w, cache, first, {0: 5, 3: 70, 5: 130}, cont)
    print(f"{name}: packed call max err {max(errs):.2e}, later steps {max(later):.2e}")
    assert max(errs) <= KERNEL_TOL
    assert max(later) <= LONG_TOL
    lens = {1: 9 + 7, 6: 12 + 7, 0: 5 + 6, 3: 70 + 6, 5: 130 + 6}
    if cont is not None:
        lens[2] = 6 + 7 + 6
    assert [cache.slot_len(s) for s in range(8)] == [lens.get(s, 0) for s in range(8)]


def test_mixtral_routing_is_reported_in_ids_order():
    """fl_cache_moe_routing after a packed call: row r of the record is row r of the caller's ids, whatever order the rows ran in."""
    from fastllm_b200 import models
    cfg = replace(TINY["mixtral"], max_position_embeddings=512)
    w = ocl.synth_weights(cfg, 31, 0.08)
    model, _ = product_model(cfg, w)
    packed, lone = models.DeviceCache(model.dev, 4, 256), models.DeviceCache(model.dev, 4, 256)
    parts = [synth.token_ids(800 + i, cfg.vocab_size, (n,)) for i, n in enumerate([5, 40, 1, 17])]
    for c in (packed, lone):
        c.forward_slots([2], np.array([[7, 8, 9]], dtype=np.uint32), [0])
    slots = [0, 1, 2, 3]
    packed.forward_packed(slots, parts, [0, 0, 3, 0])
    ex, mg = packed.moe_routing(sum(len(p) for p in parts))
    o = 0
    for slot, p, ro in zip(slots, parts, [0, 0, 3, 0]):
        lone.forward_slots([slot], p[None], [ro])
        ex1, mg1 = lone.moe_routing(len(p))
        sure = (mg1 > 1e-3) & (mg[:, o:o + len(p)] > 1e-3)      # top-k routing is discontinuous: compare away from near-ties
        assert sure.any()
        assert np.array_equal(ex[:, o:o + len(p)][sure], ex1[sure])
        o += len(p)


@pytest.mark.parametrize("name", list(TC_CASES))
def test_tcgen05_prefill_work_items(name):
    """head_dim 64 / 128: fresh prompts of 65 to 900 tokens take the tcgen05 prefill kernel through its work-item list, next to decode
    rows and a 3-token prompt (mma.sync kernel) in the same call."""
    from fastllm_b200 import models
    cfg = TC_CASES[name]
    w = ocl.synth_weights(cfg, 29, 0.06)
    model, _ = product_model(cfg, w)
    cache = models.DeviceCache(model.dev, 8, 1024)
    cont = (4, 10) if cfg.arch != "llama" else None
    errs, later, _ = _mixed_call_then_steps(cfg, w, cache, {4: 40, 7: 100}, {0: 65, 1: 900, 2: 300, 3: 3, 5: 129}, cont, steps=3)
    print(f"{name}: packed call max err {max(errs):.2e}, later steps {max(later):.2e}")
    # the prefill bar of tests/test_attn_streamk_gpu.py on these shapes (900-token prompts under the hi + lo split)
    assert max(errs) <= LONG_TOL and max(later) <= LONG_TOL


def _two_caches(model, cfg, n=8, max_seq=512):
    from fastllm_b200 import models
    caches = [models.DeviceCache(model.dev, n, max_seq) for _ in range(2)]
    for c in caches:
        for slot, k in ((1, 9), (4, 70)):
            c.forward_slots([slot], synth.token_ids(900 + slot, cfg.vocab_size, (k,))[None], [0])
    return caches


def test_caller_order_does_not_change_a_row():
    from fastllm_b200 import models
    cfg = TC_CASES["d64_window"]
    w = ocl.synth_weights(cfg, 29, 0.06)
    model, _ = product_model(cfg, w)
    a, b = _two_caches(model, cfg)
    slots = [1, 4, 0, 2, 3]
    parts = [np.array([11], np.uint32), np.array([12], np.uint32)] + [synth.token_ids(950 + i, cfg.vocab_size, (n,)) for i, n in
                                                                      enumerate([65, 3, 200])]
    ropes = [1, 1, 0, 0, 0]
    got_a = a.forward_packed(slots, parts, ropes)
    p = [3, 0, 4, 2, 1]
    got_b = b.forward_packed([slots[i] for i in p], [parts[i] for i in p], [ropes[i] for i in p])
    for j, i in enumerate(p):
        assert np.array_equal(got_a[i], got_b[j])
    assert [a.slot_len(s) for s in range(8)] == [b.slot_len(s) for s in range(8)]


@pytest.mark.parametrize("t", [1, 5, 70])
def test_equal_lengths_are_forward_slots(t):
    from fastllm_b200 import models
    cfg = replace(TINY["mistral"], max_position_embeddings=512)
    w = ocl.synth_weights(cfg, 31, 0.08)
    model, _ = product_model(cfg, w)
    a, b = _two_caches(model, cfg)
    slots = [4, 1, 6] if t == 1 else [0, 2, 3]          # decode rows of running requests, or fresh prompts of one length
    ids = synth.token_ids(990 + t, cfg.vocab_size, (3, t))
    ropes = [70, 9, 0] if t == 1 else [0, 0, 0]
    got_p = a.forward_packed(slots, list(ids), ropes)
    got_s = b.forward_slots(slots, ids, ropes)
    assert np.array_equal(got_p, got_s)
    assert [a.slot_len(s) for s in range(8)] == [b.slot_len(s) for s in range(8)]


def test_slot_bookkeeping():
    from fastllm_b200 import FastllmError, models
    cfg = replace(TINY["qwen2"], max_position_embeddings=512)
    w = ocl.synth_weights(cfg, 31, 0.08)
    model, _ = product_model(cfg, w)
    cache = models.DeviceCache(model.dev, 4, 256)
    ids = lambda n, s=0: synth.token_ids(1000 + n + s, cfg.vocab_size, (n,))      # noqa: E731
    cache.forward_packed([0, 2], [ids(9), ids(20)], [0, 0])
    assert [cache.slot_len(s) for s in range(4)] == [9, 0, 20, 0]
    cache.forward_packed([2, 0, 3], [ids(1), ids(4), ids(33)], [1, 1, 0])
    assert [cache.slot_len(s) for s in range(4)] == [13, 0, 21, 33]
    cache.slot_reset(0)
    cache.forward_slots([2, 3], np.array([[5], [6]], dtype=np.uint32), [2, 1])
    cache.forward_packed([0, 3], [ids(8, 1), ids(1)], [0, 2])
    assert [cache.slot_len(s) for s in range(4)] == [8, 0, 22, 35]
    with pytest.raises(FastllmError) as e:       # a slot-driven cache refuses the uniform calls until it is reset
        cache.forward(ids(3)[None], 0)
    assert e.value.code == FL_ERR_STATE
    cache.reset()
    cache.forward(ids(3)[None], 0)
    with pytest.raises(FastllmError) as e:       # and a cache that holds uniform tokens refuses packed calls
        cache.forward_packed([0, 1], [ids(2), ids(3)], [0, 0])
    assert e.value.code == FL_ERR_STATE


def test_errors_leave_the_cache_unchanged(monkeypatch):
    from fastllm_b200 import FastllmError, _lib, models
    cfg = replace(TINY["llama_gqa8"], max_position_embeddings=512)
    w = ocl.synth_weights(cfg, 31, 0.08)
    model, _ = product_model(cfg, w)
    a, b = (models.DeviceCache(model.dev, 4, 128) for _ in range(2))
    for c in (a, b):
        c.forward_slots([1], synth.token_ids(1100, cfg.vocab_size, (9,))[None], [0])
    good = ([0, 1], [synth.token_ids(1101, cfg.vocab_size, (20,)), np.array([7], np.uint32)], [0, 9])
    V = cfg.vocab_size
    cases = [
        (FL_ERR_INVALID, ([], [], [])),                                                        # n < 1
        (FL_ERR_INVALID, ([0, 1, 2, 3, 0], [np.array([3], np.uint32)] * 5, [0] * 5)),          # n > max_batch (and a repeat)
        (FL_ERR_INVALID, ([0, 1], [np.zeros(0, np.uint32), np.array([7], np.uint32)], [0, 9])),   # a length < 1
        (FL_ERR_INVALID, ([0, 4], good[1], good[2])),                                          # slot out of range
        (FL_ERR_INVALID, ([1, 1], [np.array([3], np.uint32), np.array([7], np.uint32)], [9, 9])),  # a slot twice
        (FL_ERR_INVALID, ([0, 1], [np.array([3, V], np.uint32), np.array([7], np.uint32)], [0, 9])),  # id >= vocab
        (FL_ERR_INVALID, ([0, 1], good[1], [cfg.max_position_embeddings - 19, 9])),            # RoPE position beyond the table
        (FL_ERR_INVALID, ([0, 1], [good[1][0], np.array([7, 8], np.uint32)], [0, 9])),         # Llama: multi-token on a non-empty slot
        (FL_ERR_STATE, ([0, 1], [synth.token_ids(1102, V, (129,)), np.array([7], np.uint32)], [0, 9])),   # slot_len + length > max_seq
    ]
    for code, (slots, parts, ropes) in cases:
        with pytest.raises(FastllmError) as e:
            a.forward_packed(slots, parts, ropes)
        assert e.value.code == code, (slots, [len(p) for p in parts])
    lib = _lib.load()
    out = np.empty((2, V), np.float32)
    rc = lib.fl_forward_packed(model.dev.h, a.h, None, None, 2, None, None, out.ctypes.data_as(C.c_void_p))
    assert rc == FL_ERR_INVALID                                                                 # NULL pointers
    assert [a.slot_len(s) for s in range(4)] == [0, 9, 0, 0]
    assert np.array_equal(a.forward_packed(*good), b.forward_packed(*good))
    # a model whose shapes keep it off the dense path cannot take packed calls
    monkeypatch.setenv("FL_NO_DENSE", "1")
    off, _ = product_model(cfg, w)
    c = models.DeviceCache(off.dev, 2, 64)
    with pytest.raises(FastllmError) as e:
        c.forward_packed([0, 1], [np.array([3, 4], np.uint32), np.array([5], np.uint32)], [0, 0])
    assert e.value.code == FL_ERR_UNSUPPORTED


def test_mistral_7b_true_width():
    """Mistral-7B (synthetic weights, the real 32 000-token vocabulary): 3 decode rows and prompts of 17, 300 and 1000 tokens in one
    call against lone forward_slots calls of each sequence.  Different kernels and summation orders, so: the arg-max agrees wherever
    the top-2 gap is more than twice the observed error."""
    from fastllm_b200 import models, presets
    cls, cf = presets.PRESETS["mistral7b"]
    model, _ = cls.initialize_model(cf, None, "bf16", 0, random_seed=0)
    V = cf.vocab_size
    a, b = (models.DeviceCache(model.dev, 8, 1100) for _ in range(2))
    for c in (a, b):
        for slot, n in ((0, 20), (3, 50), (5, 80)):
            c.forward_slots([slot], synth.token_ids(1200 + slot, V, (n,))[None], [0])
    slots = [1, 0, 2, 3, 4, 5]
    parts = [synth.token_ids(1300 + s, V, (n,)) for s, n in ((1, 17), (0, 1), (2, 300), (3, 1), (4, 1000), (5, 1))]
    ropes = [0, 1, 0, 1, 0, 1]
    got = a.forward_packed(slots, parts, ropes)
    errs = []
    for i, (s, p, r) in enumerate(zip(slots, parts, ropes)):
        want = b.forward_slots([s], p[None], [r])[0]
        err = float(np.abs(got[i] - want).max())
        errs.append(err)
        top2 = np.sort(want)[-2:]
        if top2[1] - top2[0] > 2 * err:
            assert models.sample_argmax(got[i]) == models.sample_argmax(want)
    assert np.isfinite(got).all()
    print(f"mistral7b packed vs lone calls: max-abs logits err per row {['%.2e' % e for e in errs]}")


def test_packed_batcher_tokens_are_the_per_request_argmax():
    """PackedBatcher on the device: 7 requests over 3 slots.  Packed steps run the dense path while a lone request runs the persistent
    / GEMV path, so (as for ContinuousBatcher) the check is teacher-forced: every emitted token is the arg-max of the single-sequence
    logits up to twice the kernel tolerance.  Admitting prompts into the decode steps takes fewer forwards."""
    from fastllm_b200 import models
    cfg, w, g = golden_weights("mistral")
    model, _ = product_model(cfg, w)
    lengths = [9, 3, 40, 9, 17, 70, 5]
    prompts = [list(map(int, synth.token_ids(140 + i, cfg.vocab_size, (n,)))) for i, n in enumerate(lengths)]
    pb = models.PackedBatcher(model, max_batch=3, eos_token_id=None)
    outs = pb.generate(prompts, 6)
    assert [len(t) for t in outs] == [6] * len(prompts)
    cb = models.ContinuousBatcher(model, max_batch=3, eos_token_id=None)
    cb.generate(prompts, 6)
    assert pb.forwards < cb.steps + len(prompts)
    for p, toks in zip(prompts, outs):
        c = model.initialize_cache()
        logits = np.asarray(model.forward(np.asarray([p], dtype=np.uint32), 0, c))[0].reshape(-1)
        pos = len(p)
        for tok in toks:
            assert logits[tok] >= logits.max() - 2 * KERNEL_TOL
            logits = np.asarray(model.forward(np.array([[tok]], dtype=np.uint32), pos, c))[0].reshape(-1)
            pos += 1


def test_cpp_packed_batcher_equals_the_python_mirror(tmp_path):
    """host/fastllm_host.hpp PackedBatcher (compiled, `host_selftest --packed`) issues the same fl_forward_packed calls as the Python
    PackedBatcher: the ids must be identical (5 requests of different lengths over 2 slots)."""
    from fastllm_b200 import models
    from test_host_cpp_gpu import EXE, _write_inputs
    cfg, w, g = golden_weights("llama_gqa8")
    _write_inputs(str(tmp_path), cfg, w)
    prompts = [list(map(int, synth.token_ids(200 + i, cfg.vocab_size, (n,)))) for i, n in enumerate([7, 3, 19, 5, 11])]
    args = []
    for i, p in enumerate(prompts):
        args += (["/"] if i else []) + [str(t) for t in p]
    out = subprocess.run([EXE, str(tmp_path / "manifest.txt"), str(tmp_path / "weights.bin"), "5", "--packed", "2"] + args,
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    model, _ = product_model(cfg, w)
    want = models.PackedBatcher(model, max_batch=2, eos_token_id=None).generate(prompts, 5)
    assert json.loads(out.stdout.strip().splitlines()[0]) == want
