"""FP8 (e4m3) KV caches on the device (fl_cache_create_pool_kv(..., FL_KV_FP8_E4M3, ...)).

Every case runs all three attention kernels on e4m3 pages: stream-K decode rows, fresh prompts of more than a page on the tcgen05
prefill (head_dim 64 / 128, K read from the call's bf16 K scratch) and the mma.sync prefill (short prompts, continuations of
non-empty slots).  Logits are checked against the oracle with e4m3 K / V (kv_fp8_ref.Fp8KvCausalLM; FP8_TOL: why the bar is wider than
the bf16 tests' 3e-3).  The bitwise identities of bf16 caches hold on FP8 caches too: packed = lone slot calls, caller order, scrambled
pools, forks, and refused entry points leave the cache unchanged."""
from dataclasses import replace

import numpy as np
import pytest

from oracle import causal_lm as ocl
from oracle import synth

from helpers import TINY, product_model
from kv_fp8_ref import Fp8KvCausalLM

pytestmark = pytest.mark.gpu

# Logits against the fp8-KV oracle.  The bf16 tests' bar (3e-3) does not hold: the kernel's f32 K and V differ from the oracle's by
# ~1e-5 relative (hi + lo bf16 activations), and e4m3's 2^-3 relative spacing turns the few values that sit that close to a rounding
# boundary into whole-step differences (measured on a B200: up to 6.6e-2 at head_dim 128, 1.6e-2 at 64, 6.4e-3 at 32; the oracle's
# own logits move by 1.2e-3 when its K / V are perturbed by 1e-6 relative before rounding).  The fp8 and bf16 oracles differ by ~1.2
# on the same rows, so the bar still separates the e4m3 rule from bf16 K / V by more than an order of magnitude.
FP8_TOL = 0.1
FL_ERR_INVALID, FL_ERR_STATE, FL_ERR_UNSUPPORTED = -1, -3, -5
FP8 = "fp8_e4m3"

CASES = {
    "llama_d64": ocl.CausalLMConfig("llama", 256, 352, 384, 2, 4, 2, 1e-5, 1e4, 1024),
    "mistral_window_d128": ocl.CausalLMConfig("mistral", 512, 704, 384, 2, 4, 2, 1e-5, 1e4, 1024, 100),
    "qwen2_bias_d128": ocl.CausalLMConfig("qwen2", 512, 704, 384, 2, 4, 1, 1e-6, 1e6, 1024, 4096, qkv_bias=True),
    "mixtral_d64": ocl.CausalLMConfig("mixtral", 256, 352, 384, 2, 4, 2, 1e-5, 1e6, 1024, 4096, num_local_experts=4,
                                      num_experts_per_tok=2),
    "tiny_d32": replace(TINY["mistral"], max_position_embeddings=512),
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


class _Seq:
    """One request: its slot, its oracle (e4m3 K/V like the cache) and the adapter's RoPE rule."""

    def __init__(self, cfg, w, slot):
        self.slot, self.oracle, self.pos = slot, Fp8KvCausalLM(cfg, w), 0
        self.per_call = cfg.arch != "llama"

    def feed(self, ids):
        ro = self.pos
        self.want = self.oracle.forward(np.asarray(ids, dtype=np.uint32)[None], ro)[0]
        self.pos += 1 if self.per_call else len(ids)
        return ro


def _calls(cfg):
    """(kind, slots, parts) of a run through every attention kernel: one packed admission (130 / 70 tokens: tcgen05 at head_dim
    64 / 128; 5 tokens: mma.sync), decode steps across a page boundary (stream-K), a packed call with decode rows, a fresh prompt
    and (Mistral / Qwen2) a continuation of a non-empty slot (mma.sync)."""
    out = [("packed", [0, 1, 2], [_ids(10, cfg, 130), _ids(11, cfg, 5), _ids(12, cfg, 70)])]
    for k in range(4):
        out.append(("slots", [0, 1, 2], [_ids(20 + k, cfg, 1) for _ in range(3)]))
    cont = [("packed", [1], [_ids(40, cfg, 9)])] if cfg.arch != "llama" else []
    out.append(("packed", [3, 0, 2], [_ids(30, cfg, 20), _ids(31, cfg, 1), _ids(32, cfg, 1)]))
    out += cont
    for k in range(3):
        out.append(("slots", [0, 1, 2, 3], [_ids(50 + k, cfg, 1) for _ in range(4)]))
    return out


def _run(cache, cfg, seqs, kind, slots, parts):
    ropes = [seqs[s].feed(p) for s, p in zip(slots, parts)]
    if kind == "packed":
        return cache.forward_packed(slots, parts, ropes)
    return cache.forward_slots(slots, np.stack(parts), ropes)


@pytest.mark.parametrize("name", list(CASES))
def test_slot_and_packed_logits_match_the_fp8_oracle(name):
    from fastllm_b200 import models
    cfg = CASES[name]
    model, w = _model(cfg)
    cache = models.DeviceCache(model.dev, 4, 512, kv_dtype=FP8)
    seqs = {s: _Seq(cfg, w, s) for s in range(4)}
    errs = []
    for kind, slots, parts in _calls(cfg):
        got = _run(cache, cfg, seqs, kind, slots, parts)
        errs += [float(np.abs(got[i] - seqs[s].want).max()) for i, s in enumerate(slots)]
    print(f"{name}: max |logit - fp8 oracle| = {max(errs):.2e}")
    assert max(errs) <= FP8_TOL, (name, errs)


@pytest.mark.parametrize("name", ["llama_d64", "mistral_window_d128", "mixtral_d64", "tiny_d32"])
def test_packed_calls_are_slot_calls_and_do_not_depend_on_order(name):
    """Equal lengths: a packed call is fl_forward_slots bit for bit (prompts of 130 tokens, then decode rows).  Mixed lengths: the
    caller's order of the sequences does not change a bit."""
    from fastllm_b200 import models
    cfg = CASES[name]
    model, _ = _model(cfg)
    packed, lone, rev = (models.DeviceCache(model.dev, 4, 512, kv_dtype=FP8) for _ in range(3))
    for k, n in enumerate([130, 1, 1]):
        parts = [_ids(60 + 3 * k + s, cfg, n) for s in range(3)]
        ropes = [0, 0, 0] if k == 0 else [k, k, k]
        assert np.array_equal(packed.forward_packed([0, 1, 2], parts, ropes), lone.forward_slots([0, 1, 2], np.stack(parts), ropes))
    rev.forward_packed([2, 1, 0], [_ids(62, cfg, 130), _ids(61, cfg, 130), _ids(60, cfg, 130)], [0, 0, 0])
    for k in (1, 2):
        rev.forward_slots([0, 1, 2], np.stack([_ids(60 + 3 * k + s, cfg, 1) for s in range(3)]), [k, k, k])
    step = [_ids(70, cfg, 1), _ids(71, cfg, 1), _ids(72, cfg, 20), _ids(73, cfg, 7)]      # decode rows, a fresh prompt, a continuation
    slots, ropes = [0, 1, 3, 2], [3, 3, 0, 3]
    if cfg.arch == "llama":
        step[3] = _ids(73, cfg, 1)
    got = packed.forward_packed(slots, step, ropes)
    back = rev.forward_packed(slots[::-1], step[::-1], ropes[::-1])[::-1]
    assert np.array_equal(got, back)


@pytest.mark.parametrize("name", ["qwen2_bias_d128", "mixtral_d64", "tiny_d32"])
def test_scrambled_small_pool_equals_the_default_pool(name):
    """Live garbage sequences in slots 4-7 push the test sequences onto scattered, non-home pages of a 20-page FP8 pool."""
    from fastllm_b200 import models
    cfg = CASES[name]
    model, _ = _model(cfg)
    ref = models.DeviceCache(model.dev, 8, 256, kv_dtype=FP8)
    pool = models.DeviceCache(model.dev, 8, 256, pool_tokens=20 * 64, kv_dtype=FP8)
    assert ref.pool_pages() == (32, 32) and pool.pool_pages() == (20, 20)
    for c in (ref, pool):
        c.forward_packed([5, 6, 7], [_ids(900, cfg, 64), _ids(901, cfg, 64), _ids(902, cfg, 100)], [0, 0, 0])
        c.slot_reset(6)
        c.forward_packed([4], [_ids(906, cfg, 65)], [0])
    for kind, slots, parts in _calls(cfg):
        got = []
        for c in (ref, pool):
            ropes = [0] * len(slots)      # positions do not matter for the identity; keep them valid
            got.append(c.forward_packed(slots, parts, ropes) if kind == "packed" else c.forward_slots(slots, np.stack(parts), ropes))
        assert np.array_equal(got[0], got[1]), (name, kind, slots)
        assert np.isfinite(got[1]).all()
    assert [pool.slot_len(s) for s in range(8)] == [ref.slot_len(s) for s in range(8)]


@pytest.mark.parametrize("src_len", [100, 128])
def test_fork_equals_the_unforked_sequence(src_len):
    """A partial last page (copied at fork time, bytes of e4m3) and a full one (shared): the fork continues as its source would."""
    from fastllm_b200 import models
    cfg = CASES["mistral_window_d128"]
    model, _ = _model(cfg)
    a = models.DeviceCache(model.dev, 4, 256, pool_tokens=16 * 64, kv_dtype=FP8)
    twin = models.DeviceCache(model.dev, 4, 256, kv_dtype=FP8)
    prompt = _ids(70, cfg, src_len)
    for c in (a, twin):
        c.forward_slots([0], prompt[None], [0])
    free = a.pool_pages()[0]
    a.slot_fork(0, 1)
    assert a.pool_pages()[0] == free - (1 if src_len % 64 else 0) and a.slot_len(1) == src_len
    for k in range(70):              # across a page boundary
        tok = _ids(300 + k, cfg, 1)[None]
        assert np.array_equal(a.forward_slots([1], tok, [1 + k]), twin.forward_slots([0], tok, [1 + k]))
    cont = _ids(80, cfg, 9)
    assert np.array_equal(a.forward_packed([1, 2], [cont, _ids(81, cfg, 3)], [71, 0])[0],
                          twin.forward_packed([0, 2], [cont, _ids(81, cfg, 3)], [71, 0])[0])


@pytest.mark.parametrize("name", ["mistral_window_d128", "qwen2_bias_d128"])
@pytest.mark.parametrize("plen", [64, 70])
def test_prefix_continuation_matches_the_one_call_prompt(name, plen):
    from fastllm_b200 import models
    cfg = CASES[name]
    model, w = _model(cfg)
    c = models.DeviceCache(model.dev, 4, 256, pool_tokens=8 * 64, kv_dtype=FP8)
    prompt = _ids(95, cfg, plen + 20)
    c.forward_slots([0], prompt[None, :plen], [0])
    c.slot_fork(0, 2)
    got = c.forward_slots([2], prompt[None, plen:], [plen])[0]
    whole = models.DeviceCache(model.dev, 1, 256, kv_dtype=FP8).forward_slots([0], prompt[None], [0])[0]
    want = Fp8KvCausalLM(cfg, w).forward(prompt[None], 0)[0]
    assert float(np.abs(got - want).max()) <= FP8_TOL
    assert float(np.abs(got - whole).max()) <= FP8_TOL


def test_refused_entry_points_and_exhaustion_leave_the_cache_unchanged():
    import ctypes as C
    from fastllm_b200 import models
    cfg = CASES["mistral_window_d128"]
    model, _ = _model(cfg)
    c = models.DeviceCache(model.dev, 4, 256, pool_tokens=4 * 64, kv_dtype=FP8)
    twin = models.DeviceCache(model.dev, 4, 256, pool_tokens=4 * 64, kv_dtype=FP8)
    for x in (c, twin):
        x.forward_packed([0, 1], [_ids(1, cfg, 70), _ids(2, cfg, 10)], [0, 0])
    state = lambda: (c.pool_pages(), [c.slot_len(s) for s in range(4)], c.kv_len())
    before = state()
    ids = np.stack([_ids(3, cfg, 4)])
    lp = models.LogitsProcessor(0, 0.7)
    refused = [lambda: c.forward(ids, 0), lambda: c.forward_greedy(ids, 0), lambda: c.forward_logprobs(ids, ids, 0),
               lambda: c.forward_sample(ids, 0, lp), lambda: c.forward_sample_device(ids, 0, lp),
               lambda: c.decode_greedy_loop(np.array([3], dtype=np.uint32), 0, 4), lambda: c.fill_synthetic(1, 64)]
    for fn in refused:
        assert _code(fn) == FL_ERR_UNSUPPORTED
        assert state() == before
    # exhaustion as on bf16: the call is refused before any device work and changes nothing
    assert _code(lambda: c.forward_packed([2, 3], [_ids(4, cfg, 100), _ids(5, cfg, 10)], [0, 0])) == FL_ERR_STATE
    assert state() == before
    step = [_ids(6, cfg, 1), _ids(7, cfg, 1)]
    assert np.array_equal(c.forward_packed([0, 1], step, [1, 1]), twin.forward_packed([0, 1], step, [1, 1]))
    c.reset()
    assert c.pool_pages() == (4, 4) and [c.slot_len(s) for s in range(4)] == [0] * 4
    lib, h = model.dev.lib, model.dev.h
    out = C.c_void_p()
    assert lib.fl_cache_create_pool_kv(h, 4, 256, 256, 7, C.byref(out)) == FL_ERR_INVALID
    with pytest.raises(ValueError):
        models.DeviceCache(model.dev, 4, 256, kv_dtype="int8")


def test_fp8_pool_of_2n_tokens_fits_in_a_bf16_pool_of_n():
    """Device memory around creation: an FP8 pool of 2N tokens takes no more than a bf16 pool of N (the pool dominates at 1 GiB);
    then PackedBatcher(kv_dtype="fp8_e4m3") on a 2N-token pool completes a trace that holds more than N tokens at once."""
    import torch
    from fastllm_b200 import models
    cfg = CASES["qwen2_bias_d128"]
    model, w = _model(cfg)
    per_token_bf16 = 2 * cfg.num_hidden_layers * cfg.num_key_value_heads * cfg.head_dim * 2
    n = (1 << 30) // per_token_bf16

    def created(tokens, kv_dtype):
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        c = models.DeviceCache(model.dev, 4, 256, pool_tokens=tokens, kv_dtype=kv_dtype)
        used = free0 - torch.cuda.mem_get_info()[0]
        del c
        return used

    bf16, fp8 = created(n, "bf16"), created(2 * n, FP8)
    print(f"bf16 pool of {n} tokens: {bf16 / 2**20:.1f} MiB; fp8 pool of {2 * n} tokens: {fp8 / 2**20:.1f} MiB")
    assert fp8 <= bf16 + (8 << 20)       # allocation granularity

    small = 8 * 64                       # N of the trace: 8 pages
    pb = models.PackedBatcher(model, max_batch=4, eos_token_id=None, pool_tokens=2 * small, kv_dtype=FP8)
    prompts = [list(map(int, _ids(500 + i, cfg, 150))) for i in range(4)]
    outs = pb.generate(prompts, 40)
    assert [len(t) for t in outs] == [40] * 4
    assert pb.peak_pages * 64 > small and pb.cache.pool_pages() == (16, 16)


def test_packed_batcher_greedy_ids_match_the_fp8_oracle():
    """32 greedy steps of PackedBatcher on an FP8 cache against the oracle's fp8-KV greedy ids; a request is compared up to the
    first step whose oracle top-2 gap lies within twice the measured logit error (from there on the paths may part)."""
    from fastllm_b200 import models
    cfg = CASES["mistral_window_d128"]
    model, w = _model(cfg)
    prompts = [list(map(int, _ids(700 + i, cfg, n))) for i, n in enumerate([130, 12, 70])]
    c = models.DeviceCache(model.dev, 1, 256, kv_dtype=FP8)
    err = float(np.abs(c.forward_slots([0], np.asarray([prompts[0]], dtype=np.uint32), [0])[0]
                       - Fp8KvCausalLM(cfg, w).forward(np.asarray([prompts[0]], dtype=np.uint32), 0)[0]).max())
    pb = models.PackedBatcher(model, max_batch=3, eos_token_id=None, kv_dtype=FP8)
    outs = pb.generate(prompts, 32)
    compared = 0
    for p, toks in zip(prompts, outs):
        s = _Seq(cfg, w, 0)
        s.feed(p)
        for tok in toks:
            top = np.sort(s.want)[-2:]
            if top[1] - top[0] <= 2 * max(err, 1e-6):
                break
            assert tok == int(models.sample_argmax(s.want))
            compared += 1
            s.feed([tok])
    assert compared >= 48
