"""PackedBatcher (continuous batching above fl_forward_packed): host logic, tested on CPU against stand-in caches.

Every step is one packed forward that carries the running requests' next tokens and newly admitted prompts.  The property under test
is that each request still gets exactly what Model.generate gives it alone, with prompts admitted next to decode rows under the
step's token budget."""
import zlib

import numpy as np
import pytest

from fastllm_b200 import models

VOCAB = 97


def _row(hist):
    rs = np.random.RandomState(zlib.crc32(np.asarray(hist, dtype=np.uint32).tobytes()))
    row = (rs.standard_normal(VOCAB) * 2).astype(np.float32)
    row[2] += 2.5                       # "</s>" (id 2) is likely enough that requests stop at different steps
    return row


class _Cache:
    def __init__(self):
        self.hist = None


class _HistoryModel:
    """Model.generate's view: logits of a row are a pure function of the sequence's token history."""

    def initialize_cache(self, *a):
        return _Cache()

    def forward(self, ids, pos, cache):
        ids = np.asarray(ids)
        if pos == 0:
            cache.hist = [int(x) for x in ids[0]]
        else:
            cache.hist.append(int(ids[0, 0]))
        return _row(cache.hist)[None]


class _PackedCache:
    """Stand-in for DeviceCache.forward_packed: row i is a pure function of slot slots[i]'s token history."""

    def __init__(self, nslots):
        self.hist = [None] * nslots
        self.calls = []

    def forward_packed(self, slots, seqs, rope_offsets):
        self.calls.append([(int(s), len(q), int(r)) for s, q, r in zip(slots, seqs, rope_offsets)])
        assert len(set(slots)) == len(slots) == len(seqs) == len(rope_offsets)
        rows = []
        for s, q, ro in zip(slots, seqs, rope_offsets):
            assert len(q) >= 1
            if self.hist[s] is None:
                assert ro == 0
                self.hist[s] = []
            else:
                assert len(q) == 1 and ro == len(self.hist[s])          # a decode row; Llama rule: the caller's position
            self.hist[s] += [int(x) for x in q]
            rows.append(_row(self.hist[s]))
        return np.stack(rows)

    def slot_reset(self, slot):
        assert self.hist[slot] is not None
        self.hist[slot] = None


class _Llama:
    arch = "llama"


class _Mistral:
    arch = "mistral"


def _prompts(seed, lengths):
    rs = np.random.RandomState(seed)
    return [list(map(int, rs.randint(3, VOCAB, size=n))) for n in lengths]


@pytest.mark.parametrize("temperature", [0.0, 0.9])
def test_packed_batcher_equals_per_request_generate(temperature):
    prompts = _prompts(5, [5, 9, 2, 7, 3, 11, 4, 6])
    single = [models.Model(_HistoryModel(), None, eos_token_id=2).generate(p, 10, temperature=temperature) for p in prompts]
    assert len({len(s) for s in single}) > 1, "the case must include requests that hit EOS at different steps"
    cache = _PackedCache(3)
    pb = models.PackedBatcher(_Llama(), max_batch=3, eos_token_id=2, cache=cache)
    assert pb.generate(prompts, 10, temperature=temperature) == single
    assert all(h is None for h in cache.hist)                          # every slot was handed back
    assert pb.forwards == len(cache.calls)
    # a prompt is admitted in the same call as decode rows of running requests
    assert any(any(q > 1 for _, q, _ in call) and any(q == 1 and r > 0 for _, q, r in call) for call in cache.calls)
    # fewer forwards than prefilling every prompt alone plus one per decode step
    cb_cache = _PackedCache(3)
    cb_cache.forward_slots = lambda slots, ids, ro: cb_cache.forward_packed(slots, [list(r) for r in np.asarray(ids)], ro)
    cb = models.ContinuousBatcher(_Llama(), max_batch=3, eos_token_id=2, cache=cb_cache)
    assert cb.generate(prompts, 10, temperature=temperature) == single
    assert pb.forwards < len(cb_cache.calls)


def test_packed_batcher_token_budget():
    prompts = _prompts(6, [6, 6, 6, 30, 4])
    cache = _PackedCache(4)
    pb = models.PackedBatcher(_Llama(), max_batch=4, eos_token_id=None, cache=cache, token_budget=14)
    single = [models.Model(_HistoryModel(), None, eos_token_id=None).generate(p, 3) for p in prompts]
    assert pb.generate(prompts, 3) == single
    for call in cache.calls:
        tokens = sum(q for _, q, _ in call)
        prompts_in = [q for _, q, r in call if r == 0]
        # within the budget, unless the call admits a single prompt that alone exceeds it
        assert tokens <= 14 or (len(prompts_in) == 1 and prompts_in[0] > 14 - (len(call) - 1)), call
    # first call: two 6-token prompts fit 14, the third does not; the 30-token prompt is admitted alone once a slot frees up
    assert [q for _, q, _ in cache.calls[0]] == [6, 6]
    big = [call for call in cache.calls if any(q == 30 for _, q, _ in call)]
    assert len(big) == 1 and sum(q for _, q, r in big[0] if r == 0) == 30


def test_packed_batcher_position_rule_of_the_mistral_adapter_and_edge_cases():
    class _C:
        def __init__(self):
            self.calls = []

        def forward_packed(self, slots, seqs, rope_offsets):
            self.calls.append((tuple(slots), tuple(len(q) for q in seqs), tuple(int(r) for r in rope_offsets)))
            return np.tile(np.arange(VOCAB, dtype=np.float32), (len(slots), 1))      # arg-max = VOCAB - 1, never EOS

        def slot_reset(self, slot):
            pass

    cache = _C()
    out = models.PackedBatcher(_Mistral(), max_batch=2, eos_token_id=2, cache=cache).generate([[5, 6, 7], [8], [9, 9]], 3)
    assert out == [[VOCAB - 1] * 3] * 3
    # mistral.rs:234 / qwen.rs:143: the offset grows by ONE per call, whatever the prompt length; the third request waits for a slot
    assert cache.calls == [((0, 1), (3, 1), (0, 0)), ((0, 1), (1, 1), (1, 1)), ((0, 1), (1, 1), (2, 2)),
                           ((1,), (2,), (0,)), ((1,), (1,), (1,)), ((1,), (1,), (2,))]
    llama = _C()
    models.PackedBatcher(_Llama(), max_batch=2, eos_token_id=2, cache=llama).generate([[5, 6, 7]], 3)
    assert [c[2] for c in llama.calls] == [(0,), (3,), (4,)]          # Llama: the caller's position
    assert models.PackedBatcher(_Mistral(), 2, cache=_C()).generate([], 4) == []
    assert models.PackedBatcher(_Mistral(), 2, cache=_C()).generate([[3, 4]], 0) == [[]]
