"""PackedBatcher on a KV page pool and with a shared prefix: host logic, tested on CPU against a stand-in cache that keeps each slot's
token history and counts pages as the library's allocator does (full prefix pages shared by the forks)."""
import numpy as np
import pytest

from fastllm_b200 import models

from test_packed_batcher_cpu import VOCAB, _HistoryModel, _prompts, _row

PAGE = 64


class _PoolCache:
    """forward_packed / slot_reset / slot_fork over token histories; every call is checked against the pool's page count."""

    def __init__(self, nslots, pool_pages, max_seq=4096):
        self.hist = [None] * nslots
        self.shared = [0] * nslots          # full pages a forked slot shares with the prefix slot
        self.pool_pages, self.max_seq = pool_pages, max_seq
        self.calls, self.peak = [], 0

    def pages(self):
        return sum(-(-len(h) // PAGE) - sh for h, sh in zip(self.hist, self.shared) if h is not None)

    def forward_packed(self, slots, seqs, rope_offsets):
        self.calls.append([(int(s), len(q), int(r)) for s, q, r in zip(slots, seqs, rope_offsets)])
        rows = []
        for s, q, ro in zip(slots, seqs, rope_offsets):
            if self.hist[s] is None:
                self.hist[s] = []
            self.hist[s] += [int(x) for x in q]
            rows.append(_row(self.hist[s]))
        self.peak = max(self.peak, self.pages())
        assert self.pages() <= self.pool_pages
        return np.stack(rows)

    def slot_fork(self, src, dst):
        assert self.hist[dst] is None and self.hist[src]
        self.hist[dst] = list(self.hist[src])
        self.shared[dst] = len(self.hist[src]) // PAGE

    def slot_reset(self, slot):
        self.hist[slot], self.shared[slot] = None, 0


class _Mistral:
    arch = "mistral"

    class cfg:
        sliding_window = 4096


class _MistralWindow(_Mistral):
    class cfg:
        sliding_window = 100


class _Llama:
    arch = "llama"


def _single(prompts, n):
    return [models.Model(_HistoryModel(), None, eos_token_id=2).generate(p, n) for p in prompts]


def test_admission_by_pages_never_exceeds_the_pool():
    prompts = _prompts(7, [100, 30, 200, 5, 64, 150, 20, 90])
    cache = _PoolCache(6, pool_pages=6)
    pb = models.PackedBatcher(_Llama(), max_batch=6, eos_token_id=2, cache=cache, pool_tokens=6 * PAGE)
    assert pb.generate(prompts, 10) == _single(prompts, 10)
    assert cache.peak <= 6 and pb.peak_pages <= 6
    # free slots were left unused for lack of pages: some call ran fewer sequences than slots while requests waited
    assert max(len(c) for c in cache.calls) < 6
    with pytest.raises(ValueError):
        models.PackedBatcher(_Llama(), max_batch=2, cache=_PoolCache(2, 1), pool_tokens=PAGE).generate([[3] * 70], 4)


def test_shared_prefix_feeds_the_prefix_once_at_the_one_call_positions():
    rs = np.random.RandomState(3)
    prefix = list(map(int, rs.randint(3, VOCAB, size=70)))
    prompts = [prefix + p for p in _prompts(8, [9, 3, 40])] + _prompts(9, [12]) + [prefix[:30], list(prefix)]
    cache = _PoolCache(4, pool_pages=20)
    pb = models.PackedBatcher(_Mistral(), max_batch=4, eos_token_id=2, cache=cache, pool_tokens=20 * PAGE)
    got = pb.generate(prompts, 8, shared_prefix=prefix)
    assert got == _single(prompts, 8)                  # the stand-in's rows depend on token histories only
    assert cache.calls[0] == [(0, 70, 0)]              # the prefix, alone, into the held slot
    suffix_calls = [(s, n, r) for call in cache.calls[1:] for s, n, r in call if r == 70]
    assert sorted(n for _, n, _ in suffix_calls) == [3, 9, 40]      # only the rest of each prompt, at RoPE offset len(prefix)
    assert pb.prefill_tokens == 70 + 9 + 3 + 40 + 12 + 30 + 70
    assert all(h is None for h in cache.hist)          # the prefix slot is released at the end


def test_prefix_is_not_used_on_llama_or_past_the_window():
    prefix = [5] * 70
    prompts = [prefix + [6] * 9, prefix + [7] * 40]
    for model, used in ((_Llama(), []), (_MistralWindow(), [9])):    # 79 tokens fit the 100-token window, 110 do not
        cache = _PoolCache(3, pool_pages=20)
        assert models.PackedBatcher(model, max_batch=3, eos_token_id=2, cache=cache, pool_tokens=20 * PAGE).generate(
            prompts, 4, shared_prefix=prefix) == _single(prompts, 4)
        assert sorted(n for call in cache.calls for _, n, r in call if r == 70) == used
        assert (cache.calls[0] == [(0, 70, 0)]) == bool(used)


def test_empty_prefix_or_a_single_slot_takes_the_normal_path():
    prompts = _prompts(10, [5, 9])
    for max_batch, prefix in ((3, []), (1, prompts[0][:2])):
        cache = _PoolCache(max_batch, pool_pages=20)
        pb = models.PackedBatcher(_Mistral(), max_batch=max_batch, eos_token_id=2, cache=cache, pool_tokens=20 * PAGE)
        assert pb.generate(prompts, 4, shared_prefix=prefix) == _single(prompts, 4)
        assert all(r == 0 or n == 1 for call in cache.calls for _, n, r in call)     # no prefix call, no suffix at an offset
