"""Dev tool: what a KV page pool and prefix forks buy a serving loop on Mistral-7B (synthetic weights, seed 0).

  (a) capacity trace: --requests requests (seeded prompt lengths in [16, 1024], --new-tokens new tokens each: PackedBatcher takes one
      max_tokens per trace) through PackedBatcher at max_batch 32 on the default cache (32 slots x 4096 tokens = 131 072 tokens of
      KV) and at max_batch 128 on a pool of the same 131 072 tokens: total time, generated tok/s, mean / p90 time to first token
      (from the start of the trace), and the most pages in use after any call;
  (b) shared-prefix trace: 64 requests sharing a 1024-token prefix, seeded suffixes of 16-256 tokens, --prefix-new-tokens new tokens
      each, max_batch 32 on the default cache, with and without shared_prefix: total time, time to first token, prompt tokens fed;
  (c) fork: the device time of fl_cache_slot_fork's partial-page copy (kv_page_copy, from fl_prof) at a 1000-token source, and the
      host time of the whole call (fork + device synchronise), over --forks forks.

(a) and (b): one short warm-up trace per form, then --rounds alternating traces; host clock around whole traces (every packed call
ends in a synchronising read-back).  One JSON line per measurement, after one with the card's name and power limit, on stdout and in
--out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fastllm_b200 import _lib, models, presets  # noqa: E402


class _Timed:
    """A DeviceCache as PackedBatcher sees it, recording when each admitted prompt's first token is ready (the end of the packed call
    that fed it) and the most pages in use after any call.  The first call of a shared-prefix trace feeds the prefix alone."""

    def __init__(self, cache, prefix_call=False):
        self.c, self.max_seq = cache, cache.max_seq
        self.skip = prefix_call
        self.first, self.peak = [], 0

    def forward_packed(self, slots, seqs, ropes):
        out = self.c.forward_packed(slots, seqs, ropes)
        now = time.perf_counter()
        if self.skip:
            self.skip = False
        else:
            self.first += [now] * sum(len(q) > 1 for q in seqs)      # prompts and suffixes are >= 16 tokens, decode rows 1
        free, total = self.c.pool_pages()
        self.peak = max(self.peak, total - free)
        return out

    def slot_reset(self, slot):
        self.c.slot_reset(slot)

    def slot_fork(self, src, dst):
        self.c.slot_fork(src, dst)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--requests", type=int, default=256)
    ap.add_argument("--new-tokens", type=int, default=96)
    ap.add_argument("--prefix-new-tokens", type=int, default=32)
    ap.add_argument("--forks", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kv_pool_perf.jsonl"))
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    lines = [{"card": card.strip().splitlines()[0] if card.strip() else "unknown (nvidia-smi gave nothing)"}]
    print(json.dumps(lines[0]), flush=True)

    def emit(line):
        lines.append(line)
        print(json.dumps(line), flush=True)

    cls, cf = presets.PRESETS["mistral7b"]
    model, _ = cls.initialize_model(cf, None, "bf16", 0, random_seed=0)
    V = cf.vocab_size
    rs = np.random.RandomState(0)

    def ids(n):
        return [int(x) for x in rs.randint(3, V, size=n)]

    def run(cache, max_batch, prompts, new_tokens, pool_tokens=None, prefix=None):
        t = _Timed(cache, prefix_call=prefix is not None and max_batch > 1)
        pb = models.PackedBatcher(model, max_batch=max_batch, eos_token_id=None, cache=t, pool_tokens=pool_tokens)
        t0 = time.perf_counter()
        outs = pb.generate(prompts, new_tokens, shared_prefix=prefix)
        total = time.perf_counter() - t0
        ttft = np.array(t.first) - t0
        for s in range(max_batch):
            assert cache.slot_len(s) == 0
        return {"total_s": round(total, 3), "generated_tok_s": round(sum(map(len, outs)) / total, 1),
                "ttft_mean_s": round(float(ttft.mean()), 3), "ttft_p90_s": round(float(np.percentile(ttft, 90)), 3),
                "peak_pages": t.peak, "prefill_tokens": pb.prefill_tokens, "forwards": pb.forwards}

    def alternate(name, forms, warm):
        for f in forms.values():
            f(warm)
        res = {k: [] for k in forms}
        for _ in range(a.rounds):
            for k, f in forms.items():
                res[k].append(f(None))
        for k, v in res.items():
            emit({"measurement": name, "form": k, "runs": v})

    # (a) capacity
    prompts = [ids(int(n)) for n in rs.randint(16, 1025, size=a.requests)]
    default = models.DeviceCache(model.dev, 32, 4096)
    pool = models.DeviceCache(model.dev, 128, 4096, pool_tokens=32 * 4096)
    alternate("capacity_trace", {
        "max_batch 32, default cache (131072 tokens)": lambda w: run(default, 32, w or prompts, a.new_tokens),
        "max_batch 128, pool of 131072 tokens": lambda w: run(pool, 128, w or prompts, a.new_tokens, pool_tokens=32 * 4096),
    }, prompts[:8])
    del default, pool

    # (b) shared prefix
    prefix = ids(1024)
    sp = [prefix + ids(int(n)) for n in rs.randint(16, 257, size=64)]
    cache = models.DeviceCache(model.dev, 32, 4096)
    alternate("shared_prefix_trace", {
        "without shared_prefix": lambda w: run(cache, 32, w or sp, a.prefix_new_tokens),
        "with shared_prefix": lambda w: run(cache, 32, w or sp, a.prefix_new_tokens, prefix=prefix),
    }, sp[:4])

    # (c) fork at 1000 tokens: kv_page_copy copies the partial last page, K and V of 32 layers (2 x 32 x 8 x 64 x 128 x 2 B = 8 MiB,
    # read and written)
    cache.reset()
    cache.forward_packed([0], [ids(1000)], [0])
    cache.slot_fork(0, 1)
    cache.slot_reset(1)
    lib = _lib.load()
    t0 = time.perf_counter()
    for _ in range(a.forks):
        cache.slot_fork(0, 1)
        _lib.check(lib.fl_device_synchronize())
        cache.slot_reset(1)
    host_ms = (time.perf_counter() - t0) * 1e3 / a.forks
    models.prof_begin()
    for _ in range(a.forks):
        cache.slot_fork(0, 1)
        cache.slot_reset(1)
    prof = {p["kernel"]: p for p in models.prof_end()}["kv_page_copy"]
    dev_ms = prof["ms"] / prof["launches"]
    emit({"measurement": "fork_1000_tokens", "kv_page_copy_device_ms": round(dev_ms, 4), "bytes_moved": prof["bytes"] // prof["launches"],
          "achieved_GB_s": round(prof["bytes"] / prof["launches"] / dev_ms / 1e6, 1),
          "fork_call_host_ms_incl_sync_and_slot_reset": round(host_ms, 4)})

    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
