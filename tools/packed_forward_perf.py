"""Dev tool: what packing prompts into one forward buys on Mistral-7B (synthetic weights, seed 0) -- fl_forward_packed against the
fl_forward_slots calls a scheduler makes without it.

  (a) admission: k prompts (seeded lengths in [16, 512]) as k lone fl_forward_slots calls, or as ONE fl_forward_packed call;
  (b) mixed step: 32 running decode rows plus one 512-token prompt as a slots decode step + a lone prefill, or ONE packed call;
  (c) serving trace: 64 requests (seeded prompt lengths in [16, 1024], 64 new tokens each, max_batch 32) through ContinuousBatcher
      and PackedBatcher: total time, generated tok/s, mean / p90 time to first token (from the start of the trace).

(a) and (b): every call on a freshly reset cache, host clock around the synchronous calls (uploads and read-backs included); one
warm-up of each form, then --rounds alternating runs; median / min / max.  (c) one warm-up trace per batcher, then --rounds
alternating traces.  Then one fl_prof run of the packed admission call at k = 1 with a 4096-token prompt and one decode row,
against the lone 4096-token prefill, for what the one-row q|k|v epilogue costs.  One JSON line per measurement, after one with the
card's name and power limit, on stdout and in --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fastllm_b200 import models, presets  # noqa: E402


def stats(v):
    return {"median": round(float(np.median(v)), 3), "min": round(float(min(v)), 3), "max": round(float(max(v)), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ks", default="4,16,64")
    ap.add_argument("--requests", type=int, default=64)
    ap.add_argument("--new-tokens", type=int, default=64)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "packed_forward_perf.jsonl"))
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

    def alternate(forms, rounds):
        for f in forms.values():            # warm-up: workspaces, kernel modules
            f()
        ms = {k: [] for k in forms}
        for _ in range(rounds):
            for k, f in forms.items():
                t0 = time.perf_counter()
                f()
                ms[k].append((time.perf_counter() - t0) * 1e3)
        return ms

    # (a) admission
    cache = models.DeviceCache(model.dev, 64, 4200)
    for k in (int(x) for x in a.ks.split(",")):
        rs = np.random.RandomState(k)
        prompts = [rs.randint(3, V, size=int(n)).astype(np.uint32) for n in rs.randint(16, 513, size=k)]

        def lone():
            cache.reset()
            for i, p in enumerate(prompts):
                cache.forward_slots([i], p[None], [0])

        def packed():
            cache.reset()
            cache.forward_packed(list(range(k)), prompts, [0] * k)

        ms = alternate({"lone": lone, "packed": packed}, a.rounds)
        emit({"case": "admission", "model": "mistral7b", "prompts": k, "tokens": int(sum(len(p) for p in prompts)),
              "lone_slots_calls_ms": stats(ms["lone"]), "packed_call_ms": stats(ms["packed"]),
              "speedup": round(float(np.median(ms["lone"]) / np.median(ms["packed"])), 2)})

    # (b) mixed step: 32 running requests (contexts of 256 tokens) + one 512-token prompt
    rs = np.random.RandomState(32)
    ctx = [rs.randint(3, V, size=256).astype(np.uint32) for _ in range(32)]
    prompt = rs.randint(3, V, size=512).astype(np.uint32)
    dec = [np.array([int(t)], dtype=np.uint32) for t in rs.randint(3, V, size=32)]

    def fill():
        cache.reset()
        cache.forward_slots(list(range(32)), np.stack(ctx), [0] * 32)

    def split():
        fill()
        t0 = time.perf_counter()
        cache.forward_slots(list(range(32)), np.stack(dec), [256] * 32)
        cache.forward_slots([32], prompt[None], [0])
        return time.perf_counter() - t0

    def one():
        fill()
        t0 = time.perf_counter()
        cache.forward_packed(list(range(33)), dec + [prompt], [256] * 32 + [0])
        return time.perf_counter() - t0

    split(), one()
    ms = {"split": [], "packed": []}
    for _ in range(a.rounds):
        ms["split"].append(split() * 1e3)
        ms["packed"].append(one() * 1e3)
    emit({"case": "mixed_step", "model": "mistral7b", "decode_rows": 32, "context": 256, "prompt": 512,
          "decode_step_plus_lone_prefill_ms": stats(ms["split"]), "packed_call_ms": stats(ms["packed"]),
          "speedup": round(float(np.median(ms["split"]) / np.median(ms["packed"])), 2)})
    del cache

    # (c) serving trace
    rs = np.random.RandomState(64)
    prompts = [list(map(int, rs.randint(3, V, size=int(n)))) for n in rs.randint(16, 1025, size=a.requests)]
    serve_cache = models.DeviceCache(model.dev, 32, 1024 + a.new_tokens + 1)
    res = {"continuous": [], "packed": []}
    ttfts = {"continuous": [], "packed": []}
    for kind in res:                                    # warm-up
        _trace(model, serve_cache, prompts, a.new_tokens, kind)
    for _ in range(a.rounds):
        for kind in res:
            outs, total, ttft = _trace(model, serve_cache, prompts, a.new_tokens, kind)
            res[kind].append(total)
            ttfts[kind].append(ttft)
    gen = a.requests * a.new_tokens
    line = {"case": "serving_trace", "model": "mistral7b", "requests": a.requests, "new_tokens": a.new_tokens, "max_batch": 32,
            "prompt_tokens": int(sum(len(p) for p in prompts))}
    for kind in res:
        tt = np.array(ttfts[kind])                        # [rounds, requests] seconds
        line[kind] = {"total_s": stats(res[kind]), "tok_per_s": round(gen / float(np.median(res[kind])), 1),
                      "ttft_mean_s": round(float(np.median(tt.mean(1))), 3), "ttft_p90_s": round(float(np.median(np.percentile(tt, 90, axis=1))), 3)}
    line["speedup_total"] = round(float(np.median(res["continuous"]) / np.median(res["packed"])), 2)
    emit(line)
    del serve_cache

    # what the one-row q|k|v epilogue costs a 4096-token prompt: packed (4096 + one decode row) vs the lone prefill, per kernel
    cache = models.DeviceCache(model.dev, 2, 4200)
    p4k = np.random.RandomState(4096).randint(3, V, size=4096).astype(np.uint32)
    prof = {}
    for kind in ("lone", "packed"):
        for _ in range(2):                              # the second run is profiled
            cache.reset()
            cache.forward_slots([1], np.array([[5, 6, 7]], dtype=np.uint32), [0])
            if _:
                models.prof_begin()
            if kind == "lone":
                cache.forward_slots([0], p4k[None], [0])
            else:
                cache.forward_packed([0, 1], [p4k, np.array([9], dtype=np.uint32)], [0, 3])
            if _:
                prof[kind] = {p["kernel"]: round(p["ms"], 3) for p in models.prof_end()}
    emit({"case": "qkv_epilogue_4k", "model": "mistral7b", "prompt": 4096,
          "lone_qkv_epilogue_ms": prof["lone"].get("dense_qkv_rope_append"), "packed_qkv_epilogue_ms": prof["packed"].get("dense_qkv_rope_append"),
          "kernels_ms_lone": prof["lone"], "kernels_ms_packed": prof["packed"],
          "timing": "fl_prof: every kernel bracketed by events, launched without programmatic dependent launch; 32 layers"})
    if a.out:
        with open(a.out, "w") as fo:
            for ln in lines:
                fo.write(json.dumps(ln) + "\n")


def _trace(model, cache, prompts, new_tokens, kind):
    """One serving trace.  -> (outputs, total seconds, per-request seconds from the start to the forward that returned the logits of
    its first token)"""
    cache.reset()
    b = (models.ContinuousBatcher if kind == "continuous" else models.PackedBatcher)(model, max_batch=32, eos_token_id=None, cache=cache)
    first = [None] * len(prompts)
    # a request's first token is sampled from the forward that took its prompt: the batchers create its LogitsProcessor just before
    # that forward, in request order, so the k-th processor created belongs to request k
    created = []
    real = models.LogitsProcessor

    class _Marked(real):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.req, self.first = len(created), True
            created.append(self)

        def sample(self, logits):
            if self.first:
                first[self.req] = time.perf_counter()
                self.first = False
            return super().sample(logits)

    models.LogitsProcessor = _Marked
    try:
        t0 = time.perf_counter()
        outs = b.generate(prompts, new_tokens)
        total = time.perf_counter() - t0
    finally:
        models.LogitsProcessor = real
    return outs, total, [f - t0 for f in first]


if __name__ == "__main__":
    main()
