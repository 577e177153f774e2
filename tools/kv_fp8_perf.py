"""Dev tool: what an FP8 (e4m3) KV cache buys against a bf16 one on Mistral-7B (synthetic weights, seed 0).

  (a) decode: batch 8 and 64 at 2k context, both caches prefilled through packed calls (the synthetic KV fill is uniform-only): the
      fl_forward_slots step time (host clock around --steps steps, each ending in the logits read-back) and, in a separate profiled
      window, the attn_sk_decode kernel time from fl_prof and the K/V bytes it reads (from the shapes);
  (b) capacity trace at equal pool bytes: --requests requests (seeded prompt lengths in [16, 1024], --new-tokens new tokens each)
      through PackedBatcher, bf16 on a 131 072-token pool at max_batch 128 and FP8 on a 262 144-token pool at max_batch 256: total time,
      generated tok/s, mean time to first token, most pages in use;
  (c) one 4096-token prompt admitted into an empty slot: host time of the call, and the q|k|v epilogue and tcgen05 prefill attention
      times from fl_prof (the FP8 cache's epilogue also writes the call's bf16 K scratch).

bf16 and FP8 alternate in one session (--rounds each).  One JSON line per measurement, after one with the card's name and power limit,
on stdout and in --out."""
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

DTYPES = ("bf16", "fp8_e4m3")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--context", type=int, default=2048)
    ap.add_argument("--requests", type=int, default=256)
    ap.add_argument("--new-tokens", type=int, default=96)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kv_fp8_perf.jsonl"))
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
        return rs.randint(3, V, size=n).astype(np.uint32)

    def prof(fn, names):
        models.prof_begin()
        fn()
        p = {r["kernel"]: r for r in models.prof_end()}
        return {k: {"ms_per_launch": round(p[k]["ms"] / p[k]["launches"], 4), "bytes_per_launch": p[k]["bytes"] // p[k]["launches"]}
                for k in names if k in p}

    # (a) decode at batch 8 and 64, 2k context
    for B in (8, 64):
        max_seq = a.context + 64 + a.rounds * (a.steps + 2) + 8
        caches = {dt: models.DeviceCache(model.dev, B, max_seq, kv_dtype=dt) for dt in DTYPES}
        for dt, c in caches.items():
            for s0 in range(0, B, 8):           # 8 prompts of `context` tokens per packed call
                sl = list(range(s0, min(B, s0 + 8)))
                c.forward_packed(sl, [ids(a.context) for _ in sl], [0] * len(sl))
        pos = {dt: 1 for dt in DTYPES}           # the Mistral adapter's RoPE rule: +1 per call

        def steps(dt, k):
            c = caches[dt]
            for _ in range(k):
                c.forward_slots(list(range(B)), ids(B)[:, None], [pos[dt]] * B)
                pos[dt] += 1

        for dt in DTYPES:
            steps(dt, 2)                         # warm-up: captures the step's CUDA graph
        res = {dt: [] for dt in DTYPES}
        for _ in range(a.rounds):
            for dt in DTYPES:
                t0 = time.perf_counter()
                steps(dt, a.steps)
                res[dt].append(round((time.perf_counter() - t0) * 1e3 / a.steps, 3))
        for dt in DTYPES:
            k = prof(lambda: steps(dt, 2), ["attn_sk_decode"])["attn_sk_decode"]
            # K/V bytes one launch (one layer) reads, from the shapes (fl_prof's byte count of slot calls does not see their lengths)
            kv = B * (a.context + pos[dt] - 1) * cf.num_key_value_heads * (cf.hidden_size // cf.num_attention_heads) * 2 * (2 if dt == "bf16" else 1)
            k.pop("bytes_per_launch")
            k["kv_bytes_per_launch"] = kv
            k["achieved_TB_s"] = round(kv / k["ms_per_launch"] / 1e9, 2)
            emit({"measurement": "decode_step", "batch": B, "context": a.context, "kv_dtype": dt, "step_ms_runs": res[dt],
                  "attn_sk_decode": k})
        del caches

    # (b) capacity trace at equal pool bytes
    prompts = [list(map(int, ids(int(n)))) for n in rs.randint(16, 1025, size=a.requests)]
    forms = {"bf16": (128, 131072), "fp8_e4m3": (256, 262144)}
    pools = {dt: models.DeviceCache(model.dev, mb, 4096, pool_tokens=tok, kv_dtype=dt) for dt, (mb, tok) in forms.items()}

    def trace(dt, ps):
        mb, tok = forms[dt]
        cache = pools[dt]
        first, peak = [], [0]

        class Timed:
            max_seq = cache.max_seq

            def forward_packed(self, slots, seqs, ropes):
                out = cache.forward_packed(slots, seqs, ropes)
                first.extend([time.perf_counter()] * sum(len(q) > 1 for q in seqs))
                free, total = cache.pool_pages()
                peak[0] = max(peak[0], total - free)
                return out

            def slot_reset(self, slot):
                cache.slot_reset(slot)

        pb = models.PackedBatcher(model, max_batch=mb, eos_token_id=None, cache=Timed(), pool_tokens=tok)
        t0 = time.perf_counter()
        outs = pb.generate(ps, a.new_tokens)
        total = time.perf_counter() - t0
        return {"total_s": round(total, 3), "generated_tok_s": round(sum(map(len, outs)) / total, 1),
                "ttft_mean_s": round(float(np.mean(np.array(first) - t0)), 3), "peak_pages": peak[0]}

    for dt in DTYPES:
        trace(dt, prompts[:8])
    res = {dt: [] for dt in DTYPES}
    for _ in range(a.rounds - 1):
        for dt in DTYPES:
            res[dt].append(trace(dt, prompts))
    for dt in DTYPES:
        emit({"measurement": "capacity_trace", "kv_dtype": dt, "max_batch": forms[dt][0], "pool_tokens": forms[dt][1],
              "pool_bytes": forms[dt][1] * 2 * cf.num_hidden_layers * cf.num_key_value_heads * (cf.hidden_size // cf.num_attention_heads)
              * (2 if dt == "bf16" else 1), "runs": res[dt]})
    del pools

    # (c) a 4096-token prompt admitted as one call
    caches = {dt: models.DeviceCache(model.dev, 2, 4096 + 64, kv_dtype=dt) for dt in DTYPES}
    prompt = ids(4096)

    def admit(dt):
        c = caches[dt]
        c.slot_reset(0)
        c.forward_packed([0], [prompt], [0])

    for dt in DTYPES:
        admit(dt)
    res = {dt: [] for dt in DTYPES}
    for _ in range(a.rounds):
        for dt in DTYPES:
            t0 = time.perf_counter()
            admit(dt)
            res[dt].append(round((time.perf_counter() - t0) * 1e3, 2))
    for dt in DTYPES:
        emit({"measurement": "admit_4096_tokens", "kv_dtype": dt, "call_ms_runs": res[dt],
              "kernels_per_layer": prof(lambda: admit(dt), ["dense_qkv_rope_append", "attn_prefill_tc"])})

    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
