"""Dev tool: what scoring costs on top of a prefill -- fl_forward against fl_forward_logprobs on Qwen2.5-7B (synthetic weights, seed 0,
vocabulary 152 064) at b = 1, t = 4096 and b = 8, t = 512.

Per shape: one warm-up call of each, then --rounds alternating runs of --calls calls each, every call on a freshly reset cache and
timed with a host clock around the synchronous call (the id / target upload and the read-back included); median / min / max of the
per-call mean.  Then one fl_prof run of each for the per-kernel split (every kernel bracketed by events and launched without
programmatic dependent launch, so the kernels sum to more than the pipelined call).  Reported: the extra milliseconds of a scoring
call, the scoring lm_head GEMM's achieved TFLOP/s (2 R V H useful, twice that issued for the hi / lo activation pair), the combine
kernel's time, and the bytes of the soft-max partials against the R V 4 bytes of materialised f32 logits.  One JSON line per shape,
after one with the card's name and power limit (a query only), on stdout and in --out."""
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

PART_BYTES = 12          # LogprobPart: max, sum, index
PARTS_PER_TILE = 4       # one per column slice of a 256-wide vocab tile (gemm_tc.cuh)


def stats(v):
    return {"median": round(float(np.median(v)), 3), "min": round(float(min(v)), 3), "max": round(float(max(v)), 3)}


def per_kernel(prof):
    return {p["kernel"]: round(p["ms"], 4) for p in prof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--shapes", default="1x4096,8x512")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "logprobs_perf.jsonl"))
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    lines = [{"card": card.strip().splitlines()[0] if card.strip() else "unknown (nvidia-smi gave nothing)"}]
    print(json.dumps(lines[0]), flush=True)
    cls, cf = presets.PRESETS["qwen25_7b"]
    model, _ = cls.initialize_model(cf, None, "bf16", 0, random_seed=0)
    H, V = cf.hidden_size, cf.vocab_size
    for shape in a.shapes.split(","):
        b, t = (int(x) for x in shape.split("x"))
        R = b * t
        rs = np.random.RandomState(R)
        ids = rs.randint(0, V, size=(b, t)).astype(np.uint32)
        targets = np.concatenate([ids[:, 1:], rs.randint(0, V, size=(b, 1)).astype(np.uint32)], axis=1)
        cache = models.DeviceCache(model.dev, b, t)
        calls = {"forward": lambda: cache.forward(ids, 0), "logprobs": lambda: cache.forward_logprobs(ids, targets, 0)}

        def timed(name):
            total = 0.0
            for _ in range(a.calls):
                cache.reset()
                t0 = time.perf_counter()
                calls[name]()
                total += time.perf_counter() - t0
            return total / a.calls * 1e3

        for name in calls:          # warm-up: workspaces, kernel modules
            cache.reset()
            calls[name]()
        ms = {name: [] for name in calls}
        for _ in range(a.rounds):
            for name in calls:
                ms[name].append(timed(name))
        prof = {}
        for name in calls:
            cache.reset()
            models.prof_begin()
            calls[name]()
            prof[name] = per_kernel(models.prof_end())
        gemm = prof["logprobs"]["gemm_tc_lm_head_logprob"]
        useful = 2.0 * R * V * H
        ntn = (V + 255) // 256
        line = {"model": "qwen25_7b", "b": b, "t": t, "rows": R, "vocab": V,
                "forward_ms": stats(ms["forward"]), "logprobs_ms": stats(ms["logprobs"]),
                "extra_ms": round(float(np.median(ms["logprobs"]) - np.median(ms["forward"])), 3),
                "lm_head_logprob_ms": gemm, "lm_head_logprob_tflops": round(useful / (gemm / 1e3) / 1e12, 1),
                "lm_head_logprob_tflops_issued": round(2 * useful / (gemm / 1e3) / 1e12, 1),
                "combine_ms": prof["logprobs"].get("logprob_combine"),
                "forward_lm_head_ms": prof["forward"].get("gemm_tc_lm_head"),
                "partials_mb": round(R * ntn * PARTS_PER_TILE * PART_BYTES / 1e6, 1), "logits_mb": round(R * V * 4 / 1e6, 1),
                "kernels_ms_forward": prof["forward"], "kernels_ms_logprobs": prof["logprobs"],
                "timing": f"host clock around synchronous calls on a reset cache, {a.rounds} alternating runs of {a.calls} calls; kernel "
                          "times from a separate fl_prof run"}
        lines.append(line)
        print(json.dumps(line), flush=True)
        del cache
    if a.out:
        with open(a.out, "w") as fo:
            for ln in lines:
                fo.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
