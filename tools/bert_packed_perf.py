"""Dev tool: MiniLM-L6 embeddings/s of sentences of different lengths -- one packed call (fl_embed_packed) against equal-length
grouping (embed_many: one fl_embed per distinct length) and fl_embed padded to the longest sentence with a pooling mask (fast but
NOT the lone-sentence result: the pad tokens are attended to; its max-abs deviation is reported with its speed).

Synthetic weights (seed 0), seeded lengths and ids.  Workloads: (a) 256 x 128 uniform, (b) 256 sentences with lengths uniform in
[8, 128], (c) 256 sentences, 90 % in [8, 64] and 10 % in [129, 512].  Each variant is warmed up, then timed with a host clock around
the synchronous calls (each ends in a stream sync) over windows of >= 1 s, the variants alternating, `--rounds` windows each; the
per-kernel times of the packed call come from a separate fl_prof run.  One JSON line per workload (+ one with the card's name and
power limit) on stdout and in --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fastllm_b200 import models  # noqa: E402

N = 256


def lengths_of(name, rs):
    if name == "a_uniform_256x128":
        return np.full(N, 128)
    if name == "b_uniform_8_128":
        return rs.randint(8, 129, size=N)
    long = rs.rand(N) < 0.1
    return np.where(long, rs.randint(129, 513, size=N), rs.randint(8, 65, size=N))


def rate(f, n, window):
    calls, t0 = 0, time.perf_counter()
    while True:
        f()
        calls += 1
        dt = time.perf_counter() - t0
        if dt >= window:
            return n * calls / dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    lines = [{"card": card.strip().splitlines()[0] if card.strip() else "unknown (nvidia-smi gave nothing)"}]
    print(json.dumps(lines[0]), flush=True)
    cfg = models.BertConfig()
    m = models.MiniLMModel(cfg, None, random_seed=0)
    rs = np.random.RandomState(0)
    for name in ("a_uniform_256x128", "b_uniform_8_128", "c_long_tail"):
        lengths = lengths_of(name, rs)
        sents = [rs.randint(3, cfg.vocab_size, size=int(n)).astype(np.uint32) for n in lengths]
        t = int(lengths.max())
        pad_ids = np.zeros((N, t), dtype=np.uint32)
        pad_mask = np.zeros((N, t), dtype=np.uint32)
        for i, s in enumerate(sents):
            pad_ids[i, :len(s)], pad_mask[i, :len(s)] = s, 1
        variants = {"packed": lambda: m.embed_packed(sents), "grouped": lambda: m.embed_many(sents),
                    "padded_mask": lambda: m.embed_ids(pad_ids, pad_mask)}
        lone = m.embed_many(sents)                      # exact by construction: the lone-sentence results
        for f in variants.values():                     # warm every shape
            for _ in range(3):
                f()
        rates = {k: [] for k in variants}
        for _ in range(a.rounds):
            for k, f in variants.items():
                rates[k].append(rate(f, N, a.window))
        models.prof_begin()
        m.embed_packed(sents)
        prof = models.prof_end()
        line = {"workload": name, "sentences": N, "real_tokens": int(lengths.sum()), "padded_tokens": N * t,
                "distinct_lengths": int(len(set(lengths.tolist()))),
                "emb_per_s": {k: {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))} for k, v in rates.items()},
                "packed_equals_lone_bitwise": bool(np.array_equal(m.embed_packed(sents), lone)),
                "padded_mask_max_abs_vs_lone": float(np.abs(m.embed_ids(pad_ids, pad_mask) - lone).max()),
                "packed_kernels_ms": {p["kernel"]: round(p["ms"], 4) for p in prof},
                "timing": f"host clock around synchronous calls, {a.rounds} alternating windows of >= {a.window} s per variant"}
        lines.append(line)
        print(json.dumps(line), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
