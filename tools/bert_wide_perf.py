"""Dev tool: embeddings/s and achieved TFLOP/s of the BERT encoder at three widths -- all-MiniLM-L6-v2 (hidden 384, head_dim 32),
BERT-base (768, head_dim 64) and BERT-large (1024, head_dim 64) -- with the per-kernel split from fl_prof.

Synthetic weights (seed 0), seeded ids.  Two batches per model: (a) 256 x 128 uniform, timed device-resident (fl_embed_timed:
repeats of the encoder over the uploaded batch between two CUDA events, >= 0.5 s per window); (b) 256 packed sentences with lengths
uniform in [8, 512], one fl_embed_packed call, timed with a host clock around the synchronous calls (so it includes the id upload and
the read-back; >= 1 s per window).  `--rounds` windows each; median / min / max.  FLOP from shapes: per sentence of t tokens,
t * 2 L (4 H^2 + 2 H I) for the linear layers + 4 L t^2 H for Q K^T and P V.  The per-kernel times come from a separate fl_prof run
(each kernel bracketed by events, without programmatic dependent launch, so they sum to more than the pipelined time).  Every GEMM
uses one 128 x 192 output tile: a width N that 192 does not divide computes ceil(N / 192) * 192 columns, and `partial_tile_ms_est`
is the kernel's time times the dead fraction of those columns.  One JSON line per (model, batch), after one with the card's name and
power limit, on stdout and in --out."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fastllm_b200 import models, presets  # noqa: E402

N = 256
BN = 192                        # kBertBN, fl_bert.cu
GROUPS = {"gemm": ("bert_gemm_qkv", "bert_gemm_o", "bert_gemm_up_gelu", "bert_gemm_down"), "attention": ("bert_attn",),
          "layernorm": ("bert_embed_ln", "bert_layernorm"), "pool": ("bert_pool_l2",)}


def flop(cfg, lengths):
    H, I, L = cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
    t = np.asarray(lengths, dtype=np.float64)
    return float((t * 2 * L * (4 * H * H + 2 * H * I) + 4 * L * t * t * H).sum())


def gemm_shapes(cfg):
    H, I = cfg.hidden_size, cfg.intermediate_size
    return {"bert_gemm_qkv": (3 * H, H), "bert_gemm_o": (H, H), "bert_gemm_up_gelu": (I, H), "bert_gemm_down": (H, I)}


def split(cfg, prof, tokens):
    ms = {p["kernel"]: p["ms"] for p in prof}
    out = {"kernels_ms": {k: round(v, 4) for k, v in ms.items()},
           "groups_ms": {g: round(sum(ms.get(k, 0.0) for k in ks), 4) for g, ks in GROUPS.items()}}
    L = cfg.num_hidden_layers
    gemms = {}
    for k, (n, kk) in gemm_shapes(cfg).items():
        cols = math.ceil(n / BN) * BN
        gemms[k] = {"N": n, "K": kk, "n_tiles": cols // BN, "live_fraction": round(n / cols, 4),
                    "tflops": round(2.0 * tokens * n * kk * L / (ms[k] / 1e3) / 1e12, 1),
                    "partial_tile_ms_est": round(ms[k] * (1 - n / cols), 4)}
    out["gemms"] = gemms
    out["partial_tile_ms_est_total"] = round(sum(g["partial_tile_ms_est"] for g in gemms.values()), 4)
    return out


def stats(v):
    return {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))}


def host_rate(f, window):
    calls, t0 = 0, time.perf_counter()
    while True:
        f()
        calls += 1
        dt = time.perf_counter() - t0
        if dt >= window:
            return dt / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--models", default="minilm_l6,bert_base,bert_large")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bert_wide_perf.jsonl"))
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    lines = [{"card": card.strip().splitlines()[0] if card.strip() else "unknown (nvidia-smi gave nothing)"}]
    print(json.dumps(lines[0]), flush=True)
    for name in a.models.split(","):
        cfg = presets.BERT_PRESETS[name]
        m = models.MiniLMModel(cfg, None, random_seed=0)
        rs = np.random.RandomState(0)
        # (a) 256 x 128, device-resident
        ids = rs.randint(3, cfg.vocab_size, size=(N, 128)).astype(np.uint32)
        m.embed_ids(ids)
        _, ms = m.embed_ids_timed(ids, 3)
        reps = max(5, math.ceil(500.0 / (ms / 3)))
        per = []
        for _ in range(a.rounds):
            _, ms = m.embed_ids_timed(ids, reps)
            per.append(ms / reps)
        f = flop(cfg, [128] * N)
        models.prof_begin()
        m.embed_ids(ids)
        prof = models.prof_end()
        line = {"model": name, "config": cfg.__dict__, "batch": "a_uniform_256x128", "sentences": N, "tokens": N * 128,
                "tflop_per_batch": round(f / 1e12, 3), "device_ms_per_batch": stats(per),
                "emb_per_s": round(N / (np.median(per) / 1e3)), "tflops": round(f / (np.median(per) / 1e3) / 1e12, 1),
                **split(cfg, prof, N * 128),
                "timing": f"fl_embed_timed, {a.rounds} windows of {reps} device-resident batches; kernel split from a separate fl_prof run"}
        lines.append(line)
        print(json.dumps(line), flush=True)
        # (b) 256 packed sentences, lengths 8..512
        lengths = rs.randint(8, 513, size=N)
        sents = [rs.randint(3, cfg.vocab_size, size=int(n)).astype(np.uint32) for n in lengths]
        for _ in range(3):
            m.embed_packed(sents)
        per = [host_rate(lambda: m.embed_packed(sents), 1.0) for _ in range(a.rounds)]
        f = flop(cfg, lengths)
        models.prof_begin()
        m.embed_packed(sents)
        prof = models.prof_end()
        line = {"model": name, "config": cfg.__dict__, "batch": "b_packed_256_len_8_512", "sentences": N, "tokens": int(lengths.sum()),
                "tflop_per_batch": round(f / 1e12, 3), "host_ms_per_batch": stats([x * 1e3 for x in per]),
                "emb_per_s": round(N / np.median(per)), "tflops": round(f / np.median(per) / 1e12, 1),
                **split(cfg, prof, int(lengths.sum())),
                "timing": f"host clock around synchronous fl_embed_packed calls (upload + encoder + read-back), {a.rounds} windows of "
                          ">= 1 s; kernel split from a separate fl_prof run"}
        lines.append(line)
        print(json.dumps(line), flush=True)
        del m
    if a.out:
        with open(a.out, "w") as fo:
            for ln in lines:
                fo.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
