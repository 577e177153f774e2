#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json): decode tok/s and % of the HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one decode step of the workload's batch through the whole model (all layers + lm_head + arg-max).
Default workload: Mistral-7B-v0.1 bf16, batch 1, 2k context (the configuration the headline metric is quoted on).
  value  = whole-job tokens/s, device-resident greedy loop (CUDA graph per step), CUDA-event timed on the library's stream
  e2e    = the same metric through the reference-facing call fl_forward(): host ids in (H2D), f32 logits out (D2H),
           host arg-max, exactly the per-token traffic of the reference's generate loop (models/mod.rs:411-453)
  roofline = the GEMV family (dominant kernels), algorithmic weight bytes / CUDA-event duration, live in this run
  cpu_baseline = the oracle port (numpy f32 restatement of candle's CPU path) on this box's host cores, bounded sample
`--impl reference` times that CPU port alone.  Weights are synthetic (device-generated, bit-identical to oracle/synth.py).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries ONE JSON line: NCCL's INFO log (communicator size, transports, NVLS) goes to stderr, where a driver can read the
# `nranks` of the communicator the library created.  An explicit NCCL_DEBUG=INFO/TRACE or NCCL_DEBUG_FILE from the caller wins.
if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
    os.environ["NCCL_DEBUG"] = "INFO"
    os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
if os.environ.get("FL_BENCH_ENV_DEBUG"):
    sys.stderr.write("bench.py env: " + repr({k: v for k, v in os.environ.items() if k.startswith(("NCCL", "TORCH_NCCL", "OMP"))}) + "\n")
# torch.distributed.run exports OMP_NUM_THREADS=1 to every rank.  The CPU arm (`--impl reference`) runs on rank 0 ALONE and must
# use all host cores at every N, so the BLAS pool is sized before numpy loads it (and pinned again at run time, run_reference).
if "--impl" in sys.argv and "reference" in sys.argv and int(os.environ.get("RANK", "0")) == 0:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (arch key, batch, context, description)
    "mistral7b_b1": ("mistral7b", 1, 2048, "Mistral-7B-v0.1 bf16 decode, batch 1, 2k context"),
    "mistral7b_b8": ("mistral7b", 8, 2048, "Mistral-7B-v0.1 bf16 decode, batch 8, 2k context"),
    "tinyllama_b1": ("tinyllama", 1, 128, "TinyLlama-1.1B bf16 decode, batch 1, 128-token prompt"),
    "qwen25_7b_b1": ("qwen25_7b", 1, 2048, "Qwen2.5-7B bf16 decode, batch 1, 2k context"),
    "mistral7b_b64": ("mistral7b", 64, 2048, "Mistral-7B-v0.1 bf16 decode, batch 64, 2k context"),
    "minilm_256x128": ("minilm", 256, 128, "all-MiniLM-L6-v2 (BertModel) embeddings, batch 256 x seq 128"),
    "mixtral8x7b_b32": ("mixtral8x7b", 32, 2048, "Mixtral-8x7B bf16 top-2 MoE decode, batch 32, 2k context"),
    "qwen25_7b_prefill4k": ("qwen25_7b", 1, 4096, "Qwen2.5-7B bf16 prefill 4096 tokens (+ 256 decode steps reported beside it)"),
}
QWEN_PREFILL_TFLOP_4K = 56.83         # SURVEY.md section 8d: 53.46 linear + 3.37 causal attention
MINILM_FLOP_PER_TOKEN = 22.41e6      # SURVEY.md section 8d: 2 x 10.617 M linear + 4 T H 6 attention at T = 128


def oracle_config(key):
    """CPU legs only (cpu_baseline / --impl reference): the oracle's config for the workload."""
    from oracle import causal_lm as ocl
    return {"mistral7b": ocl.MISTRAL_7B, "tinyllama": ocl.TINYLLAMA, "qwen25_7b": ocl.QWEN25_7B}[key]


def peaks(kind="hbm"):
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"] if kind == "hbm" else d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json)"
    return (6650.0 if kind == "hbm" else 1400.0), "fallback (B200_PROFILING.md)"


def ncu_traffic_per_step():
    """(DRAM bytes per decode step, source) of decode_persistent_kernel from the newest committed `ncu --set full` capture
    (profiles/rNN_persistent*_full_raw.csv: one launch of Mistral-7B b=1 at KV 2048; `_<n>step_` in the file name = decode steps
    inside the captured launch, 8 when absent).  The figure is NOT measured in this run -- ncu cannot run inside a timed bench --
    so the line names the file it comes from; (None, None) if unavailable."""
    import csv
    import glob
    import re
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_persistent*_full_raw.csv")))
    if not cands:
        return None, None
    p = cands[-1]
    try:
        rows = list(csv.reader(open(p)))
        hdr, units, r = rows[0], rows[1], rows[2]
        scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        tot = 0.0
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = hdr.index(name)
            tot += float(r[i]) * scale[units[i]]
        m = re.search(r"_(\d+)step_", os.path.basename(p))
        steps = int(m.group(1)) if m else 8
        return tot / steps, "committed ncu capture " + os.path.relpath(p, ROOT) + f" ({steps} step(s) per launch)"
    except Exception:
        return None, None


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array the last timed step handed its caller, as out_dir/<name>.npy -- token ids as float64 (exact),
    real values as float32 (float64 stays float64).  The inputs are seeded, so two builds run with the same arguments can be
    compared output for output."""
    conv = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        conv[name] = a.astype(np.float32 if a.dtype.kind == "f" and a.dtype.itemsize <= 4 else np.float64)
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def minilm_measure(local_rank, b, t, repeats, e2e_iters, warm=3):
    """-> dict(device ms/batch, e2e s/batch, embeddings of the timed batch) for b x t synthetic sentences on this rank's GPU."""
    from fastllm_b200 import models
    m = models.MiniLMModel(models.BertConfig(), None, local_rank, random_seed=0)
    ids = (np.arange(b * t, dtype=np.uint64).reshape(b, t) * 7919 % 30000 + 3).astype(np.uint32)
    for _ in range(warm):
        m.embed_ids(ids)
    emb, ms = m.embed_ids_timed(ids, repeats)
    t0 = time.perf_counter()
    for _ in range(e2e_iters):
        m.embed_ids(ids)                                   # host ids in (H2D), f32 [b, 384] out (D2H)
    e2e_s = (time.perf_counter() - t0) / e2e_iters
    return {"ms": ms / repeats, "e2e_s": e2e_s, "embeddings": emb}


def cpu_minilm_sample(b=16, t=128, iters=2):
    from oracle import bert as obert
    from oracle import synth
    cfg = obert.MINILM_L6
    m = obert.MiniLM(cfg, obert.synth_weights(cfg, 0, 0.02))
    ids = synth.token_ids(2, cfg.vocab_size, (b, t))
    m.embed_ids(ids)
    t0 = time.perf_counter()
    for _ in range(iters):
        m.embed_ids(ids)
    dt = (time.perf_counter() - t0) / iters
    return b / dt, f"{iters} batches of {b} x {t} tokens, f32 numpy/BLAS port of the reference's CPU encoder (embeddings.rs), all host threads"


def run_minilm(args, rank, world, local_rank):
    import torch
    from fastllm_b200 import models
    _, B, T, desc = WORKLOADS["minilm_256x128"]
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    b = B // world                                        # batch-data-parallel: 256 / N sentences per GPU, no collective
    K, W = args.steps, args.warmup
    l0 = models.launch_count()
    with ClockSampler(local_rank) as clk:
        minilm_measure(local_rank, b, T, W, 1, warm=1)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0w = time.time()
        r = minilm_measure(local_rank, b, T, K, max(3, min(K, 20)), warm=0)
        torch.cuda.synchronize()
        t1w = time.time()
        time.sleep(0.12)
    launches = models.launch_count() - l0
    if args.dump_outputs and rank == 0:           # every rank embeds the same sentences
        dump_outputs(args.dump_outputs, {"embeddings": r["embeddings"]})
    tt = torch.tensor([r["ms"], r["e2e_s"]], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, e2e_s = float(tt[0]), float(tt[1])
    if rank != 0:
        return
    value = B / (ms / 1e3)
    peak, src = peaks("tensor")
    tflops = MINILM_FLOP_PER_TOKEN * b * T / (ms / 1e3) / 1e12           # per GPU
    cpu = None
    if world == 1 and not args.no_cpu:
        v, sample = cpu_minilm_sample()
        cpu = {"value": v, "unit": "emb/s", "cores": os.cpu_count(), "kind": "port", "sample": sample}
    line = {"metric": "embeddings_per_s", "value": value, "unit": "emb/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": desc, "batch": B, "seq_len": T, "per_gpu_batch": b, "l2": "L2 not flushed: activations of one batch (25-100 MB per tensor) cycle through L2 as in production",
                       "parallelism": "single GPU" if world == 1 else f"dp{world}: {b} sentences per GPU, no collective",
                       "weights": "synthetic N(0,0.02^2)-like bf16, seed 0"},
            "clocks": clk.summary(t0w, t1w),
            "e2e": {"value": B / e2e_s, "unit": "emb/s", "h2d_bytes_per_step": int(b * T * 4), "d2h_bytes_per_step": int(b * 384 * 4)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": tflops, "peak": peak, "unit": "TFLOP/s", "frac": tflops / peak, "traffic": None,
                         "kernel": "gemm_tc_kernel<128,EPI> (tcgen05/TMEM/TMA) x 24 + bert_attn_kernel x 6 per batch: whole-encoder algorithmic FLOPs / device time",
                         "peak_source": src},
            "cpu_baseline": cpu}
    print(json.dumps(line), flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons.  Started before the warm-up (nvidia-smi takes ~1 s to produce its first line);
    `summary(t0, t1)` keeps the samples whose timestamp falls inside the timed region [t0, t1] (host clock)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev, self.rows, self.proc = dev, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.dev)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        import datetime
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = time.time()
            self.rows.append([ts] + f[1:])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0=None, t1=None):
        rows = [r for r in self.rows if t0 is None or (t0 - 0.05 <= r[0] <= t1 + 0.05)]
        where = "timed region"
        if not rows:                       # very short timed region: fall back to everything sampled under load
            rows, where = self.rows, "warm-up + timed region"
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "window": where}


# --------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores.  `--impl reference` runs WHOLE decode steps of the full model when its f32 weights
# fit the host's free memory (TinyLlama 4.1 GB, Mistral-7B 29 GB, Qwen2.5-7B 30 GB), so ms_per_step x steps is wall time actually
# spent; otherwise (and for the bounded cpu_baseline sample of the GPU arm) a 2-layer slice is timed and extrapolated, and the
# line says so ("extrapolated": true).
# --------------------------------------------------------------------------------------------------------------------
def _mem_available_bytes():
    """Free host memory this process may use: /proc/meminfo MemAvailable, capped by the cgroup limit when there is one."""
    avail = 0
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
    except Exception:
        return 0
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            m = open(lim).read().strip()
            if m != "max":
                avail = min(avail, int(m) - int(open(cur).read().strip()))
        except Exception:
            pass
    return max(avail, 0)


def _pin_blas_threads():
    """All host cores for the BLAS pool, whatever OMP_NUM_THREADS the launcher exported (torchrun sets 1) -> threads in use."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=n)
        return max([p.get("num_threads", 1) for p in threadpool_info()] or [n])
    except Exception:
        return n


class CpuSample:
    """`sample_layers` layers of the model (all of them when sample_layers == L) at KV length `ctx` on the host cores (oracle
    port, numpy f32 / BLAS).  One step = one decode step of the slice + one lm_head; a partial slice is extrapolated:
    T_full = L * T_layer + T_head."""

    def __init__(self, cfg, batch, ctx, sample_layers=2, max_steps=64):
        from dataclasses import replace
        from oracle import causal_lm as ocl
        self.cfg, self.batch, self.ctx = cfg, batch, ctx
        self.sample_layers = min(sample_layers, cfg.num_hidden_layers)
        self.full = self.sample_layers == cfg.num_hidden_layers
        self.small = replace(cfg, num_hidden_layers=self.sample_layers, max_position_embeddings=ctx + max_steps + 8)
        self.w = ocl.synth_weights(self.small, 0, 0.02)
        self.m = ocl.CausalLM(self.small, self.w)
        self.rng = np.random.default_rng(0)
        self.ids = np.full((batch, 1), 5, dtype=np.uint32)
        self.x = self.rng.standard_normal((batch, self.small.hidden_size), dtype=np.float32)
        self.pos = ctx
        self.reset_kv()

    def reset_kv(self):
        d, nkv = self.small.head_dim, self.small.num_key_value_heads
        self.m.kv = [(self.rng.standard_normal((self.batch, nkv, self.ctx, d), dtype=np.float32) * 0.5,
                      self.rng.standard_normal((self.batch, nkv, self.ctx, d), dtype=np.float32) * 0.5)
                     for _ in range(self.sample_layers)]
        self.pos = self.ctx

    def step(self):
        """-> seconds per full-model decode step (measured whole when the slice is the full model, else extrapolated)."""
        from oracle import candle_ops as ops
        t0 = time.perf_counter()
        self.m.forward(self.ids, self.pos)
        t_total = time.perf_counter() - t0
        self.pos += 1
        if self.full:
            return t_total
        t0 = time.perf_counter()
        ops.linear(ops.rms_norm(self.x, self.w["model.norm.weight"], self.small.rms_norm_eps), self.w["lm_head.weight"])
        t_head = time.perf_counter() - t0
        t_layer = max(t_total - t_head, 1e-9) / self.sample_layers
        return self.cfg.num_hidden_layers * t_layer + t_head

    def describe(self, n):
        L = self.cfg.num_hidden_layers
        if self.full:
            return (f"{n} whole decode steps of the full model ({L} layers + lm_head) at KV length {self.ctx}, f32 numpy/BLAS port of "
                    f"candle's CPU path, nothing extrapolated")
        return (f"{n} decode steps of {self.sample_layers}/{L} layers + lm_head at KV length {self.ctx}, "
                f"f32 numpy/BLAS port of candle's CPU path, extrapolated to {L} layers")


def cpu_full_model_fits(cfg, batch, ctx):
    """f32 weights + f32 KV of the whole model against the host's available memory (x1.25 head-room for temporaries)."""
    H, I, V, L = cfg.hidden_size, cfg.intermediate_size, cfg.vocab_size, cfg.num_hidden_layers
    d = cfg.head_dim
    per_layer = H * (cfg.num_attention_heads + 2 * cfg.num_key_value_heads) * d + H * cfg.num_attention_heads * d + 3 * H * I
    need = 4 * (L * per_layer + 2 * V * H) + 4 * 2 * L * batch * cfg.num_key_value_heads * ctx * d
    return need * 1.25 < _mem_available_bytes()


def cpu_decode_sample(cfg, batch, ctx, n_steps=3, warmup=1, budget_s=60.0, full=False):
    threads = _pin_blas_threads()
    full = full and cpu_full_model_fits(cfg, batch, ctx)
    cs = CpuSample(cfg, batch, ctx, sample_layers=cfg.num_hidden_layers if full else 2, max_steps=n_steps + warmup)
    for _ in range(warmup):
        cs.step()
    ts, t0 = [], time.perf_counter()
    for _ in range(n_steps):
        ts.append(cs.step())
        if time.perf_counter() - t0 > budget_s:
            break
    return batch / float(np.mean(ts)), cs.describe(len(ts)), threads, len(ts), (not cs.full)


def run_reference(args, rank):
    if rank != 0:
        return
    arch, batch, ctx, desc = WORKLOADS[args.workload]
    if args.workload in ("mixtral8x7b_b32", "qwen25_7b_prefill4k"):
        print(json.dumps({"impl": "reference", "unavailable": f"no CPU leg for workload {args.workload}: the reference does not wire Mixtral "
                          "and a 4096-token f32 prefill of a 7B model does not fit a bounded CPU sample; the decode workloads carry the CPU baseline"}),
              flush=True)
        return
    v, sample, threads, n, extrapolated = cpu_decode_sample(oracle_config(arch), batch, ctx, args.steps, max(1, min(args.warmup, 3)), 150.0,
                                                            full=True)
    line = {"impl": "reference", "metric": "decode_tokens_per_s", "value": v, "unit": "tok/s", "n_gpus": args.gpus, "steps": n,
            "warmup": args.warmup, "ms_per_step": 1000.0 * batch / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "extrapolated": extrapolated,
            "config": {"workload": desc, "batch": batch, "context": ctx, "parallelism": "host cores"},
            "cpu_baseline": {"value": v, "unit": "tok/s", "cores": threads, "kind": "port", "sample": sample, "extrapolated": extrapolated},
            "e2e": {"value": v, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------------------
def _setup_dist(world, local_rank):
    import torch
    if world <= 1:
        return None
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    return dist


def decode_loop_ms(cache, batch, ctx, steps, warm):
    """Device-resident greedy decode of `steps` steps from KV length ctx -> CUDA-event ms on the library's stream."""
    first = np.full((batch,), 5, dtype=np.uint32)
    cache.fill_synthetic(batch, ctx)
    cache.decode_greedy_loop(first, ctx, warm)
    cache.fill_synthetic(batch, ctx)
    _, ms = cache.decode_greedy_loop(first, ctx, steps)
    return ms


def teacher_forced_logits(model_dev, prompts, feed, routing=False):
    """Real prefill of `prompts` [b, T], then one decode step per row of `feed` [steps, b] (FIXED tokens, not the arg-max: random-init
    logits have top-2 gaps down to 1e-3, and one flipped arg-max would turn a summation-order difference into a different
    continuation) -> f32 logits [steps + 1, b, vocab].  Used by the correctness legs of the sharded runs.  routing=True (Mixtral)
    also returns the router's picks [steps + 1, b, layers, top_k] and margins [steps + 1, b, layers] of each call's LAST position."""
    from fastllm_b200 import models
    b, T = prompts.shape
    cache = models.DeviceCache(model_dev, b, T + feed.shape[0] + 8)
    out, sel, mar = [cache.forward(prompts, 0)], [], []

    def record(t):
        if routing:
            ex, mg = cache.moe_routing(b * t)                      # [L, b*t, k], rows are sequence-major
            sel.append(ex.reshape(ex.shape[0], b, t, -1).transpose(1, 2, 0, 3))       # [b, t, L, k]
            mar.append(mg.reshape(mg.shape[0], b, t).transpose(1, 2, 0))

    record(T)
    for s in range(feed.shape[0]):
        out.append(cache.forward(np.ascontiguousarray(feed[s]).reshape(b, 1), T + s))
        record(1)
    if not routing:
        return np.stack(out)
    # per call: did ANY position of the call route differently is what matters (a rerouted prompt token changes the KV every later
    # step attends to), so the prefill keeps all its positions: sel[0] is [b, T, L, k], the rest [b, 1, L, k]
    return np.stack(out), sel, mar


SHARD_TOL = 1.5e-2      # sharded vs single-GPU logits at full depth: the split changes f32 summation order, which flips single bf16
                        # roundings of the KV cache (1 ulp = 2^-8 relative) -- the same bound as the 22-layer kernel-vs-oracle
                        # tolerance in tests/helpers.py; measured 9.7e-3 at TP-8 over 32 layers x 33 positions, 3e-4 at 2 layers
ROUTE_TIE = 1e-3        # a router pick may differ between the runs only where the single-GPU softmax-probability margin is below this


def compare_sharded(got, want, what, routing=None):
    """N-GPU logits against the single-GPU logits of the same synthetic weights and tokens: max-abs difference (the split changes the
    summation order) and arg-max identity -- a differing arg-max is explained only by a single-GPU top-2 gap inside twice that
    difference.  Mixtral (routing = (picks_sharded, picks_single, margins_single), per call [b, t, L, k] / [b, t, L]): top-k routing is
    discontinuous, so a (sequence, step) row is compared only while the sequence has been routed identically in both runs so far;
    every ROOT routing disagreement (one that no earlier disagreement of the same sequence can have caused) must sit on a
    single-GPU router margin below ROUTE_TIE or the check fails."""
    steps, b = got.shape[0], got.shape[1]
    live = np.ones((steps, b), dtype=bool)
    rec = {}
    if routing is not None:
        sel_g, sel_w, mar_w = routing
        rerouted = np.zeros(b, dtype=bool)
        n_diff = n_bad = 0
        worst = 0.0
        n_casc = 0
        for s in range(steps):
            d = (np.sort(sel_g[s], -1) != np.sort(sel_w[s], -1)).any(-1)          # [b, t, L]: the picked SET differs
            n_diff += int(d.sum())
            # Only ROOT disagreements have to sit on a tie.  The router input of (position p, layer l) depends on the routing of every
            # (p' <= p, l' < l) of the same sequence (MoE output -> residual -> attention of the later layers), and on everything routed
            # in earlier calls (the KV cache): once a sequence has been rerouted, its later picks are made on different hidden states
            # and may differ at any margin -- those are consequences, not causes, and the sequence's rows are no longer compared.
            casc = np.zeros_like(d)
            if d.shape[2] > 1:
                before = np.logical_or.accumulate(np.logical_or.accumulate(d, axis=1), axis=2)      # any (p' <= p, l' <= l)
                casc[:, :, 1:] = before[:, :, :-1]                                                   # any (p' <= p, l' <  l)
            casc |= rerouted[:, None, None]
            root = d & ~casc
            n_casc += int((d & casc).sum())
            if root.any():
                worst = max(worst, float(mar_w[s][root].max()))
                n_bad += int((mar_w[s][root] >= ROUTE_TIE).sum())
            rerouted |= d.any((1, 2))
            live[s] = ~rerouted
        rec = {"router_decisions": int(sum(x.shape[0] * x.shape[1] * x.shape[2] for x in sel_w)), "router_disagreements": n_diff,
               "consequences_of_an_earlier_reroute": n_casc, "largest_margin_of_a_root_disagreement": worst, "route_tie": ROUTE_TIE,
               "disagreements_off_a_tie": n_bad,
               "rows_compared": int(live.sum()), "max_abs_all_rows": float(np.abs(got - want).max())}
    diff = float(np.abs(got - want)[live].max()) if live.any() else float("nan")
    top2 = np.partition(want, -2, axis=-1)[..., -2:]
    margin = top2[..., 1] - top2[..., 0]
    ag, aw = got.argmax(-1), want.argmax(-1)
    unexplained = int(((ag != aw) & (margin > 2 * diff) & live).sum())
    ok = unexplained == 0 and diff <= SHARD_TOL and rec.get("disagreements_off_a_tie", 0) == 0 and live.mean() >= 0.5
    return {"check": what, "max_abs": diff, "tol": SHARD_TOL, "argmax_identical": int(((ag == aw) & live).sum()), "of": int(live.sum()),
            "unexplained_flips": unexplained, "min_margin": float(margin.min()), **rec, "greedy32": bool(ok)}


def tinyllama_parity(local_rank):
    """BASELINE.json config 1 against the committed f32-oracle golden (tests/golden/fulldepth_tinyllama.*, written by
    tests/golden/make_fulldepth_golden.py): TinyLlama-1.1B, all 22 layers, 128-token prompt + 64 greedy steps through the
    reference's generate loop.  No oracle code runs here: ids and three full logits rows are compared with the stored ones."""
    from fastllm_b200 import models, presets
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "fulldepth_tinyllama.json")))
    z = np.load(os.path.join(ROOT, "tests", "golden", "fulldepth_tinyllama_logits.npz"))
    cls, cf = presets.PRESETS["tinyllama"]
    model, cache = cls.initialize_model(cf, None, "bf16", local_rank, random_seed=0, std=0.02)
    prompt = z["prompt"]
    t0 = time.perf_counter()
    ids, logits = models.Model(model, cache, eos_token_id=None).generate(prompt, 64, return_logits=True)
    dt = time.perf_counter() - t0
    same = next((i for i, (a, b) in enumerate(zip(ids, g["ids"])) if a != b), len(g["ids"]))
    errs = [float(np.abs(logits[int(k)] - z["logits_" + k]).max()) for k in ("0", "31", "63") if int(k) < max(same, 1)]
    return {"config": "TinyLlama-1.1B (22 layers) random-init, 128-token prompt + 64 greedy steps, vs the committed f32-oracle golden",
            "greedy32": bool(same >= 32), "identical_ids": int(same), "of": 64, "max_abs": max(errs) if errs else None,
            "tol": 6e-2, "tol_note": "max-abs over full 32000-logit rows of steps 0/31/63 vs the pure-f32 oracle; the product keeps a bf16 KV cache "
                                     "(the reference server's dtype, main.rs:120), which is the whole gap (vs the bf16-KV oracle: <= 1.5e-2, tests/test_fulldepth_gpu.py)",
            "min_oracle_margin": g["min_margin"], "e2e_tok_per_s": 64 / dt}


def run_ours(args, rank, world, local_rank):
    import torch
    from dataclasses import replace
    from fastllm_b200 import models, presets, tp as fltp
    arch, batch, ctx, desc = WORKLOADS[args.workload]
    cls, cf = presets.PRESETS[arch]
    # Mistral / Qwen2 shard with tensor parallelism (strong scaling; batch-1 decode all-reduces over NVLink peer memory inside the
    # persistent kernel, the dense path through NCCL); Mixtral shards its experts (expert parallelism, sequences data-parallel,
    # dispatch / combine all-to-all); TinyLlama runs as independent batch-data-parallel replicas (no collective, weak scaling)
    # -- BASELINE.json configs / SURVEY.md section 8e.
    use_tp = world > 1 and arch in ("mistral7b", "qwen25_7b")
    use_ep = world > 1 and arch == "mixtral8x7b"
    dist = _setup_dist(world, local_rank)
    if world > 1 and arch != "tinyllama":
        fltp.init_tensor_parallel(rank, world, local_rank)
    cf1 = cf                                               # the unsharded config (single-GPU twin of the correctness legs)
    if use_tp or use_ep:
        cf = replace(cf, tp_rank=rank, tp_size=world, ep_dp_attention=use_ep)
    sharded = use_tp or use_ep
    jobs = 1 if (sharded or world == 1) else world       # independent model instances in the job
    local_batch = batch // world if use_ep else batch    # expert parallelism: the sequences are dealt out to the ranks

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    model, _ = cls.initialize_model(cf, None, "bf16", local_rank, random_seed=0, std=0.02)
    K, W = args.steps, args.warmup
    cap = ctx + max(K, W, 16) + 8
    cache = models.DeviceCache(model.dev, local_batch, cap)
    first = np.full((local_batch,), 5, dtype=np.uint32)

    # ---- device-resident decode: W warm-up steps, then exactly K timed steps -------------------------------------------
    with ClockSampler(local_rank) as clk:
        cache.fill_synthetic(local_batch, ctx)
        cache.decode_greedy_loop(first, ctx, W)
        cache.fill_synthetic(local_batch, ctx)                # back to KV length = ctx for the timed region
        barrier()
        l0 = models.launch_count()
        t_wall0 = time.time()
        timed_ids, ms = cache.decode_greedy_loop(first, ctx, K)
        barrier()
        t_wall1 = time.time()
        time.sleep(0.12)                                      # let the sampler flush its last lines
    gpu_launches = models.launch_count() - l0
    if args.dump_outputs:
        last_ids = timed_ids[-1]                              # [local_batch]: the token ids the last timed step returned
        if use_ep:                                            # sequences are dealt out to the ranks: collect them in order
            parts = [None] * world
            dist.all_gather_object(parts, last_ids)
            last_ids = np.concatenate(parts)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"next_token_ids": last_ids})
    ms = max_over_ranks(ms)
    value = jobs * batch * K / (ms / 1e3)

    # ---- end to end through the reference-facing call: host ids -> fl_forward -> host logits -> host arg-max ------------
    cache.fill_synthetic(local_batch, ctx)
    ids = first.reshape(local_batch, 1).copy()
    for s in range(min(W, 4)):
        logits = cache.forward(ids, ctx + s)
    cache.fill_synthetic(local_batch, ctx)
    barrier()
    t0 = time.perf_counter()
    for s in range(K):
        logits = cache.forward(ids, ctx + s)                                   # H2D ids + D2H logits inside
        ids = models.sample_argmax_rows(logits).reshape(-1, 1)                 # LogitsProcessor arg-max on the host, every row
    torch.cuda.synchronize()
    e2e = jobs * batch * K / max_over_ranks(time.perf_counter() - t0)

    if rank != 0 and not sharded:
        barrier()
        return

    # ---- roofline of the dominant kernel (family), measured live with CUDA events ---------------------------------------
    # (under tensor / expert parallelism every rank runs this pass: the forward contains collectives)
    cache.fill_synthetic(local_batch, ctx)
    models.prof_begin()
    cache.decode_greedy_loop(first, ctx, 4)
    prof = models.prof_end()
    head_dim = cf.hidden_size // cf.num_attention_heads
    streamed = model.dev.streamed_bytes()                  # this rank's shard under TP / EP
    peak, peak_src = peaks()

    def kv_bytes_per_gpu(bb):
        # TP: this rank's kv heads (a kv head replicated on tp / nkv ranks is read by each of them); EP: this rank's sequences
        nkv_local = max(1, cf.num_key_value_heads // world) if use_tp else cf.num_key_value_heads
        return (bb // world if use_ep else bb) * ctx * cf.num_hidden_layers * nkv_local * head_dim * 2 * 2

    # ---- correctness of the sharded run, inside the measured job: the greedy ids of a REAL prefill + 32 decode steps on N GPUs
    # must equal the ids rank 0 computes alone on an unsharded copy of the same synthetic weights -------------------------------
    parity = None
    if sharded:
        steps_p = 32 if use_tp else 12
        ptoks = 96 if use_tp else 40
        allp = (np.arange(batch * ptoks, dtype=np.uint64).reshape(batch, ptoks) * 7919 % (cf.vocab_size - 3) + 3).astype(np.uint32)
        feed = (np.arange(steps_p * batch, dtype=np.uint64).reshape(steps_p, batch) * 104729 % (cf.vocab_size - 3) + 3).astype(np.uint32)
        sl = slice(rank * local_batch, (rank + 1) * local_batch) if use_ep else slice(None)
        mine = teacher_forced_logits(model.dev, allp[sl], feed[:, sl], routing=use_ep)     # every rank: the forward contains collectives
        got, sel_g = mine, None
        if use_ep:                                                                # sequences are data-parallel: collect every rank's rows
            parts = [None] * world
            dist.all_gather_object(parts, mine)
            got = np.concatenate([p[0] for p in parts], axis=1)
            sel_g = [np.concatenate([p[1][s] for p in parts], axis=0) for s in range(steps_p + 1)]
        barrier()
        if rank == 0:
            solo, _ = cls.initialize_model(cf1, None, "bf16", local_rank, random_seed=0, std=0.02)
            what = (f"{'tp' if use_tp else 'ep'}{world} logits vs single-GPU logits (same synthetic weights; real {ptoks}-token "
                    f"prefill + {steps_p} teacher-forced decode steps, batch {batch})")
            if use_ep:      # the single-GPU run takes the sequences in the ranks' groups (see moe_leg: the dense path is not batch-invariant)
                solo_parts = [teacher_forced_logits(solo.dev, allp[r * local_batch:(r + 1) * local_batch],
                                                    feed[:, r * local_batch:(r + 1) * local_batch], routing=True) for r in range(world)]
                want = np.concatenate([p[0] for p in solo_parts], axis=1)
                sel_w = [np.concatenate([p[1][s] for p in solo_parts], axis=0) for s in range(steps_p + 1)]
                mar_w = [np.concatenate([p[2][s] for p in solo_parts], axis=0) for s in range(steps_p + 1)]
                parity = compare_sharded(got, want, what + f", taken in the ranks' groups of {local_batch}; rows compared while both runs routed "
                                                           "the sequence to the same experts", routing=(sel_g, sel_w, mar_w))
            else:
                parity = compare_sharded(got, teacher_forced_logits(solo.dev, allp, feed), what)
            del solo
        barrier()

    # ---- the rest of the headline metric in the same job: Mistral-7B batch 8 / 64 (tensor-parallel at N > 1), and Mixtral-8x7B
    # batch 32 (single GPU at N = 1, expert-parallel at N = 2 / 4 / 8) -----------------------------------------------------------
    sweep = None
    if args.workload == "mistral7b_b1" and not args.no_extras:
        sweep = []
        try:
            for bb in (8, 64):
                cb = models.DeviceCache(model.dev, bb, ctx + 80)
                msb = max_over_ranks(decode_loop_ms(cb, bb, ctx, 64, 4)) / 64
                by = streamed + kv_bytes_per_gpu(bb)
                sweep.append({"batch": bb, "context": ctx, "value": bb / (msb / 1e3), "unit": "tok/s", "ms_per_step": msb,
                              "algorithmic_bytes_per_gpu": by, "achieved_gbs_per_gpu": by / (msb / 1e3) / 1e9,
                              "hbm_frac": by / (msb / 1e3) / 1e9 / peak, "parallelism": f"tp{world}" if use_tp else "single GPU"})
                del cb
        except Exception as ex:
            sweep.append({"error": str(ex)})
    if rank != 0:
        if args.workload == "mistral7b_b1" and not args.no_extras:
            del cache, model
            moe_leg(args, rank, world, local_rank, dist, peak)
        barrier()
        return

    pk = [p for p in prof if p["kernel"] == "decode_persistent"]
    if pk:      # batch-1: the whole step is ONE persistent kernel; its algorithmic bytes = streamed weights + KV read
        dom, dom_name = pk, "decode_persistent_kernel<D> (whole decode step: weight stream + attention + arg-max, 4 steps per launch here)"
    elif any(p["kernel"].startswith("gemm_tc_") for p in prof):   # dense path: tcgen05 swap-AB weight-streaming GEMMs
        dom = [p for p in prof if p["kernel"].startswith("gemm_tc_")]
        dom_name = "gemm_tc_kernel<BN, F32_T, DUAL_B> family (tcgen05 swap-AB split-K weight streaming: qkv, o, gate|up / experts, down, lm_head)"
    else:       # multi-kernel path: the GEMV family dominates
        dom = [p for p in prof if p["kernel"].startswith("gemv_")]
        dom_name = "gemv_kernel<M,CPT,PRO,EPI> family (qkv+rope, o+resid, gate/up+silu, down+resid, lm_head)"
    gemv_ms = sum(p["ms"] for p in dom)
    gemv_bytes = sum(p["bytes"] for p in dom)
    all_ms = sum(p["ms"] for p in prof)
    achieved = gemv_bytes / (gemv_ms / 1e3) / 1e9 if gemv_ms > 0 else 0.0
    step_bytes = streamed + kv_bytes_per_gpu(batch)
    step_gbs = step_bytes / (ms / K / 1e3) / 1e9
    traffic, traffic_src = None, None
    if pk and args.workload == "mistral7b_b1" and world == 1:
        per_step, traffic_src = ncu_traffic_per_step()
        traffic = per_step * 4 if per_step else None          # the profiled launch runs 4 steps
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "kernel": dom_name,
                "peak_source": peak_src, "kernel_share_of_step": gemv_ms / all_ms if all_ms else None,
                "whole_step": {"algorithmic_bytes_per_gpu": step_bytes, "achieved_gbs": step_gbs, "frac": step_gbs / peak,
                               "frac_of_nominal_8tbs": step_gbs / 8000.0},
                "per_kernel": prof}

    cpu = None
    if world == 1 and not args.no_cpu and arch != "mixtral8x7b":
        v, sample, threads, _, extrap = cpu_decode_sample(oracle_config(arch), batch, ctx, 4, 1, 40.0)
        cpu = {"value": v, "unit": "tok/s", "cores": threads, "kind": "port", "sample": sample, "extrapolated": extrap}

    secondary, moe, prefill = None, None, None
    if args.workload == "mistral7b_b1" and not args.no_extras:
        del cache, model
        moe = moe_leg(args, rank, world, local_rank, dist, peak)
        if world == 1:
            try:
                r = minilm_measure(local_rank, 256, 128, 100, 10, warm=5)     # 100 device-resident batches (~0.2 s): short runs read 5-10 % apart
                secondary = {"metric": "embeddings_per_s", "workload": WORKLOADS["minilm_256x128"][3], "value": 256 / (r["ms"] / 1e3),
                             "e2e": 256 / r["e2e_s"], "unit": "emb/s", "ms_per_batch": r["ms"],
                             "tensor_tflops": MINILM_FLOP_PER_TOKEN * 256 * 128 / (r["ms"] / 1e3) / 1e12}
            except Exception as ex:   # never lose the headline line over the secondary one
                secondary = {"error": str(ex)}
            try:
                parity = tinyllama_parity(local_rank)
            except Exception as ex:
                parity = {"error": str(ex)}
    if world == 1:
        par = "single GPU"
    elif use_tp:
        par = (f"tp{world}: column/row tensor parallel; batch-1 decode all-reduces (x2 per layer) over NVLink peer memory inside the "
               f"persistent kernel, vocab-parallel logits / arg-max exchange")
    elif use_ep:
        par = (f"ep{world}: {cf.num_local_experts // world} expert(s) per GPU, {local_batch} sequences per GPU (attention data-parallel), "
               f"dispatch + combine all-to-all per layer (grouped ncclSend/Recv)")
    else:
        par = f"{world} independent replicas (batch-data-parallel)"
    line = {"metric": "decode_tokens_per_s", "value": value, "unit": "tok/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak" if arch == "tinyllama" else "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": desc, "batch": batch, "context": ctx, "l2": "inputs larger than L2 (weights streamed once per step)",
                       "parallelism": par, "kv_cache": "bf16 paged, synthetic prefill", "weights": "synthetic N(0,0.02^2)-like bf16, seed 0"},
            "clocks": clk.summary(t_wall0, t_wall1),
            "e2e": {"value": e2e, "unit": "tok/s", "h2d_bytes_per_step": int(local_batch * 4), "d2h_bytes_per_step": int(local_batch * cf.vocab_size * 4)},
            "gpu_launches": int(gpu_launches), "roofline": roofline, "parity": parity, "cpu_baseline": cpu, "secondary": secondary,
            "batch_sweep": sweep, "moe": moe}
    print(json.dumps(line), flush=True)
    barrier()
    for leg in (parity if sharded else None, (moe or {}).get("parity")):
        if leg is not None and leg.get("greedy32") is False:
            sys.stderr.write("bench.py: the sharded run does not reproduce the single-GPU results: " + json.dumps(leg) + "\n")
            sys.exit(3)


def moe_leg(args, rank, world, local_rank, dist, peak):
    """Mixtral-8x7B bf16 top-2 MoE decode, batch 32, 2k context, inside the default job: one GPU at N = 1 (93 GB of weights),
    expert-parallel with data-parallel attention at N = 2 / 4 / 8 -- with the N-GPU greedy ids checked against rank 0's
    single-GPU run of the same weights.  Every rank calls this (the forward contains collectives); rank 0 returns the record."""
    import torch
    from dataclasses import replace
    from fastllm_b200 import models, presets
    _, batch, ctx, desc = WORKLOADS["mixtral8x7b_b32"]
    cls, cf1 = presets.PRESETS["mixtral8x7b"]
    if world > 1 and (cf1.num_local_experts % world or batch % world):
        return None

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    try:
        cf = replace(cf1, tp_rank=rank, tp_size=world, ep_dp_attention=True) if world > 1 else cf1
        lb = batch // world
        model, _ = cls.initialize_model(cf, None, "bf16", local_rank, random_seed=0, std=0.02)
        cache = models.DeviceCache(model.dev, lb, ctx + 80)
        ms = max_over_ranks(decode_loop_ms(cache, lb, ctx, 48, 4)) / 48
        del cache
        head_dim = cf.hidden_size // cf.num_attention_heads
        by = model.dev.streamed_bytes() + lb * ctx * cf.num_hidden_layers * cf.num_key_value_heads * head_dim * 4
        rec = {"workload": desc, "value": batch / (ms / 1e3), "unit": "tok/s", "ms_per_step": ms,
               "parallelism": "single GPU" if world == 1 else f"ep{world}: {cf.num_local_experts // world} expert(s) + {lb} sequences per GPU, dispatch/combine all-to-all",
               "algorithmic_bytes_per_gpu": by, "achieved_gbs_per_gpu": by / (ms / 1e3) / 1e9, "hbm_frac": by / (ms / 1e3) / 1e9 / peak}
        if world > 1:
            steps_p, ptoks = 12, 40
            allp = (np.arange(batch * ptoks, dtype=np.uint64).reshape(batch, ptoks) * 7919 % (cf.vocab_size - 3) + 3).astype(np.uint32)
            feed = (np.arange(steps_p * batch, dtype=np.uint64).reshape(steps_p, batch) * 104729 % (cf.vocab_size - 3) + 3).astype(np.uint32)
            mine = teacher_forced_logits(model.dev, allp[rank * lb:(rank + 1) * lb], feed[:, rank * lb:(rank + 1) * lb], routing=True)
            parts = [None] * world
            dist.all_gather_object(parts, mine)
            got = np.concatenate([p[0] for p in parts], axis=1)
            sel_g = [np.concatenate([p[1][s] for p in parts], axis=0) for s in range(steps_p + 1)]
            del model
            dist.barrier()
            if rank == 0:
                solo, _ = cls.initialize_model(cf1, None, "bf16", local_rank, random_seed=0, std=0.02)
                # the single-GPU run takes the sequences in the SAME groups the ranks own (lb sequences per call): the dense path is not
                # batch-invariant (the stream-K attention cuts the step's page stream by the batch it sees, many-row calls pick other
                # kernels), and with a bf16 KV cache every summation-order difference flips roundings that top-2 routing then amplifies
                # -- measured at EP-8 against ONE batch-32 run: 46 near-tie reroutes in 53 k decisions, 89 % of the rows rerouted.
                # Group for group the two runs differ only by what expert parallelism changes (dispatch, per-expert row blocks, combine).
                solo_parts = [teacher_forced_logits(solo.dev, allp[r * lb:(r + 1) * lb], feed[:, r * lb:(r + 1) * lb], routing=True)
                              for r in range(world)]
                del solo
                want = np.concatenate([p[0] for p in solo_parts], axis=1)
                sel_w = [np.concatenate([p[1][s] for p in solo_parts], axis=0) for s in range(steps_p + 1)]
                mar_w = [np.concatenate([p[2][s] for p in solo_parts], axis=0) for s in range(steps_p + 1)]
                rec["parity"] = compare_sharded(got, want, f"ep{world} logits vs single-GPU logits of the same sequence groups (real {ptoks}-token "
                                                            f"prefill + {steps_p} teacher-forced decode steps, {world} x batch {lb}); rows compared "
                                                            "while both runs routed the sequence to the same experts", routing=(sel_g, sel_w, mar_w))
            dist.barrier()
        return rec if rank == 0 else None
    except Exception as ex:
        return {"error": str(ex)} if rank == 0 else None


def run_prefill(args, rank, world, local_rank):
    """Qwen2.5-7B: a "step" is one 4096-token prefill from an empty cache (tensor-core bound); the 256 decode steps that follow
    in BASELINE.json's config are timed once and reported beside it."""
    import torch
    from dataclasses import replace
    from fastllm_b200 import models, presets, tp as fltp
    arch, batch, T, desc = WORKLOADS[args.workload]
    cls, cf = presets.PRESETS[arch]
    dist = _setup_dist(world, local_rank)
    if world > 1:
        fltp.init_tensor_parallel(rank, world, local_rank)
        cf = replace(cf, tp_rank=rank, tp_size=world)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    model, _ = cls.initialize_model(cf, None, "bf16", local_rank, random_seed=0, std=0.02)
    K, W = args.steps, min(args.warmup, 3)
    ids = (np.arange(T, dtype=np.uint64) * 7919 % 150000 + 3).astype(np.uint32)[None]
    cache = models.DeviceCache(model.dev, 1, T + 264)
    with ClockSampler(local_rank) as clk:
        for _ in range(W):
            cache.reset(); cache.forward_greedy(ids, 0)
        barrier()
        l0 = models.launch_count()
        t_wall0 = time.time()
        t0 = time.perf_counter()
        for _ in range(K):
            cache.reset()
            nxt = cache.forward_greedy(ids, 0)                  # host ids in (H2D 16 KB), next id out (D2H): the e2e call IS the step
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / K
        barrier()
        t_wall1 = time.time()
        launches = models.launch_count() - l0
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"next_token_ids": nxt})
        _, dec_ms = cache.decode_greedy_loop(nxt, T, 256)
        time.sleep(0.12)
    tt = torch.tensor([dt, dec_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt, dec_ms = float(tt[0]), float(tt[1])
    cache.reset()
    models.prof_begin(); cache.forward_greedy(ids, 0); prof = models.prof_end()
    if rank != 0:
        barrier()
        return
    dev_ms = sum(p["ms"] for p in prof)
    gemm_ms = sum(p["ms"] for p in prof if p["kernel"].startswith("gemm_tc_"))
    peak, src = peaks("tensor")
    tflop = QWEN_PREFILL_TFLOP_4K * T / 4096
    lin_tflop = 53.46 * T / 4096
    line = {"metric": "prefill_tokens_per_s", "value": T / dt, "unit": "tok/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": desc, "batch": 1, "prompt_tokens": T, "l2": "weights (14 GB) and activations exceed L2",
                       "parallelism": "single GPU" if world == 1 else f"tp{world}: column/row tensor parallel, NCCL all-reduce x2 per layer",
                       "weights": "synthetic N(0,0.02^2)-like bf16, seed 0"},
            "clocks": clk.summary(t_wall0, t_wall1),
            "e2e": {"value": T / dt, "unit": "tok/s", "h2d_bytes_per_step": int(T * 4), "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": lin_tflop / world / (gemm_ms / 1e3), "peak": peak, "unit": "TFLOP/s",
                         "frac": lin_tflop / world / (gemm_ms / 1e3) / peak, "traffic": None,
                         "kernel": "gemm_tc_kernel<128, F32, DUAL_A> (tcgen05 prefill GEMMs; algorithmic linear FLOPs per GPU / their CUDA-event time; "
                                   "the hi/lo activation split issues 2x these FLOPs on the tensor pipe)",
                         "peak_source": src, "kernel_share_of_step": gemm_ms / dev_ms if dev_ms else None,
                         "whole_step": {"algorithmic_tflop": tflop, "achieved_tflops_per_gpu": tflop / world / dt, "frac": tflop / world / dt / peak},
                         "per_kernel": prof},
            "decode_after_prefill": {"steps": 256, "ms_per_step": dec_ms / 256, "tok_per_s": 256 / (dec_ms / 1e3)},
            "cpu_baseline": None}
    print(json.dumps(line), flush=True)
    barrier()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--workload", default="mistral7b_b1", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="default workload: skip the batch sweep / Mixtral / MiniLM / parity legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to its caller as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.workload == "minilm_256x128":
            if rank == 0:
                v, sample = cpu_minilm_sample(16, 128, max(1, min(args.steps, 4)))
                print(json.dumps({"impl": "reference", "metric": "embeddings_per_s", "value": v, "unit": "emb/s", "n_gpus": args.gpus,
                                  "steps": args.steps, "warmup": args.warmup, "ms_per_step": 256e3 / v, "higher_is_better": True,
                                  "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                                  "config": {"workload": WORKLOADS[args.workload][3], "parallelism": "host cores"},
                                  "cpu_baseline": {"value": v, "unit": "emb/s", "cores": os.cpu_count(), "kind": "port", "sample": sample},
                                  "e2e": {"value": v, "unit": "emb/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
            return
        run_reference(args, rank)
        return
    from fastllm_b200 import _lib
    _lib.load()         # built by __graft_entry__.build(): the benchmark compiles nothing, so it also runs from a read-only tree
    if args.workload == "minilm_256x128":
        run_minilm(args, rank, world, local_rank)
    elif args.workload == "qwen25_7b_prefill4k":
        run_prefill(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the project's modules load lazily below: leave no __pycache__ in the tree
    main()
