"""The tensor table each model's plan step lays out (csrc/weights_plan.cuh), checked on the CPU: tests/tensor_table_dump.cu runs
the plan step alone (no CUDA call) and prints the slots.  Names and shapes are checked against the oracle, windows against
tp.shard_window, and at tiny sizes every slot is expanded element by element into the slab.  This covers the tensor-parallel and
expert-parallel layouts of every rank, which otherwise only the multi-GPU tests reach."""
import json
import os
import subprocess

import numpy as np
import pytest

from fastllm_b200 import _lib, tp
from helpers import TINY as TINY_CFG
from oracle import bert as obert
from oracle import causal_lm as ocl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dump_exe(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("tensor_table") / "tensor_table_dump")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "--expt-relaxed-constexpr",
                    os.path.join(ROOT, "tests", "tensor_table_dump.cu"), "-o", exe], check=True, capture_output=True)
    return exe


def _dump(exe, cfg, tp_size=1, rank=0):
    if isinstance(cfg, obert.BertConfig):
        args = [_lib.FL_ARCH["bert"], cfg.hidden_size, cfg.intermediate_size, cfg.vocab_size, cfg.num_hidden_layers,
                cfg.num_attention_heads, cfg.num_attention_heads, cfg.max_position_embeddings, 0, 0, 1, 0]
    else:
        args = [_lib.FL_ARCH[cfg.arch], cfg.hidden_size, cfg.intermediate_size, cfg.vocab_size, cfg.num_hidden_layers,
                cfg.num_attention_heads, cfg.num_key_value_heads, cfg.max_position_embeddings, int(cfg.qkv_bias),
                cfg.num_local_experts, tp_size, rank]
    out = subprocess.run([exe, *map(str, args)], check=True, capture_output=True, text=True).stdout
    return json.loads(out)


def _ep_owned(name, cfg, tp_size, rank):
    """False for an expert of another expert-parallel rank (Mixtral shards by expert: rank r holds E / tp of them)."""
    if cfg.arch != ocl.ARCH_MIXTRAL or ".experts." not in name:
        return True
    e = int(name.split(".experts.")[1].split(".")[0])
    per = cfg.num_local_experts // tp_size
    return rank * per <= e < (rank + 1) * per


def _row_map(m, r):
    row0, mode, head_dim, lane = m
    if mode == 1:       # rope-pair permutation within each head
        h, i = np.divmod(r, head_dim)
        half = head_dim // 2
        return row0 + h * head_dim + np.where(i < half, 2 * i, 2 * (i - half) + 1)
    if mode == 2:       # gate / up interleave
        return row0 + 2 * r + lane
    return row0 + r


def _bytes(s):
    """Slab byte offsets slot s writes: every element of its local block through its RowMap."""
    size = 2 if s["mat"] else 4
    rows = _row_map(s["map"], np.arange(s["rows"], dtype=np.int64))
    elems = (rows[:, None] * s["ld"] + np.arange(s["cols"])[None, :]).ravel()
    return (s["off"] + elems[:, None] * size + np.arange(size)[None, :]).ravel()


def _check_table(t, cfg, tp_size=1, rank=0):
    """Names, shapes, init rule and windows of one table."""
    bert = isinstance(cfg, obert.BertConfig)
    names = obert.tensor_names(cfg) if bert else ocl.tensor_names(cfg)
    want = {n: (shape, kind) for n, shape, kind in names if bert or _ep_owned(n, cfg, tp_size, rank)}
    slots = {s["name"]: s for s in t["slots"]}
    assert len(slots) == len(t["slots"]), "a name is registered twice"
    assert sorted(slots) == sorted(want)
    # tensor parallelism shards the dense models by tensor; Mixtral shards by expert and replicates every tensor it holds
    shard_tp = 1 if bert or cfg.arch == ocl.ARCH_MIXTRAL else tp_size
    nh = cfg.num_attention_heads
    nkv = nh if bert else cfg.num_key_value_heads
    for name, s in slots.items():
        shape, kind = want[name]
        if s["mat"]:
            assert tuple(s["full"]) == shape, name
        else:       # a vector takes [n], or (causal LMs) any [rows, cols] with n elements, like the [E, H] router
            assert s["full"] == [int(np.prod(shape)), 1], name
            assert s["round"] == (not bert), name
        assert s["ones"] == (kind == "norm"), name
        assert s["required"] == (name != "lm_head.weight"), name
        rs, cs = tp.shard_window(name, shape, nh, nkv, rank, shard_tp)
        full_rows, full_cols = s["full"]
        assert (s["win"][0], s["win"][0] + s["rows"]) == rs.indices(full_rows)[:2], name
        assert (s["win"][1], s["win"][1] + s["cols"]) == cs.indices(full_cols)[:2], name


def _check_writes(t, cfg, tp_size=1, rank=0):
    """Every slot stays in the slab and no slab byte is written twice; gate|up fill wgu and q|k|v fill wqkv exactly, except the
    zero heads a rank pads with when there are more ranks than kv heads."""
    per_slot = {s["name"]: _bytes(s) for s in t["slots"]}
    allb = np.concatenate(list(per_slot.values()))
    assert allb.min() >= 0 and allb.max() < t["size"]
    assert np.bincount(allb).max() == 1
    slots = {s["name"]: s for s in t["slots"]}
    if isinstance(cfg, obert.BertConfig):
        for l in range(cfg.num_hidden_layers):
            p, H = f"encoder.layer.{l}.attention.self.", cfg.hidden_size
            for part, elem in (("weight", 2 * H), ("bias", 4)):
                got = np.sort(np.concatenate([per_slot[p + x + "." + part] for x in ("query", "key", "value")]))
                off = slots[p + "query." + part]["off"]
                assert np.array_equal(got, off + np.arange(3 * H * elem)), (l, part)
        return
    shard_tp = 1 if cfg.arch == ocl.ARCH_MIXTRAL else tp_size
    _, q_real, nh_local, _, nkv_local = tp.head_layout(cfg.num_attention_heads, cfg.num_key_value_heads, rank, shard_tp)
    d, H = cfg.head_dim, cfg.hidden_size
    # local rows of wqkv that hold a tensor: the real q heads, then k and v; rows [q_real d, nh_local d) stay zero
    rows = np.concatenate([np.arange(q_real * d), nh_local * d + np.arange(2 * nkv_local * d)])
    for l in range(cfg.num_hidden_layers):
        p = f"model.layers.{l}."
        parts = [("weight", H * 2)] + ([("bias", 4)] if cfg.qkv_bias else [])
        for part, row_bytes in parts:
            got = np.sort(np.concatenate([per_slot[p + f"self_attn.{x}_proj.{part}"] for x in "qkv"]))
            off = slots[p + f"self_attn.q_proj.{part}"]["off"]
            assert np.array_equal(got, off + (rows[:, None] * row_bytes + np.arange(row_bytes)[None, :]).ravel()), (l, part)
        if cfg.arch == ocl.ARCH_MIXTRAL:
            gus = [(n, n.replace("w1.", "w3.")) for n in slots if n.startswith(p) and n.endswith("w1.weight")]
        else:
            gus = [(p + "mlp.gate_proj.weight", p + "mlp.up_proj.weight")]
        for g, u in gus:
            got = np.sort(np.concatenate([per_slot[g], per_slot[u]]))
            rows_local, cols = slots[g]["rows"], slots[g]["cols"]
            assert np.array_equal(got, slots[g]["off"] + np.arange(2 * rows_local * cols * 2)), g


def _tiny(arch, H, I, V, nh, nkv, **kw):
    return ocl.CausalLMConfig(arch, H, I, V, 2, nh, nkv, 1e-5, 1e4, 64, 4096, **kw)


# (name, config, tensor-parallel size): every rank of each is checked
FULL_SIZE = [
    ("tinyllama", ocl.TINYLLAMA, 1),
    *[(f"mistral7b_tp{n}", ocl.MISTRAL_7B, n) for n in (1, 2, 4, 8)],
    ("qwen25_7b_tp8", ocl.QWEN25_7B, 8),
    ("mixtral8x7b_ep4", ocl.MIXTRAL_8X7B, 4),
    ("minilm_l6", obert.BertConfig(384, 12, 6, 1536, 512, 1e-12, 30522), 1),
    ("bert_base", obert.BertConfig(768, 12, 12, 3072, 512, 1e-12, 30522), 1),
    ("bert_large", obert.BertConfig(1024, 16, 24, 4096, 512, 1e-12, 30522), 1),
]
# the same head / expert structure at sizes small enough to expand every element
TINY = [
    ("llama", TINY_CFG["llama"], 1),
    ("qwen2_bias", TINY_CFG["qwen2"], 1),
    *[(f"mistral_heads_tp{n}", _tiny("mistral", 512, 256, 256, 32, 8), n) for n in (1, 2, 4, 8)],
    ("qwen25_heads_tp8", _tiny("qwen2", 448, 256, 256, 28, 4, qkv_bias=True), 8),
    ("mixtral_ep4", _tiny("mixtral", 64, 96, 128, 4, 2, num_local_experts=8), 4),
    ("bert_d32", obert.BertConfig(64, 2, 2, 128, 16, 1e-12, 100), 1),
    ("bert_d64", obert.BertConfig(128, 2, 2, 256, 16, 1e-12, 100), 1),
]


@pytest.mark.parametrize("name,cfg,tp_size", FULL_SIZE, ids=[c[0] for c in FULL_SIZE])
def test_table_names_shapes_windows(dump_exe, name, cfg, tp_size):
    for rank in range(tp_size):
        _check_table(_dump(dump_exe, cfg, tp_size, rank), cfg, tp_size, rank)


@pytest.mark.parametrize("name,cfg,tp_size", TINY, ids=[c[0] for c in TINY])
def test_table_writes(dump_exe, name, cfg, tp_size):
    for rank in range(tp_size):
        t = _dump(dump_exe, cfg, tp_size, rank)
        _check_table(t, cfg, tp_size, rank)
        _check_writes(t, cfg, tp_size, rank)


def test_qwen_tp8_pads_with_zero_heads(dump_exe):
    """Qwen2.5-7B at TP-8: 28 q heads over 8 ranks of 4 local heads; the last rank of each kv group keeps 3 real heads, and
    its q window (and o_proj's column window) ends one head early."""
    d = ocl.QWEN25_7B.head_dim
    for rank in range(8):
        slots = {s["name"]: s for s in _dump(dump_exe, ocl.QWEN25_7B, 8, rank)["slots"]}
        q, o = slots["model.layers.0.self_attn.q_proj.weight"], slots["model.layers.0.self_attn.o_proj.weight"]
        real = 4 if rank % 2 == 0 else 3
        assert q["rows"] == real * d and o["cols"] == real * d and o["ld"] == 4 * d, rank
