"""Tensor-parallel plumbing on the host side: one process per GPU, torch.distributed for the rendezvous, the library
owns the NCCL communicator (fl_comm_*).  Also the Python statement of the sharding scheme the library applies when a model
is created with tp_size > 1 (csrc/weights_plan.cuh plan_weights): column-parallel q/k/v (by head) and gate/up, row-parallel
o_proj / down_proj (+ all-reduce), vocab-parallel lm_head (+ all-gather); embeddings and norms replicated.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


def init_tensor_parallel(rank: int, world: int, device: int):
    """Rank 0 creates the NCCL unique id, torch.distributed broadcasts it, every rank joins the communicator."""
    import torch
    import torch.distributed as dist
    _lib.init(device)
    lib = _lib.load()
    buf = (C.c_uint8 * 128)()
    if rank == 0:
        _lib.check(lib.fl_comm_unique_id(buf))
    on_gpu = dist.get_backend() == "nccl"
    t = torch.tensor(list(bytes(buf)), dtype=torch.uint8, device=f"cuda:{device}" if on_gpu else "cpu")
    dist.broadcast(t, 0)
    raw = bytes(t.cpu().tolist())
    _lib.check(lib.fl_comm_init(rank, world, (C.c_uint8 * 128).from_buffer_copy(raw)))
    if world > 1:
        # peer-mapped exchange area for the persistent decode kernel's in-kernel all-reduce (CUDA IPC over NVLink)
        h = (C.c_uint8 * 64)()
        _lib.check(lib.fl_comm_ipc_export(h))
        handles = [None] * world
        dist.all_gather_object(handles, bytes(h))
        allh = (C.c_uint8 * (64 * world)).from_buffer_copy(b"".join(handles))
        _lib.check(lib.fl_comm_ipc_import(allh, world, rank))
    return raw


def head_layout(nh: int, nkv: int, rank: int, tp: int):
    """(q_head0, q_real, nh_local, kv_head0, nkv_local) of `rank`: the statement of plan_weights() in csrc/weights_plan.cuh.
    tp <= kv heads: an equal split by head.  tp > kv heads (Qwen2.5-7B at TP-8: 28 q / 4 kv heads): every kv head lives on
    rep = tp / nkv ranks and its query group is dealt out ceil(group / rep) heads per rank, the last rank of a group padding
    with zero heads (zero q rows, zero o_proj columns)."""
    if tp <= nkv:
        assert nh % tp == 0 and nkv % tp == 0
        return rank * (nh // tp), nh // tp, nh // tp, rank * (nkv // tp), nkv // tp
    assert tp % nkv == 0
    rep, group = tp // nkv, nh // nkv
    hpr = -(-group // rep)
    kvh, sub = divmod(rank, rep)
    return kvh * group + sub * hpr, max(0, min(hpr, group - sub * hpr)), hpr, kvh, 1


def shard_window(name: str, shape, nh: int, nkv: int, rank: int, tp: int):
    """(row slice, col slice) of the FULL HF tensor `name` kept by `rank` of `tp` (None = whole axis)."""
    rows = shape[0]
    if tp == 1 or name in ("model.embed_tokens.weight", "model.norm.weight") or name.endswith("layernorm.weight"):
        return slice(None), slice(None)
    q0, qn, _, k0, kn = head_layout(nh, nkv, rank, tp)
    if ".q_proj." in name:
        d = rows // nh
        return slice(q0 * d, (q0 + qn) * d), slice(None)
    if ".k_proj." in name or ".v_proj." in name:
        d = rows // nkv
        return slice(k0 * d, (k0 + kn) * d), slice(None)
    if ".o_proj." in name:
        d = shape[1] // nh
        return slice(None), slice(q0 * d, (q0 + qn) * d)
    if name == "lm_head.weight" or ".gate_proj." in name or ".up_proj." in name:
        n = rows // tp
        return slice(rank * n, (rank + 1) * n), slice(None)
    if ".down_proj." in name:
        n = shape[1] // tp
        return slice(None), slice(rank * n, (rank + 1) * n)
    raise KeyError(name)


def shard_weights(weights: dict, nh: int, nkv: int, rank: int, tp: int) -> dict:
    out = {}
    for k, v in weights.items():
        rs, cs = shard_window(k, v.shape, nh, nkv, rank, tp)
        out[k] = np.ascontiguousarray(v[rs] if v.ndim == 1 else v[rs, cs])
    return out
