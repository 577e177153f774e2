"""Reference log-probs for the scoring tests: the oracle's causal-LM forward with the final RMSNorm and lm_head applied at EVERY
position, and an f64 log-softmax."""
from __future__ import annotations

import numpy as np

from oracle import candle_ops as ops
from oracle import causal_lm as ocl

F32 = np.float32


def logits_all(lm: ocl.CausalLM, ids, rope_offset: int, per_position: bool = True) -> np.ndarray:
    """ids u32 [b, t] -> f32 logits [b, t, V] of every position, feeding lm's KV cache like lm.forward does.  The layer loop is
    lm.forward's; per_position=True applies the final norm + lm_head to one position at a time with lm.forward's own expression,
    so [:, -1] is lm.forward's result bit for bit; per_position=False does all positions in one product (wide vocabularies)."""
    cfg, w = lm.cfg, lm.w
    ids = np.asarray(ids)
    assert ids.ndim == 2
    x = ops.embedding(w["model.embed_tokens.weight"], ids)
    for li in range(cfg.num_hidden_layers):
        p = f"model.layers.{li}."
        h = ops.rms_norm(x, w[p + "input_layernorm.weight"], cfg.rms_norm_eps)
        x = (lm._attention(li, h, rope_offset) + x).astype(F32)
        h = ops.rms_norm(x, w[p + "post_attention_layernorm.weight"], cfg.rms_norm_eps)
        ff = lm._moe(li, h) if cfg.arch == ocl.ARCH_MIXTRAL else lm._mlp(li, h)
        x = (ff + x).astype(F32)
    head = lambda v: ops.linear(ops.rms_norm(v, w["model.norm.weight"], cfg.rms_norm_eps), w["lm_head.weight"])
    if not per_position:
        return head(x)
    return np.stack([head(x[:, j, :]) for j in range(x.shape[1])], axis=1)


def log_softmax64(z: np.ndarray) -> np.ndarray:
    z = np.asarray(z, dtype=np.float64)
    m = z.max(axis=-1, keepdims=True)
    return z - m - np.log(np.exp(z - m).sum(axis=-1, keepdims=True))


def top2_gap(z: np.ndarray) -> np.ndarray:
    """max - second largest, per row of the last axis"""
    p = np.partition(np.asarray(z, dtype=np.float64), -2, axis=-1)
    return p[..., -1] - p[..., -2]
