"""Reference for FP8 (e4m3) KV caches (FL_KV_FP8_E4M3), kept with the tests that use it (TEST INFRASTRUCTURE).

round_e4m3 is the rounding a FL_KV_FP8_E4M3 cache applies to K (after RoPE) and V; Fp8KvCausalLM is oracle.causal_lm.CausalLM
with that rounding where kv_dtype="bf16" rounds to bf16 -- the same attention, with another rounding function."""
import numpy as np

from oracle import candle_ops as ops
from oracle import causal_lm as ocl

F32 = np.float32
E4M3_MAX = 448.0


def round_e4m3(x: np.ndarray) -> np.ndarray:
    """f32 -> FP8 e4m3 (1 sign, 4 exponent bits of bias 7, 3 mantissa bits) -> f32, rounded once to nearest even and
    saturating: a magnitude above 448 (the largest finite e4m3) becomes +-448, never NaN.  Normals have 3 mantissa bits
    (spacing 2^(e-3) for |x| in [2^e, 2^(e+1)), e >= -6); below 2^-6 the subnormal spacing 2^-9 applies."""
    x = np.asarray(x, dtype=F32)
    a = np.abs(x).astype(np.float64)
    _, e = np.frexp(a)                                      # a = m * 2^e, m in [0.5, 1): |x| in [2^(e-1), 2^e)
    step = np.ldexp(1.0, np.maximum(e - 1, -6) - 3)         # spacing of e4m3 values around |x|
    r = np.round(a / step) * step                           # exact division (power-of-two step); np.round: half to even
    r = np.minimum(r, E4M3_MAX)                             # 448 < |x| (464 would round to 512): saturate
    return np.copysign(r, x).astype(F32)


class Fp8KvCausalLM(ocl.CausalLM):
    """The oracle's causal LM with K (after RoPE) and V rounded to e4m3 before they enter its cache; every attention, a call's
    attention over its own new tokens included, reads the rounded values."""

    def __init__(self, cfg: ocl.CausalLMConfig, weights: dict, rope_len: int | None = None):
        super().__init__(cfg, weights, rope_len, kv_dtype="f32")
        self.kv_dtype = "fp8_e4m3"

    def _attention(self, li: int, x: np.ndarray, rope_offset: int) -> np.ndarray:
        # CausalLM._attention with round_e4m3 in place of the bf16 rounding
        cfg, w = self.cfg, self.w
        b, t, _ = x.shape
        nh, nkv, d = cfg.num_attention_heads, cfg.num_key_value_heads, cfg.head_dim
        p = f"model.layers.{li}.self_attn."
        bias = (lambda n: w[p + n + ".bias"]) if cfg.qkv_bias else (lambda n: None)
        q = ops.linear(x, w[p + "q_proj.weight"], bias("q_proj")).reshape(b, t, nh, d).transpose(0, 2, 1, 3)
        k = ops.linear(x, w[p + "k_proj.weight"], bias("k_proj")).reshape(b, t, nkv, d).transpose(0, 2, 1, 3)
        v = ops.linear(x, w[p + "v_proj.weight"], bias("v_proj")).reshape(b, t, nkv, d).transpose(0, 2, 1, 3)
        cos, sin = self.cos[rope_offset:rope_offset + t], self.sin[rope_offset:rope_offset + t]
        q = ops.rope_rotate_half(q, cos, sin)
        k = ops.rope_rotate_half(k, cos, sin)
        k, v = round_e4m3(k), round_e4m3(v)
        prev = self.kv[li]
        kv_before = 0 if prev is None else prev[0].shape[2]
        if prev is not None:
            k = np.concatenate([prev[0], k], axis=2)
            v = np.concatenate([prev[1], v], axis=2)
        self.kv[li] = (k, v)
        kk, vv = ops.repeat_kv(k, nh // nkv), ops.repeat_kv(v, nh // nkv)
        att = np.matmul(q, kk.transpose(0, 1, 3, 2)).astype(F32)
        if cfg.arch == ocl.ARCH_LLAMA:
            att = (att / F32(np.sqrt(np.float64(d)))).astype(F32)
        else:
            att = (att * F32(1.0 / np.sqrt(np.float64(d)))).astype(F32)
        m = self._mask(t, kv_before)
        if m is not None:
            att = att + m if cfg.arch != ocl.ARCH_LLAMA else np.where(np.isneginf(m), F32(-np.inf), att)
        att = ops.softmax_last_dim(att)
        y = np.matmul(att, vv).astype(F32).transpose(0, 2, 1, 3).reshape(b, t, nh * d)
        return ops.linear(y, w[p + "o_proj.weight"])
