"""FP8 (e4m3) KV caches without a device: the oracle's rounding rule, the ABI errors that need no device, and the SASS of the FP8
stream-K decode attention."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
import torch

from kv_fp8_ref import round_e4m3

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torch_e4m3(x):
    return torch.from_numpy(np.asarray(x, dtype=np.float32)).to(torch.float8_e4m3fn).float().numpy()


def test_rounding_matches_torch_on_in_range_values():
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.standard_normal(20000).astype(np.float32) * s for s in (1e-3, 1e-2, 0.1, 1.0, 10.0, 100.0)])
    x = x[np.abs(x) <= 448]
    assert np.array_equal(round_e4m3(x), _torch_e4m3(x))


def test_rounding_of_subnormals_ties_and_signed_zero():
    sub = np.arange(-8, 9, dtype=np.float32) * np.float32(2.0 ** -9)       # every subnormal (and 0, the smallest normal)
    assert np.array_equal(round_e4m3(sub), sub)
    ties = np.array([2.0 ** -10, 3 * 2.0 ** -10, 1.0625, 1.1875, 17.0, 19.0, 232.0, -1.0625], dtype=np.float32)
    want = np.array([0.0, 2.0 ** -8, 1.0, 1.25, 16.0, 20.0, 224.0, -1.0], dtype=np.float32)       # half to even
    assert np.array_equal(round_e4m3(ties), want)
    assert np.array_equal(round_e4m3(ties), _torch_e4m3(ties))
    z = round_e4m3(np.array([0.0, -0.0, -1e-30, 1e-30], dtype=np.float32))
    assert np.array_equal(z, [0.0, 0.0, 0.0, 0.0]) and list(np.signbit(z)) == [False, True, True, False]


def test_rounding_saturates_instead_of_nan():
    x = np.array([448.0, 460.0, 464.0, 1000.0, 1e30, np.inf, -460.0, -1000.0, -np.inf], dtype=np.float32)
    assert np.array_equal(round_e4m3(x), [448, 448, 448, 448, 448, 448, -448, -448, -448])
    assert np.isnan(_torch_e4m3(np.float32(1000.0)))      # why torch is no reference above 448


def test_create_pool_kv_errors_that_need_no_device():
    from fastllm_b200 import _lib
    lib = _lib.load()
    out = C.c_void_p()
    assert lib.fl_cache_create_pool_kv(None, 4, 256, 256, 1, C.byref(out)) == -1          # FL_ERR_INVALID: NULL model
    assert b"NULL" in lib.fl_last_error()


def test_fp8_stream_k_decode_is_tma_fed_and_does_not_spill():
    spec = importlib.util.spec_from_file_location("sass_summary", os.path.join(ROOT, "tools", "sass_summary.py"))
    ss = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ss)
    mn = ss.kernel_mnemonics()
    names = sorted(mn)
    fam = {p: mn[n] for n, p in zip(names, ss.demangle(names)) if p.startswith("attn_sk_decode_kernel<") and "unsigned char" in p}
    assert sorted(fam) == sorted(f"attn_sk_decode_kernel<{d}, unsigned char>" for d in (16, 32, 64, 128))
    for name, c in fam.items():
        assert c["UTMALDG.2D"] >= 2 and c["SYNCS"] >= 4, name       # K and V pages arrive by 2-D TMA
        assert c["HMMA.16816.F32.BF16"] >= 8 and c["LDSM"] >= 4, name
    if not os.path.exists(ss.PTXAS_LOG):
        from fastllm_b200 import build
        build.build_library(force=True)
    res = ss.ptxas_resources()
    rn = sorted(res)
    fp8 = {p: res[n] for n, p in zip(rn, ss.demangle(rn)) if "unsigned char" in p or p.startswith("attn_prefill_tc_fp8_kernel<")}
    assert len(fp8) >= 11, sorted(fp8)
    for p, r in fp8.items():
        assert r[2] == 0 and r[3] == 0, p                          # no local-memory spill stores / loads


def test_fp8_reference_is_the_oracle_with_another_rounding(monkeypatch):
    """Fp8KvCausalLM restates CausalLM's attention: with the bf16 rounding in place of round_e4m3 it returns the logits of
    CausalLM(kv_dtype="bf16") bit for bit (prompt, then a decode step on the cache it built)."""
    import kv_fp8_ref
    from oracle import causal_lm as ocl
    from oracle import synth
    from helpers import TINY
    for name in ("llama", "mistral_sw", "qwen2", "mixtral"):
        cfg = TINY[name]
        w = ocl.synth_weights(cfg, 5, 0.08)
        ids = synth.token_ids(3, cfg.vocab_size, (12,))
        monkeypatch.setattr(kv_fp8_ref, "round_e4m3", synth.round_bf16)
        a, b = kv_fp8_ref.Fp8KvCausalLM(cfg, w), ocl.CausalLM(cfg, w, kv_dtype="bf16")
        for part, ro in ((ids[None, :11], 0), (ids[None, 11:], 11)):
            assert np.array_equal(a.forward(part, ro), b.forward(part, ro)), name
        monkeypatch.undo()
        e = kv_fp8_ref.Fp8KvCausalLM(cfg, w).forward(ids[None], 0)
        assert not np.array_equal(e, ocl.CausalLM(cfg, w, kv_dtype="bf16").forward(ids[None], 0)), name
