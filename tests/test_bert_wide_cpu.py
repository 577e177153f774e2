"""BERT-base / -large shapes without a GPU: the head_dim 64 attention kernels are in the library on the mma.sync tensor-core path
with no spills next to the head_dim 32 ones, and BertConfig.from_json reads a HuggingFace config.json into the preset shapes."""
import dataclasses
import importlib.util
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("sass_summary", os.path.join(ROOT, "tools", "sass_summary.py"))
sass_summary = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(sass_summary)

ATTN = ["bert_attn_kernel<32>", "bert_attn_kernel<64>", "bert_attn_long_kernel<32>", "bert_attn_long_kernel<64>"]


def test_head_dim_64_attention_kernels_use_tensor_cores_without_spills():
    mn = sass_summary.kernel_mnemonics()
    names = sorted(mn)
    by_name = dict(zip(sass_summary.demangle(names), names))
    for k in ATTN:
        assert k in by_name, (k, sorted(p for p in by_name if p.startswith("bert_")))
        c = mn[by_name[k]]
        assert c["HMMA.16816.F32.BF16"] >= 8 and c["LDSM"] >= 4, (k, c)
    # D = 64 does twice the mma.sync work of D = 32 per key tile (Q K^T: 4 k16 steps, P V: 8 output tiles)
    for short in ("bert_attn_kernel<", "bert_attn_long_kernel<"):
        assert mn[by_name[short + "64>"]]["HMMA.16816.F32.BF16"] > mn[by_name[short + "32>"]]["HMMA.16816.F32.BF16"]
    if not os.path.exists(sass_summary.PTXAS_LOG):
        from fastllm_b200 import build
        build.build_library(force=True)
    res = sass_summary.ptxas_resources()
    rnames = sorted(res)
    spills = {p: res[n][2:] for n, p in zip(rnames, sass_summary.demangle(rnames))}
    for k in ATTN + ["embed_ln_kernel<16>", "embed_ln_kernel<32>", "layernorm_kernel<4>", "layernorm_kernel<8>"]:
        assert spills.get(k) == (0, 0), (k, spills.get(k))


def _hf_config(p):
    """A HuggingFace config.json of a BERT checkpoint with preset p's dimensions (plus the keys the encoder does not read)."""
    return {"architectures": ["BertModel"], "model_type": "bert", "attention_probs_dropout_prob": 0.1, "hidden_act": "gelu",
            "hidden_dropout_prob": 0.1, "initializer_range": 0.02, "pad_token_id": 0, "position_embedding_type": "absolute",
            "type_vocab_size": 2, "torch_dtype": "float32", "use_cache": True, **dataclasses.asdict(p)}


@pytest.mark.parametrize("name", ["minilm_l6", "bert_base", "bert_large"])
def test_from_json_gives_the_preset(name, tmp_path):
    from fastllm_b200 import models, presets
    p = presets.BERT_PRESETS[name]
    d = _hf_config(p)
    assert models.BertConfig.from_json(d) == p
    path = tmp_path / "config.json"
    path.write_text(json.dumps(d))
    assert models.BertConfig.from_json(str(path)) == p
    assert models.BertConfig.from_json(path) == p


def test_preset_dimensions():
    from fastllm_b200 import models, presets
    assert presets.MINILM_L6 == models.BertConfig()
    for p, d in ((presets.MINILM_L6, 32), (presets.BERT_BASE, 64), (presets.BERT_LARGE, 64)):
        assert p.hidden_size // p.num_attention_heads == d
    assert (presets.BERT_BASE.num_hidden_layers, presets.BERT_BASE.intermediate_size) == (12, 3072)
    assert (presets.BERT_LARGE.hidden_size, presets.BERT_LARGE.num_hidden_layers, presets.BERT_LARGE.intermediate_size) == (1024, 24, 4096)


@pytest.mark.parametrize("key", ["hidden_size", "num_attention_heads", "num_hidden_layers", "intermediate_size",
                                 "max_position_embeddings", "layer_norm_eps", "vocab_size"])
def test_from_json_missing_dimension_names_it(key):
    from fastllm_b200 import models, presets
    d = _hf_config(presets.BERT_BASE)
    del d[key]
    with pytest.raises(ValueError, match=key):
        models.BertConfig.from_json(d)
