"""BERT encoders with head_dim 64 and hidden up to 1024 (BERT-base / -large shapes: e5, gte) on the GPU, against the f32 oracle at the
bars of test_bert_gpu.py, with the packed-batch contract (each fl_embed_packed row bit-identical to the sentence alone), launch
counts, the shapes model creation rejects, and the C++ mirror."""
import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np
import pytest

from oracle import bert as obert
from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COS_TOL = 0.999
LENGTHS = [1, 2, 15, 16, 17, 63, 127, 128, 129, 255, 256, 257, 383, 511, 512]      # test_bert_packed_gpu.py's
TINY64 = obert.BertConfig(128, 2, 2, 256, 512, 1e-12, 200)                          # head_dim 64, both attention kernels
FL_ERR_INVALID, FL_ERR_UNSUPPORTED = -1, -5


def _cos(a, b):
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


def _oracle_cfg(name):
    from fastllm_b200 import presets
    return obert.BertConfig(**dataclasses.asdict(presets.BERT_PRESETS[name]))


def _product(cfg, w, **kw):
    from fastllm_b200 import models
    pc = models.BertConfig(cfg.hidden_size, cfg.num_attention_heads, cfg.num_hidden_layers, cfg.intermediate_size,
                           cfg.max_position_embeddings, cfg.layer_norm_eps, cfg.vocab_size)
    return models.MiniLMModel(pc, w, 0, **kw)


def _sentences(seed, vocab, lengths):
    return [synth.token_ids(seed * 1000 + i, vocab, (n,)) for i, n in enumerate(lengths)]


def _lone(m, sentences):
    return np.concatenate([m.embed_ids(s[None]) for s in sentences])


def _check(got, want, what):
    cos = _cos(got, want)
    err = np.abs(got - want).max()
    print(f"{what}: min cosine {cos.min():.6f}, max-abs {err:.3e}")
    assert cos.min() >= COS_TOL and err <= 2e-2, what


@pytest.fixture(scope="module")
def tiny64():
    w = obert.synth_weights(TINY64, 11, 0.05)
    return _product(TINY64, w), obert.MiniLM(TINY64, w)


@pytest.fixture(scope="module")
def base():
    """BERT-base shapes, device-side synthetic weights (seed 0, std 0.02): the same tensors synth_weights(cfg, 0, 0.02) uploads."""
    return _product(_oracle_cfg("bert_base"), None, random_seed=0, std=0.02)


@pytest.mark.parametrize("t", [1, 7, 33, 127, 128, 129, 200, 512])
def test_tiny_head_dim_64_matches_oracle(tiny64, t):
    m, o = tiny64
    b = 1 if t > 128 else 3
    ids = synth.token_ids(500 + t, TINY64.vocab_size, (b, t))
    _check(m.embed_ids(ids), o.embed_ids(ids), f"tiny d=64 {b}x{t}")
    if t > 3:
        mask = np.ones((b, t), dtype=np.uint32)
        mask[:, -2:] = 0
        _check(m.embed_ids(ids, mask), o.embed_ids(ids, mask), f"tiny d=64 {b}x{t} masked")


def test_head_count_independent_of_width():
    """hidden 384 as in MiniLM, but 6 heads of 64 instead of 12 of 32."""
    cfg = obert.BertConfig(384, 6, 2, 1536, 512, 1e-12, 1000)
    w = obert.synth_weights(cfg, 3, 0.02)
    m, o = _product(cfg, w), obert.MiniLM(cfg, w)
    ids = synth.token_ids(3, cfg.vocab_size, (4, 128))
    _check(m.embed_ids(ids), o.embed_ids(ids), "384/6 heads 4x128")
    sents = _sentences(3, cfg.vocab_size, [300, 9])
    _check(m.embed_packed(sents), np.concatenate([o.embed_ids(s[None]) for s in sents]), "384/6 heads packed 300 + 9")


def test_bert_base_matches_oracle_and_device_init_equals_upload(base):
    cfg = _oracle_cfg("bert_base")
    w = obert.synth_weights(cfg, 0, 0.02)
    o = obert.MiniLM(cfg, w)
    ids = synth.token_ids(20, cfg.vocab_size, (8, 128))
    long = synth.token_ids(21, cfg.vocab_size, (1, 512))
    got, got_long = base.embed_ids(ids), base.embed_ids(long)
    _check(got, o.embed_ids(ids), "BERT-base 8x128")
    _check(got_long, o.embed_ids(long), "BERT-base 1x512")
    up = _product(cfg, w)
    assert np.array_equal(up.embed_ids(ids), got)
    assert np.array_equal(up.embed_ids(long), got_long)


def test_bert_large_mixed_lengths_match_oracle():
    """hidden 1024 / intermediate 4096: N = 1024 and 4096 end in a partial 192-column GEMM tile."""
    cfg = _oracle_cfg("bert_large")
    w = obert.synth_weights(cfg, 5, 0.02)
    sents = _sentences(22, cfg.vocab_size, [37, 300, 128, 3])
    got = _product(cfg, w).embed_packed(sents)
    o = obert.MiniLM(cfg, w)
    _check(got, np.concatenate([o.embed_ids(s[None]) for s in sents]), "BERT-large packed 37, 300, 128, 3")


@pytest.mark.parametrize("which", ["tiny64", "base"])
def test_packed_rows_equal_lone_sentences_bitwise(which, tiny64, base):
    m = tiny64[0] if which == "tiny64" else base
    vocab = m.config.vocab_size
    lengths = list(np.random.RandomState(1).permutation(LENGTHS))
    sents = _sentences(23, vocab, lengths)
    got = m.embed_packed(sents)
    want = _lone(m, sents)
    for i, n in enumerate(lengths):
        assert np.array_equal(got[i], want[i]), (n, np.abs(got[i] - want[i]).max())
    assert np.array_equal(m.embed_packed(sents[::-1]), got[::-1])


def test_launch_counts_and_profile_tags(base):
    from fastllm_b200 import models
    L = base.config.num_hidden_layers
    vocab = base.config.vocab_size

    def launches(f):
        n0 = models.launch_count()
        f()
        return models.launch_count() - n0

    assert launches(lambda: base.embed_ids(synth.token_ids(24, vocab, (4, 128)))) == 7 * L + 2 == 86
    mixed = _sentences(24, vocab, [3, 300, 128, 129, 40])
    assert launches(lambda: base.embed_packed(mixed)) == 8 * L + 2 == 98      # one more attention launch per layer
    models.prof_begin()
    base.embed_packed(mixed)
    prof = models.prof_end()
    assert prof and all(p["kernel"].startswith("bert_") for p in prof), prof
    assert sum(p["launches"] for p in prof) == 98


@pytest.mark.parametrize("hidden,heads,why", [(192, 4, "head_dim 48"), (256, 2, "head_dim 128"), (1088, 17, "hidden 1088 > 1024"),
                                              (160, 5, "hidden not a multiple of 64")])
def test_unsupported_shapes_fail_at_model_creation(hidden, heads, why):
    from fastllm_b200 import FastllmError, models
    with pytest.raises(FastllmError) as e:
        models.MiniLMModel(models.BertConfig(hidden, heads, 1, 4 * hidden, 64, 1e-12, 200), None)
    assert e.value.code == FL_ERR_UNSUPPORTED, (why, str(e.value))


def test_wide_packed_call_over_int32_bound_is_rejected(base):
    from fastllm_b200 import _lib
    cfg = base.config
    ok = _sentences(25, cfg.vocab_size, [9, 200])
    want = base.embed_packed(ok)
    # 1,366 x 512 tokens x max(3 x 768, 3072) = 2.15e9 > 2^31 - 1: rejected on the host before any device work
    n = 1366
    ids = np.ones(n * 512, dtype=np.uint32)
    lengths = np.full(n, 512, dtype=np.int32)
    out = np.empty((n, cfg.hidden_size), dtype=np.float32)
    rc = _lib.load().fl_embed_packed(base.dev.h, ids.ctypes.data_as(C.c_void_p), lengths.ctypes.data_as(C.c_void_p), n,
                                     out.ctypes.data_as(C.c_void_p))
    assert rc == FL_ERR_INVALID
    assert np.array_equal(base.embed_packed(ok), want)


DRIVER = r"""
#include <cstdio>
#include <cstdlib>
#include "fastllm_host.hpp"
using namespace fastllm;
// argv: out.bin hidden heads layers intermediate maxpos vocab, then the sentences' ids, sentences separated by "/";
// synthetic weights (seed 0, std 0.02)
int main(int argc, char** argv) {
    check(fl_init(0));
    fl_config c{};
    c.arch = FL_ARCH_BERT; c.hidden_size = std::atoi(argv[2]); c.num_attention_heads = std::atoi(argv[3]);
    c.num_key_value_heads = c.num_attention_heads; c.num_hidden_layers = std::atoi(argv[4]); c.intermediate_size = std::atoi(argv[5]);
    c.max_position_embeddings = std::atoi(argv[6]); c.vocab_size = std::atoi(argv[7]); c.norm_eps = 1e-12f; c.tp_size = 1;
    auto dev = std::make_shared<DeviceModel>(c);
    check(fl_model_random_init(dev->h, 0, 0.02f));
    check(fl_model_finalize(dev->h));
    MiniLMModel m{dev};
    std::vector<std::vector<uint32_t>> sents(1);
    for (int i = 8; i < argc; ++i) {
        if (std::string(argv[i]) == "/") sents.emplace_back();
        else sents.back().push_back((uint32_t)std::strtoul(argv[i], nullptr, 10));
    }
    const auto rows = m.embed_packed(sents);
    FILE* f = std::fopen(argv[1], "wb");
    for (const auto& r : rows) std::fwrite(r.data(), 4, r.size(), f);
    std::fclose(f);
    return 0;
}
"""


def test_cpp_mirror_embed_packed_equals_python(tmp_path):
    cfg = TINY64
    src, exe, out = tmp_path / "wide.cpp", tmp_path / "wide", tmp_path / "out.bin"
    src.write_text(DRIVER)
    libdir = os.path.join(ROOT, "fastllm_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", str(src), "-o", str(exe), "-I", os.path.join(ROOT, "host"), "-L", libdir,
                           "-lfastllm_b200", f"-Wl,-rpath,{libdir}"])
    sents = _sentences(26, cfg.vocab_size, [7, 140, 1, 128, 33])
    args = [str(v) for v in (cfg.hidden_size, cfg.num_attention_heads, cfg.num_hidden_layers, cfg.intermediate_size,
                             cfg.max_position_embeddings, cfg.vocab_size)]
    for i, s in enumerate(sents):
        args += (["/"] if i else []) + [str(int(x)) for x in s]
    r = subprocess.run([str(exe), str(out)] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.fromfile(out, dtype=np.float32).reshape(len(sents), -1)
    assert np.array_equal(got, _product(cfg, None, random_seed=0, std=0.02).embed_packed(sents))
