"""fl_embed_packed on the GPU: sentences of different lengths in ONE encoder pass, each row bit-identical to the sentence embedded
alone (fl_embed of [1, t]), against the oracle at the existing BERT bars, with the uniform fl_embed path unchanged around it."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

from oracle import bert as obert
from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COS_TOL = 0.999
LENGTHS = [1, 2, 15, 16, 17, 63, 127, 128, 129, 255, 256, 257, 383, 511, 512]


def _cos(a, b):
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


def _product(cfg, w, **kw):
    from fastllm_b200 import models
    pc = models.BertConfig(cfg.hidden_size, cfg.num_attention_heads, cfg.num_hidden_layers, cfg.intermediate_size,
                           cfg.max_position_embeddings, cfg.layer_norm_eps, cfg.vocab_size)
    return models.MiniLMModel(pc, w, 0, **kw)


def _sentences(seed, vocab, lengths):
    return [synth.token_ids(seed * 1000 + i, vocab, (n,)) for i, n in enumerate(lengths)]


def _lone(m, sentences):
    return np.concatenate([m.embed_ids(s[None]) for s in sentences])


@pytest.fixture(scope="module")
def minilm():
    return _product(obert.MINILM_L6, None, random_seed=0, std=0.02)


def test_packed_rows_equal_lone_sentences_bitwise(minilm):
    cfg = obert.MINILM_L6
    lengths = list(np.random.RandomState(1).permutation(LENGTHS))
    sents = _sentences(1, cfg.vocab_size, lengths)
    got = minilm.embed_packed(sents)
    want = _lone(minilm, sents)
    for i, n in enumerate(lengths):
        assert np.array_equal(got[i], want[i]), (n, np.abs(got[i] - want[i]).max())
    # padding to the longest sentence with a pooling mask is NOT the same computation: the pad tokens are attended to
    t = max(lengths)
    ids = np.zeros((len(sents), t), dtype=np.uint32)
    mask = np.zeros((len(sents), t), dtype=np.uint32)
    for i, s in enumerate(sents):
        ids[i, :len(s)], mask[i, :len(s)] = s, 1
    padded = minilm.embed_ids(ids, mask)
    for i, n in enumerate(lengths):
        if n <= 128:
            assert np.abs(padded[i] - want[i]).max() > 1e-3, n


@pytest.mark.parametrize("case", ["tiny_golden", "minilm_l6"])
def test_packed_matches_oracle(case, golden_dir):
    if case == "tiny_golden":
        g = np.load(f"{golden_dir}/bert_tiny.npz")
        cfg = obert.BertConfig(128, 4, 2, 256, 64, 1e-12, 200)
        w = obert.synth_weights(cfg, int(g["seed"]), float(g["std"]))
        for k in g.files:
            if k.startswith("w:"):
                w[k[2:]] = g[k]
        lengths = [33, 1, 64, 7, 16, 2, 50]
    else:
        cfg = obert.MINILM_L6
        w = obert.synth_weights(cfg, 0, 0.02)
        lengths = [129, 5, 512, 128, 17, 300]
    sents = _sentences(2, cfg.vocab_size, lengths)
    got = _product(cfg, w).embed_packed(sents)
    o = obert.MiniLM(cfg, w)
    want = np.concatenate([o.embed_ids(s[None]) for s in sents])
    cos = _cos(got, want)
    print(f"{case}: min cosine {cos.min():.6f}, max-abs {np.abs(got - want).max():.3e}")
    assert cos.min() >= COS_TOL and np.abs(got - want).max() <= 2e-2


def test_packed_equals_grouped_batches_and_follows_request_order(minilm):
    cfg = obert.MINILM_L6
    lengths = np.random.RandomState(3).randint(1, 129, size=256)
    sents = _sentences(3, cfg.vocab_size, lengths)
    got = minilm.embed_packed(sents)
    assert np.array_equal(got, minilm.embed_many(sents))
    assert np.array_equal(minilm.embed_packed(sents[::-1]), got[::-1])


def test_workspace_reuse_after_a_larger_packed_call(minilm):
    cfg = obert.MINILM_L6
    ids = synth.token_ids(4, cfg.vocab_size, (16, 128))
    first = minilm.embed_ids(ids)
    minilm.embed_packed(_sentences(4, cfg.vocab_size, [512] * 40 + [3, 77]))
    assert np.array_equal(minilm.embed_ids(ids), first)


def test_launch_counts_and_profile_tags(minilm):
    from fastllm_b200 import models
    cfg = obert.MINILM_L6

    def launches(f):
        n0 = models.launch_count()
        f()
        return models.launch_count() - n0

    ids = synth.token_ids(5, cfg.vocab_size, (8, 128))
    assert launches(lambda: minilm.embed_ids(ids)) == 44
    short = _sentences(5, cfg.vocab_size, [3, 128, 40, 77])
    mixed = _sentences(6, cfg.vocab_size, [3, 300, 128, 129, 40])
    assert launches(lambda: minilm.embed_packed(short)) == 44
    assert launches(lambda: minilm.embed_packed(mixed)) == 50          # one more attention launch per layer
    models.prof_begin()
    minilm.embed_packed(mixed)
    prof = models.prof_end()
    assert prof and all(p["kernel"].startswith("bert_") for p in prof), prof
    assert sum(p["launches"] for p in prof) == 50


def test_packed_errors_leave_the_model_usable(minilm):
    from fastllm_b200 import FastllmError, _lib
    from helpers import golden_weights, product_model
    cfg = obert.MINILM_L6
    lib = _lib.load()
    ok = _sentences(7, cfg.vocab_size, [9, 200])
    want = minilm.embed_packed(ok)
    out = np.empty((4, cfg.hidden_size), dtype=np.float32)

    def call(h, ids, lengths, n, o=out):
        ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        return lib.fl_embed_packed(h, ptr(ids), ptr(lengths), n, ptr(o))

    ids = np.ones(16, dtype=np.uint32)
    llama, _ = product_model(*golden_weights("llama_gqa8")[:2])
    bad = [
        (minilm.dev.h, None, np.array([16], np.int32), 1),
        (minilm.dev.h, ids, None, 1),
        (None, ids, np.array([16], np.int32), 1),
        (minilm.dev.h, ids, np.array([16], np.int32), 1, None),
        (minilm.dev.h, ids, np.array([16], np.int32), 0),
        (minilm.dev.h, ids, np.array([8, 0, 8], np.int32), 3),
        (minilm.dev.h, np.ones(cfg.max_position_embeddings + 1, np.uint32), np.array([cfg.max_position_embeddings + 1], np.int32), 1),
        (minilm.dev.h, np.full(16, cfg.vocab_size, np.uint32), np.array([16], np.int32), 1),
        (llama.dev.h, ids, np.array([16], np.int32), 1),
        # 2,800 x 512 tokens x max(3 x 384, 1536) > 2^31: rejected on the host before any device work
        (minilm.dev.h, np.ones(2800 * 512, np.uint32), np.full(2800, 512, np.int32), 2800),
    ]
    for args in bad:
        assert call(*args) == -1, args[3:]                          # FL_ERR_INVALID
        assert np.array_equal(minilm.embed_packed(ok), want)
    with pytest.raises(FastllmError):
        minilm.embed_packed([np.array([], dtype=np.uint32)])
    assert np.array_equal(minilm.embed_packed(ok), want)


def test_two_threads_alternating_uniform_and_packed_calls(minilm):
    cfg = obert.MINILM_L6
    ids = synth.token_ids(8, cfg.vocab_size, (32, 64))
    sents = _sentences(8, cfg.vocab_size, list(np.random.RandomState(8).randint(1, 400, size=48)))
    want_u, want_p = minilm.embed_ids(ids), minilm.embed_packed(sents)
    got = {"u": [], "p": []}
    errs = []

    def run(key, f):
        try:
            for _ in range(8):
                got[key].append(f())
        except Exception as e:          # noqa: BLE001 -- reported by the main thread
            errs.append(e)

    th = [threading.Thread(target=run, args=("u", lambda: minilm.embed_ids(ids))),
          threading.Thread(target=run, args=("p", lambda: minilm.embed_packed(sents)))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    assert all(np.array_equal(g, want_u) for g in got["u"]) and len(got["u"]) == 8
    assert all(np.array_equal(g, want_p) for g in got["p"]) and len(got["p"]) == 8


DRIVER = r"""
#include <cstdio>
#include <cstdlib>
#include "fastllm_host.hpp"
using namespace fastllm;
// argv: out.bin then the sentences' ids, sentences separated by "/"; MiniLM-L6 shapes, synthetic weights (seed 0, std 0.02)
int main(int argc, char** argv) {
    check(fl_init(0));
    fl_config c{};
    c.arch = FL_ARCH_BERT; c.hidden_size = 384; c.intermediate_size = 1536; c.vocab_size = 30522; c.num_hidden_layers = 6;
    c.num_attention_heads = 12; c.num_key_value_heads = 12; c.max_position_embeddings = 512; c.norm_eps = 1e-12f; c.tp_size = 1;
    auto dev = std::make_shared<DeviceModel>(c);
    check(fl_model_random_init(dev->h, 0, 0.02f));
    check(fl_model_finalize(dev->h));
    MiniLMModel m{dev};
    std::vector<std::vector<uint32_t>> sents(1);
    for (int i = 2; i < argc; ++i) {
        if (std::string(argv[i]) == "/") sents.emplace_back();
        else sents.back().push_back((uint32_t)std::strtoul(argv[i], nullptr, 10));
    }
    const auto rows = m.embed_packed(sents);
    if (!m.embed_packed({}).empty()) return 3;
    FILE* f = std::fopen(argv[1], "wb");
    for (const auto& r : rows) std::fwrite(r.data(), 4, r.size(), f);
    std::fclose(f);
    return 0;
}
"""


def test_cpp_mirror_embed_packed_equals_python(minilm, tmp_path):
    src, exe, out = tmp_path / "packed.cpp", tmp_path / "packed", tmp_path / "out.bin"
    src.write_text(DRIVER)
    libdir = os.path.join(ROOT, "fastllm_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", str(src), "-o", str(exe), "-I", os.path.join(ROOT, "host"), "-L", libdir,
                           "-lfastllm_b200", f"-Wl,-rpath,{libdir}"])
    sents = _sentences(9, obert.MINILM_L6.vocab_size, [7, 140, 1, 128, 33])
    args = []
    for i, s in enumerate(sents):
        args += (["/"] if i else []) + [str(int(x)) for x in s]
    r = subprocess.run([str(exe), str(out)] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.fromfile(out, dtype=np.float32).reshape(len(sents), -1)
    assert np.array_equal(got, minilm.embed_packed(sents))
