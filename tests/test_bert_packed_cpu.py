"""MiniLMModel.embed_packed host logic on CPU against a stand-in library: the sentences travel as ONE fl_embed_packed call (ids
concatenated without padding, one length per sentence), rows come back in request order, and an empty request never reaches the
library."""
import ctypes as C

import numpy as np

from fastllm_b200 import models

H = 8


class _FakeLib:
    """fl_embed_packed stand-in: records what it was handed and writes row i = a function of sentence i's ids."""

    def __init__(self):
        self.calls = []

    def fl_embed_packed(self, h, ids, lengths, n, out):
        lens = np.ctypeslib.as_array(C.cast(lengths, C.POINTER(C.c_int32)), (n,)).copy()
        flat = np.ctypeslib.as_array(C.cast(ids, C.POINTER(C.c_uint32)), (int(lens.sum()),)).copy()
        self.calls.append((h, flat, lens, n))
        rows = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_float)), (n, H))
        o = 0
        for i, t in enumerate(lens):
            rows[i] = _row(flat[o:o + t])
            o += t
        return 0


def _row(ids):
    return np.cos(np.arange(H) * (1 + int(np.asarray(ids, dtype=np.int64).sum()) + 7 * len(ids))).astype(np.float32)


def _model():
    m = models.MiniLMModel.__new__(models.MiniLMModel)        # host logic only: no device model behind it
    m.config = models.BertConfig(hidden_size=H)
    m.dev = type("Dev", (), {})()
    m.dev.h, m.dev.lib = "handle", _FakeLib()
    return m


def test_embed_packed_is_one_call_with_concatenated_ids_and_lengths():
    m = _model()
    rs = np.random.RandomState(0)
    sentences = [list(map(int, rs.randint(0, 1000, size=n))) for n in [5, 1, 130, 17, 5]]
    sentences[2] = np.asarray(sentences[2], dtype=np.int64)          # any 1-D integer sequence
    got = m.embed_packed(sentences)
    assert len(m.dev.lib.calls) == 1
    h, flat, lens, n = m.dev.lib.calls[0]
    assert h == "handle" and n == 5
    assert lens.tolist() == [5, 1, 130, 17, 5]
    assert np.array_equal(flat, np.concatenate([np.asarray(s, dtype=np.uint32) for s in sentences]))
    assert got.dtype == np.float32 and got.shape == (5, H)
    assert np.array_equal(got, np.stack([_row(s) for s in sentences]))      # request order


def test_embed_packed_empty_request_does_not_call_the_library():
    m = _model()
    out = m.embed_packed([])
    assert out.shape == (0, H) and out.dtype == np.float32
    assert m.dev.lib.calls == []
