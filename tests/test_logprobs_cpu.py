"""Scoring without a GPU: the all-position reference the GPU tests compare with, and Model.loglikelihood's bookkeeping."""
import numpy as np
import pytest

from oracle import causal_lm as ocl
from oracle import synth

from helpers import TINY
from logprobs_ref import log_softmax64, logits_all


@pytest.mark.parametrize("name", sorted(TINY))
def test_all_positions_last_row_is_the_oracle_forward(name):
    cfg = TINY[name]
    w = ocl.synth_weights(cfg, 3, 0.05)
    ids = synth.token_ids(5, cfg.vocab_size, (2, 11))
    want = ocl.CausalLM(cfg, w).forward(ids, 0)
    got = logits_all(ocl.CausalLM(cfg, w), ids, 0)
    assert got.shape == (2, 11, cfg.vocab_size)
    assert np.array_equal(got[:, -1], want)
    # and an earlier position is the last position of the shorter call (the layers' products differ in shape: f32 rounding)
    assert np.abs(got[:, 4] - ocl.CausalLM(cfg, w).forward(ids[:, :5], 0)).max() <= 1e-5
    # the one-product form agrees to f32 rounding
    assert np.abs(logits_all(ocl.CausalLM(cfg, w), ids, 0, per_position=False) - got).max() <= 1e-5


def test_log_softmax64_is_normalised():
    z = np.array([[1.0, 2.0, 3.0], [-1e4, 0.0, 0.0]], dtype=np.float32)
    lp = log_softmax64(z)
    assert np.allclose(np.exp(lp).sum(-1), 1.0)
    assert lp[1, 0] < -9e3 and np.isclose(lp[1, 1], np.log(0.5))


class _StubAdapter:
    """stands in for a causal-LM adapter: logprobs() returns fixed arrays and records its arguments"""

    def __init__(self, lp, am):
        self.lp, self.am, self.calls = lp, am, []

    def logprobs(self, ids, targets):
        self.calls.append((np.array(ids), np.array(targets)))
        return self.lp.copy(), self.am.copy()


def _stub_model(lp, am):
    from fastllm_b200 import models
    return models.Model(_StubAdapter(np.asarray(lp, dtype=np.float32)[None], np.asarray(am, dtype=np.uint32)[None]), None)


def test_loglikelihood_shifts_targets_and_sums_the_continuation():
    # context [5, 6, 7], continuation [8, 9]: positions 2 and 3 predict 8 and 9
    lp = [-1.0, -2.0, -0.25, -0.5, -7.0]
    am = [6, 7, 8, 9, 1]
    m = _stub_model(lp, am)
    total, greedy = m.loglikelihood([5, 6, 7], [8, 9])
    ids, targets = m.model.calls[0]
    assert ids.tolist() == [[5, 6, 7, 8, 9]] and targets.tolist() == [[6, 7, 8, 9, 0]]
    assert total == -0.75 and isinstance(total, float)
    assert greedy is True


def test_loglikelihood_greedy_flag_needs_every_continuation_token():
    lp = [-1.0, -0.125, -0.5, -3.0]
    total, greedy = _stub_model(lp, [2, 3, 4, 0]).loglikelihood([1, 2], [3, 5])      # position 2 picks 4, not 5
    assert total == -0.625 and greedy is False
    # a miss inside the context does not count
    total, greedy = _stub_model(lp, [0, 3, 5, 0]).loglikelihood([1, 2], [3, 5])
    assert greedy is True


def test_loglikelihood_one_token_context():
    total, greedy = _stub_model([-0.5, -9.0], [4, 4]).loglikelihood([3], [4])
    assert total == -0.5 and greedy is True


@pytest.mark.parametrize("ctx,cont", [([], [1]), ([1], []), ([], [])])
def test_loglikelihood_rejects_empty_parts(ctx, cont):
    with pytest.raises(ValueError):
        _stub_model([0.0], [0]).loglikelihood(ctx, cont)
