"""CPU: the streamed EVAL metrics (oracle/metrics.py, trainers/model_utils.py finish_* / combine_metric_states) against the
host get_binary_metrics / get_regression_metrics, their invariance under any split into batches and ranks, closed-form
precision / recall / accuracy_baseline, and the dfm_metric_state layout of the header and the ctypes binding."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import metrics as om
from recommender_tensorflow_b200 import _lib
from recommender_tensorflow_b200.trainers.model_utils import (combine_metric_states, finish_binary_metrics, finish_metrics,
                                                              finish_regression_metrics, get_binary_metrics,
                                                              get_regression_metrics)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN_KEYS = {"accuracy", "accuracy_baseline", "auc", "auc_precision_recall", "average_loss", "loss", "label/mean",
            "precision", "prediction/mean", "recall"}


def clear_logits(n, rng, scale=3.0):
    """logits whose p keeps at least 1e-5 away from every threshold and from 0.5, in float32 and float64 alike"""
    th = om.thresholds().astype(np.float64)
    z = rng.normal(0, scale, size=4 * n).astype(np.float32)
    p = 1.0 / (1.0 + np.exp(-z.astype(np.float64)))
    gap = np.min(np.abs(p[:, None] - th[None, :]), axis=1)
    keep = (gap > 1e-5) & (np.abs(z) > 1e-4)
    z = z[keep][:n]
    assert z.size == n
    return z


def batch(n, rng, weighted=False, head="logistic"):
    z = clear_logits(n, rng)
    y = (rng.random(n) < 0.4).astype(np.float32) if head == "logistic" else rng.normal(3, 1, n).astype(np.float32)
    w = None
    if weighted:
        w = rng.choice([0.0, 0.5, 1.0, 2.25, 3.0, -0.75], size=n).astype(np.float32)
    return z, y, w


def close(a, b, rel=1e-12, abs_=1e-12):
    assert set(a) == set(b), (sorted(a), sorted(b))
    for k in a:
        assert abs(a[k] - b[k]) <= abs_ + rel * abs(b[k]), (k, a[k], b[k])


@pytest.mark.parametrize("weighted", [False, True])
def test_one_batch_equals_host_binary(weighted):
    rng = np.random.default_rng(1)
    z, y, w = batch(5000, rng, weighted)
    got = finish_binary_metrics(om.batch_state(z, y, w))
    want = get_binary_metrics(y, z, w)
    close(got, want, abs_=1e-10)
    assert set(got) == BIN_KEYS


@pytest.mark.parametrize("weighted", [False, True])
def test_one_batch_equals_host_regression(weighted):
    rng = np.random.default_rng(2)
    z, y, w = batch(3000, rng, weighted, head="squared")
    close(finish_regression_metrics(om.batch_state(z, y, w, head="squared")), get_regression_metrics(y, z, w))


@pytest.mark.parametrize("head", ["logistic", "squared"])
@pytest.mark.parametrize("weighted", [False, True])
def test_split_into_batches_and_ranks(head, weighted):
    rng = np.random.default_rng(3)
    z, y, w = batch(4097, rng, weighted, head)
    whole = om.batch_state(z, y, w, head)
    cuts = np.sort(rng.choice(np.arange(1, z.size), size=6, replace=False))
    parts = np.split(np.arange(z.size), cuts)
    streamed = om.stream_state([(z[i], y[i], None if w is None else w[i]) for i in parts], head, weighted)
    # ranks: every rank streams its own batches, then the states are combined in rank order
    ranks = [om.stream_state([(z[i], y[i], None if w is None else w[i]) for i in parts[r::3]], head, weighted) for r in range(3)]
    combined = combine_metric_states(ranks)
    for s in (streamed, combined):
        for k in ("n", "bin_count", "cls"):
            assert np.array_equal(s[k], whole[k]), k
        for k in ("bin_weight", "w_cls", "sums"):
            scale = np.abs(whole[k]) + np.abs(np.asarray(whole["sums"][0])) + 1.0
            assert np.all(np.abs(s[k] - whole[k]) <= 1e-12 * scale * 4), k
        close(finish_metrics(s), finish_metrics(whole), rel=1e-11, abs_=1e-11)


def test_combine_is_rank_ordered_and_checks_heads():
    rng = np.random.default_rng(4)
    states = [om.batch_state(*batch(100, rng, True)) for _ in range(3)]
    c = combine_metric_states(states)
    assert np.array_equal(c["sums"], (states[0]["sums"] + states[1]["sums"]) + states[2]["sums"])
    with pytest.raises(ValueError):
        combine_metric_states([states[0], om.empty_state("squared", True)])
    with pytest.raises(ValueError):
        finish_regression_metrics(states[0])


def test_closed_form_precision_recall_baseline():
    # z > 0 is the predicted class: 3 tp, 1 fp, 2 fn, 2 tn
    z = np.array([2, 1, 3, 0.5, -1, -2, -3, -0.5], np.float32)
    y = np.array([1, 1, 1, 0, 1, 1, 0, 0], np.float32)
    for m in (get_binary_metrics(y, z), finish_binary_metrics(om.batch_state(z, y))):
        assert m["precision"] == 3 / 4 and m["recall"] == 3 / 5
        assert m["accuracy"] == 5 / 8 and m["accuracy_baseline"] == 5 / 8
    # weighted: tp 2 + 1, fp 4, fn 0.5
    w = np.array([2, 1, 0, 4, 0.5, 0, 0, 0], np.float32)
    for m in (get_binary_metrics(y, z, w), finish_binary_metrics(om.batch_state(z, y, w))):
        assert m["precision"] == pytest.approx(3 / 7, rel=1e-15) and m["recall"] == pytest.approx(3 / 3.5, rel=1e-15)
        assert m["accuracy_baseline"] == pytest.approx(max(3.5 / 7.5, 4 / 7.5), rel=1e-15)
    # nothing predicted positive: tp + fp = 0 -> precision 0 (metrics_impl _safe_div), recall 0 / 1
    zn, yn = np.array([-1, -2, -3], np.float32), np.array([1, 0, 0], np.float32)
    for m in (get_binary_metrics(yn, zn), finish_binary_metrics(om.batch_state(zn, yn))):
        assert m["precision"] == 0.0 and m["recall"] == 0.0 and m["accuracy_baseline"] == 1 - 1 / 3
    # no positives: tp + fn = 0 -> recall 0
    zp, yp = np.array([1, 2], np.float32), np.array([0, 0], np.float32)
    for m in (get_binary_metrics(yp, zp), finish_binary_metrics(om.batch_state(zp, yp))):
        assert m["precision"] == 0.0 and m["recall"] == 0.0 and m["accuracy_baseline"] == 1.0


def test_new_host_keys_follow_their_definitions():
    rng = np.random.default_rng(5)
    z, y, w = batch(2000, rng, True)
    for ww in (None, w):
        m = get_binary_metrics(y, z, ww)
        wd = np.ones(z.size) if ww is None else ww.astype(np.float64)
        pred, pos = z > 0, y > 0.5
        tp, fp, fn = wd[pred & pos].sum(), wd[pred & ~pos].sum(), wd[~pred & pos].sum()
        assert m["precision"] == pytest.approx(tp / (tp + fp), rel=1e-14)
        assert m["recall"] == pytest.approx(tp / (tp + fn), rel=1e-14)
        lm = (wd * y).sum() / wd.sum()
        assert m["accuracy_baseline"] == pytest.approx(max(lm, 1 - lm), rel=1e-14)


def test_thresholds_and_bins():
    th = om.thresholds()
    assert th.dtype == np.float32 and th.size == 200
    assert th[0] == np.float32(-1e-7) and th[-1] == np.float32(1 + 1e-7) and th[-1] > 1
    assert np.all(np.diff(th) > 0)
    assert th[100] == np.float32(100 / 199)
    # bin = number of thresholds strictly below p
    s = om.batch_state(np.array([0.0], np.float32), np.array([1.0], np.float32))
    p = om.prob32(np.float32(0.0))
    assert s["bin_count"][1].argmax() == int((th < p).sum())
    assert s["cls"][2] == 1          # z = 0 is class 0: a false negative


def test_near_threshold_flags_only_boundary_samples():
    th = om.thresholds()
    t = th[50:53].astype(np.float64)
    z_on = np.log(t / (1 - t)).astype(np.float32)                      # p within a few ulps of thresholds 50..52
    assert om.near_threshold(z_on).all()
    assert not om.near_threshold(clear_logits(1000, np.random.default_rng(6))).any()


def test_state_layout_header_and_ctypes():
    src = open(os.path.join(ROOT, "include", "deepfm_b200.h")).read()
    assert re.search(r"#define DFM_METRIC_BINS 201\b", src)
    assert _lib.METRIC_BINS == om.BINS == 201
    S = _lib.MetricState
    assert ctypes.sizeof(S) == 8 * (1 + 2 * 201 + 4 + 2 * 201 + 4 + 4)
    assert S.bin_weight.offset == 8 * (1 + 2 * 201 + 4)
    assert S.sum_wloss.offset == ctypes.sizeof(S) - 8


def test_abi_rejects_without_gpu():
    lib = _lib.load()
    st = _lib.MetricState()
    assert lib.dfm_metrics_reset(None, None) == -1
    assert lib.dfm_metrics_accumulate(None, None, None, None, 4, None) == -1
    assert lib.dfm_evaluate(None, None, None) == -1
    assert lib.dfm_evaluate_host(None, None) == -1
    assert lib.dfm_metrics_read(None, ctypes.byref(st), None) == -1
