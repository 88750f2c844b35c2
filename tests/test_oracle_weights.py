"""CPU: per-example weights (weight_column) in the oracle's loss and gradients, the weighted EVAL metrics, the weight
feature's checks and the C ABI layout of the new fields."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle.deepfm import OracleDeepFM, default_opt, init_weights
from recommender_tensorflow_b200 import _lib
from recommender_tensorflow_b200 import feature_column as fc
from recommender_tensorflow_b200.trainers.model_utils import get_binary_metrics, get_weights
from tests.weighted_oracle import WeightedOracleDeepFM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAT = [dict(name="a", kind="identity", dtype="int32", num_buckets=5),
       dict(name="b", kind="identity", dtype="int32", num_buckets=3),
       dict(name="c", kind="identity", dtype="int32", num_buckets=7)]


def _cfg(**kw):
    cfg = dict(cat=CAT, num=["x0", "x1"], k=4, hidden=[8, 6], use_linear=True, use_mf=True, use_dnn=True,
               loss_reduction="mean", opt_deep=default_opt(), opt_linear=default_opt())
    cfg.update(kw)
    return cfg


def _data(B=16, seed=0):
    rng = np.random.default_rng(seed)
    ids = np.stack([rng.integers(-1, 5, B), rng.integers(0, 3, B), rng.integers(0, 7, B)], 1).astype(np.int32)
    x = rng.standard_normal((B, 2)).astype(np.float32)
    y = (rng.random(B) < 0.4).astype(np.float32)
    return ids, x, y


def _pair(cfg, seed=3, dtype=torch.float32):
    """(unweighted oracle, weighted oracle) from the same initial weights"""
    w = init_weights(cfg, seed)
    w["lin"] = np.random.default_rng(seed).standard_normal(w["lin"].shape).astype(np.float32) * 0.1
    return OracleDeepFM(cfg, w, dtype=dtype), WeightedOracleDeepFM(cfg, w, dtype=dtype)


@pytest.mark.parametrize("red", ["mean", "sum"])
def test_all_ones_weights_are_the_unweighted_step(red):
    a, b = _pair(_cfg(loss_reduction=red))
    for step in range(3):
        ids, x, y = _data(seed=step)
        la, za = a.train_step(ids, x, y)
        lb, zb = b.train_step(ids, x, y, np.ones(len(y), np.float32))
        assert la == lb and np.array_equal(za, zb)
    sa, sb = a.state(), b.state()
    for n in sa:
        assert np.array_equal(sa[n], sb[n]), n


@pytest.mark.parametrize("opt", ["Adam", "Adagrad", "SGD"])
def test_sum_integer_weights_equal_repeated_rows(opt):
    """SUM reduction: weighting sample b by the integer w_b is the step on a batch that holds it w_b times (w_b = 0:
    the sample is dropped).  Equal up to float64 reassociation."""
    cfg = _cfg(loss_reduction="sum", opt_deep=default_opt(opt, 0.01), opt_linear=default_opt(opt, 0.01))
    b, a = _pair(cfg, dtype=torch.float64)
    rng = np.random.default_rng(7)
    for step in range(3):
        ids, x, y = _data(seed=10 + step)
        w = rng.integers(0, 4, len(y)).astype(np.float32)
        w[0] = 0.0
        rep = np.repeat(np.arange(len(y)), w.astype(int))
        la, _ = a.train_step(ids, x, y, w)
        lb, _ = b.train_step(ids[rep], x[rep], y[rep])
        assert abs(la - lb) <= 1e-12 * max(1.0, abs(lb))
    sa, sb = a.state(), b.state()
    for n in sa:
        np.testing.assert_allclose(sa[n], sb[n], rtol=1e-10, atol=1e-13, err_msg=n)


def test_mean_divides_by_batch_size_not_weight_sum():
    """SUM_OVER_BATCH_SIZE (contrib head): loss = sum(w l) / B and dz = w (sigmoid(z) - y) / B."""
    _, a = _pair(_cfg(), dtype=torch.float64)
    ids, x, y = _data(B=12, seed=4)
    w = np.linspace(0.0, 3.0, 12).astype(np.float32)
    loss, z, g = a.grads(ids, x, y, w)
    lv = a.loss_vec(z, torch.as_tensor(y, dtype=torch.float64))
    wt = torch.as_tensor(w, dtype=torch.float64)
    assert abs(float(loss) - float((lv * wt).sum() / 12)) < 1e-15
    dz = (torch.sigmoid(z) - torch.as_tensor(y, dtype=torch.float64)) / 12 * wt
    assert torch.allclose(g["bias"], dz.sum().reshape(1), rtol=0, atol=1e-15)
    assert torch.allclose(g["bo"], dz.sum().reshape(1), rtol=0, atol=1e-15)


def test_weighted_backward_matches_autograd_fp64():
    for red in ("mean", "sum"):
        cfg = _cfg(loss_reduction=red)
        _, m = _pair(cfg, dtype=torch.float64)
        ids, x, y = _data(seed=5)
        w = np.random.default_rng(5).uniform(-0.5, 3.0, len(y)).astype(np.float32)    # TF accepts negative weights
        loss, z, g = m.grads(ids, x, y, w)
        leaves = {n: v.w.clone().requires_grad_(True) for n, v in m.vars.items()}
        for n, v in m.vars.items():
            v.w = leaves[n]
        lv = m.loss_vec(m.forward(ids, x), torch.as_tensor(y, dtype=torch.float64)) * torch.as_tensor(w, dtype=torch.float64)
        (lv.mean() if red == "mean" else lv.sum()).backward()
        for n, gr in g.items():
            if isinstance(gr, tuple):
                dense = torch.zeros_like(leaves[n])
                dense.index_add_(0, gr[1], gr[2])
                gr = dense
            assert torch.allclose(gr.reshape(leaves[n].shape), leaves[n].grad, atol=1e-12), n


# ---------------------------------------------------------------------------------------------------- metrics
def _auc_brute(y, p, w, curve):
    """tf.metrics.auc with weights, restated with Python loops over the 200 thresholds"""
    eps = 1e-7
    th = [0.0 - eps] + [i / 199.0 for i in range(1, 199)] + [1.0 + eps]
    xs, ys = [], []
    for t in th:
        tp = fp = fn = tn = 0.0
        for yi, pi, wi in zip(y, p, w):
            if pi > t:
                tp, fp = (tp + wi, fp) if yi > 0.5 else (tp, fp + wi)
            else:
                fn, tn = (fn + wi, tn) if yi > 0.5 else (fn, tn + wi)
        if curve == "ROC":
            xs.append(fp / (fp + tn + eps)); ys.append((tp + eps) / (tp + fn + eps))
        else:
            xs.append((tp + eps) / (tp + fn + eps)); ys.append((tp + eps) / (tp + fp + eps))
    return sum((xs[i] - xs[i + 1]) * (ys[i] + ys[i + 1]) / 2.0 for i in range(len(th) - 1))


def test_weighted_metrics_against_restatement():
    rng = np.random.default_rng(1)
    n = 300
    y = (rng.random(n) < 0.35).astype(np.float32)
    z = rng.normal(0.8 * y - 0.4, 1.2)
    w = rng.uniform(0.0, 3.0, n).astype(np.float32)
    w[rng.random(n) < 0.1] = 0.0
    m = get_binary_metrics(y, z, w)
    wd = w.astype(np.float64)
    p = [1.0 / (1.0 + np.exp(-v)) for v in z]
    ls = [max(v, 0.0) - v * yi + np.log1p(np.exp(-abs(v))) for v, yi in zip(z, y)]
    sw = float(sum(wd))
    assert abs(m["average_loss"] - sum(wi * li for wi, li in zip(wd, ls)) / sw) < 1e-12
    assert abs(m["loss"] - sum(wi * li for wi, li in zip(wd, ls))) < 1e-9
    assert abs(m["accuracy"] - sum(wi for wi, pi, yi in zip(wd, p, y) if (pi > 0.5) == (yi > 0.5)) / sw) < 1e-12
    assert abs(m["label/mean"] - sum(wi * yi for wi, yi in zip(wd, y)) / sw) < 1e-12
    assert abs(m["prediction/mean"] - sum(wi * pi for wi, pi in zip(wd, p)) / sw) < 1e-12
    assert abs(m["auc"] - _auc_brute(y, p, wd, "ROC")) < 1e-9
    assert abs(m["auc_precision_recall"] - _auc_brute(y, p, wd, "PR")) < 1e-9


def test_weighted_metrics_integer_weights_repeat_rows_and_unweighted_unchanged():
    rng = np.random.default_rng(2)
    y = (rng.random(200) < 0.4).astype(np.float32)
    z = rng.normal(0.0, 1.5, 200)
    w = rng.integers(0, 4, 200).astype(np.float32)
    rep = np.repeat(np.arange(200), w.astype(int))
    mw, mr = get_binary_metrics(y, z, w), get_binary_metrics(y[rep], z[rep])
    for k in mr:
        assert abs(mw[k] - mr[k]) <= 1e-9 * max(1.0, abs(mr[k])), k
    # weights=None is the unweighted code path, and all-ones weights give the same numbers
    base = get_binary_metrics(y, z)
    assert get_binary_metrics(y, z, None) == base
    ones = get_binary_metrics(y, z, np.ones(200, np.float32))
    for k in base:
        assert abs(ones[k] - base[k]) <= 1e-12 * max(1.0, abs(base[k])), k


def test_weight_feature_lookup_and_checks():
    feats = {"w": np.array([1, 0, 2], np.int32), "x": np.zeros(3)}
    got = get_weights(feats, "w", 3)
    assert got.dtype == np.float32 and got.tolist() == [1.0, 0.0, 2.0]          # tf.to_float of an int feature
    assert get_weights(feats, fc.numeric_column("w"), 3).tolist() == [1.0, 0.0, 2.0]
    assert get_weights({"w": np.array([[0.5], [-1.0], [2.0]])}, "w", 3).tolist() == [0.5, -1.0, 2.0]
    assert get_weights(feats, None, 3) is None
    with pytest.raises(KeyError):
        get_weights(feats, "missing", 3)
    with pytest.raises(ValueError):
        get_weights(feats, "w", 4)
    with pytest.raises(ValueError):
        get_weights({"w": np.ones((3, 2))}, "w", 3)
    with pytest.raises(TypeError):
        get_weights(feats, 3, 3)


# ---------------------------------------------------------------------------------------------------- ABI
def _struct_fields(name):
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "deepfm_b200.h")).read(), flags=re.S)
    body = re.search(r"typedef struct \{([^{}]*)\} %s;" % name, src).group(1)
    names = []
    for decl in (d.strip() for d in body.split(";")):
        if decl:      # "int32_t use_linear, use_mf, use_dnn" declares three fields
            names += [re.findall(r"(\w+)\s*$", part.strip())[0] for part in decl.split(",")]
    return names


def test_header_and_ctypes_layouts_agree():
    for cname, py in (("dfm_config", _lib.Config), ("dfm_raw_batch", _lib.RawBatch)):
        assert _struct_fields(cname) == [f[0] for f in py._fields_], cname
    assert _struct_fields("dfm_config")[-1] == "weighted" and _struct_fields("dfm_raw_batch")[-1] == "weights"
    assert _lib.RawBatch.weights.offset == _lib.RawBatch.labels.offset + ctypes.sizeof(ctypes.c_void_p)
    assert ctypes.sizeof(_lib.Config()) % 8 == 0 and _lib.Config().weighted == 0    # a zeroed struct stays unweighted
