"""CPU: the squared head (regression) in the oracle's loss and gradients, the regression predictions and EVAL metrics,
the head's argument checks in model_fn / the canned regressors / the engine, and the C ABI fields that select it."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle.deepfm import OracleDeepFM, default_opt, init_weights
from recommender_tensorflow_b200 import _lib
from recommender_tensorflow_b200.csv_reader import CSV_FLOAT32, CSV_INT32, CSV_STRING, CsvConfig
from recommender_tensorflow_b200.trainers.model_utils import get_regression_metrics, get_regression_predictions
from tests.regression_oracle import HeadOracleDeepFM
from tests.weighted_oracle import WeightedOracleDeepFM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAT = [dict(name="a", kind="identity", dtype="int32", num_buckets=5),
       dict(name="b", kind="identity", dtype="int32", num_buckets=3),
       dict(name="c", kind="identity", dtype="int32", num_buckets=7)]
OPTIMIZERS = ["Adam", "Adagrad", "Ftrl", "RMSProp", "SGD"]


def _cfg(**kw):
    cfg = dict(cat=CAT, num=["x0", "x1"], k=4, hidden=[8, 6], use_linear=True, use_mf=True, use_dnn=True,
               loss_reduction="mean", opt_deep=default_opt(), opt_linear=default_opt(), head="squared")
    cfg.update(kw)
    return cfg


def _data(B=16, seed=0):
    """ids, numerics and ratings in 1..5 (the regression label is the rating itself)"""
    rng = np.random.default_rng(seed)
    ids = np.stack([rng.integers(-1, 5, B), rng.integers(0, 3, B), rng.integers(0, 7, B)], 1).astype(np.int32)
    x = rng.standard_normal((B, 2)).astype(np.float32)
    y = rng.integers(1, 6, B).astype(np.float32)
    return ids, x, y


def _init(cfg, seed=3):
    w = init_weights(cfg, seed)
    w["lin"] = np.random.default_rng(seed).standard_normal(w["lin"].shape).astype(np.float32) * 0.1
    return w


# ---------------------------------------------------------------------------------------------------- oracle
@pytest.mark.parametrize("red,act,weighted", [("mean", "relu", False), ("sum", "relu", False), ("mean", "relu", True),
                                              ("sum", "relu", True), ("mean", "tanh", False), ("sum", "identity", True)])
def test_squared_backward_matches_autograd_fp64(red, act, weighted):
    """loss = reduce(w (y - z)^2), reduce = mean over the batch size or sum; every gradient against autograd"""
    cfg = _cfg(loss_reduction=red, activation=act)
    m = HeadOracleDeepFM(cfg, _init(cfg), dtype=torch.float64)
    ids, x, y = _data(seed=5)
    w = np.random.default_rng(5).uniform(-0.5, 3.0, len(y)).astype(np.float32) if weighted else None
    loss, z, g = m.grads(ids, x, y, w)
    leaves = {n: v.w.clone().requires_grad_(True) for n, v in m.vars.items()}
    for n, v in m.vars.items():
        v.w = leaves[n]
    zt = m.forward(ids, x)
    lv = (torch.as_tensor(y, dtype=torch.float64) - zt) ** 2           # squared_difference(labels, logits)
    if weighted:
        lv = lv * torch.as_tensor(w, dtype=torch.float64)
    ref = lv.mean() if red == "mean" else lv.sum()
    ref.backward()
    assert abs(float(loss) - float(ref.detach())) <= 1e-12 * max(1.0, abs(float(ref.detach())))
    for n, gr in g.items():
        if isinstance(gr, tuple):
            dense = torch.zeros_like(leaves[n])
            dense.index_add_(0, gr[1], gr[2])
            gr = dense
        assert torch.allclose(gr.reshape(leaves[n].shape), leaves[n].grad, atol=1e-11), n


@pytest.mark.parametrize("red", ["mean", "sum"])
def test_logistic_head_restatement_is_the_oracle_bit_for_bit(red):
    """head="logistic" through the restated backward (weights given) is OracleDeepFM / WeightedOracleDeepFM exactly:
    the restatement the squared head runs through is pinned to the oracle's own backward"""
    cfg = _cfg(loss_reduction=red, head="logistic")
    w0 = _init(cfg)
    a, b = OracleDeepFM(cfg, w0), HeadOracleDeepFM(cfg, w0)
    c, d = WeightedOracleDeepFM(cfg, w0), HeadOracleDeepFM(cfg, w0)
    rng = np.random.default_rng(9)
    for step in range(3):
        ids, x, y = _data(seed=step)
        y = (y >= 4).astype(np.float32)
        wt = rng.uniform(0.0, 3.0, len(y)).astype(np.float32)
        la, za = a.train_step(ids, x, y)
        lb, zb = b.train_step(ids, x, y, np.ones(len(y), np.float32))
        assert la == lb and np.array_equal(za, zb)
        lc, zc = c.train_step(ids, x, y, wt)
        ld, zd = d.train_step(ids, x, y, wt)
        assert lc == ld and np.array_equal(zc, zd)
    for p, q in ((a, b), (c, d)):
        sp, sq = p.state(), q.state()
        for n in sp:
            assert np.array_equal(sp[n], sq[n]), n


@pytest.mark.parametrize("opt", OPTIMIZERS)
@pytest.mark.parametrize("red", ["mean", "sum"])
def test_squared_steps_every_optimizer_fp32_tracks_fp64(opt, red):
    """three squared-head steps with each optimizer: the float32 oracle stays within float32 rounding of its float64
    twin (the pair the GPU parity tests calibrate their tolerances with), and the loss goes down on a fixed batch"""
    lr = 0.01 if red == "mean" else 0.0005        # SUM over 32 ratings: a plain SGD step at 0.01 diverges
    cfg = _cfg(loss_reduction=red, opt_deep=default_opt(opt, lr), opt_linear=default_opt(opt, lr))
    w0 = _init(cfg)
    o32, o64 = HeadOracleDeepFM(cfg, w0), HeadOracleDeepFM(cfg, w0, dtype=torch.float64)
    ids, x, y = _data(B=32, seed=11)
    losses = []
    for _ in range(3):
        l32, z32 = o32.train_step(ids, x, y)
        l64, z64 = o64.train_step(ids, x, y)
        assert abs(l32 - l64) <= 1e-5 * abs(l64) and np.allclose(z32, z64, rtol=1e-5, atol=1e-5)
        losses.append(l64)
    assert losses[-1] < losses[0], losses
    s32, s64 = o32.state(), o64.state()
    for n in s64:
        np.testing.assert_allclose(s32[n], s64[n], rtol=1e-4, atol=1e-5, err_msg=n)


@pytest.mark.parametrize("opt", OPTIMIZERS)
def test_sum_integer_weights_equal_repeated_rows(opt):
    """SUM: weighting sample b by the integer w_b is the step on a batch that holds it w_b times (0: dropped)"""
    cfg = _cfg(loss_reduction="sum", opt_deep=default_opt(opt, 0.01), opt_linear=default_opt(opt, 0.01))
    w0 = _init(cfg)
    a, b = HeadOracleDeepFM(cfg, w0, dtype=torch.float64), HeadOracleDeepFM(cfg, w0, dtype=torch.float64)
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


def test_mean_scale_and_closed_form_dz():
    """MEAN: loss = sum(w (y - z)^2) / B and dz = 2 (z - y) / B * w (the batch size, not sum(w))"""
    m = HeadOracleDeepFM(_cfg(), _init(_cfg()), dtype=torch.float64)
    ids, x, y = _data(B=12, seed=4)
    w = np.linspace(0.0, 3.0, 12).astype(np.float32)
    loss, z, g = m.grads(ids, x, y, w)
    yt, wt = torch.as_tensor(y, dtype=torch.float64), torch.as_tensor(w, dtype=torch.float64)
    assert abs(float(loss) - float(((yt - z) ** 2 * wt).sum() / 12)) < 1e-13
    dz = 2 * (z - yt) / 12 * wt
    assert torch.allclose(g["bias"], dz.sum().reshape(1), rtol=0, atol=1e-14)
    assert torch.allclose(g["bo"], dz.sum().reshape(1), rtol=0, atol=1e-14)


# ---------------------------------------------------------------------------------------------------- head outputs
def test_regression_predictions_are_the_logits():
    p = get_regression_predictions(np.array([0.5, -2.0, 3.25]))
    assert list(p) == ["predictions"]
    assert p["predictions"].shape == (3, 1) and p["predictions"].dtype == np.float32
    assert p["predictions"][:, 0].tolist() == [0.5, -2.0, 3.25]


def test_regression_metrics_closed_form():
    y = np.array([1.0, 2.0, 4.0, 5.0])
    z = np.array([1.5, 2.0, 3.0, 7.0])            # squared errors 0.25, 0, 1, 4
    m = get_regression_metrics(y, z)
    assert m == {"average_loss": 5.25 / 4, "loss": 5.25, "label/mean": 3.0, "prediction/mean": 13.5 / 4}
    w = np.array([2.0, 0.0, 1.0, 0.5], np.float32)    # sum w = 3.5
    m = get_regression_metrics(y, z, w)
    assert m["loss"] == 0.5 + 1.0 + 2.0
    assert m["average_loss"] == 3.5 / 3.5
    assert m["label/mean"] == (2.0 + 4.0 + 2.5) / 3.5
    assert m["prediction/mean"] == (3.0 + 3.0 + 3.5) / 3.5
    # [B, 1] labels / logits are the same as [B]; all-ones weights give the unweighted numbers
    assert get_regression_metrics(y.reshape(-1, 1), z.reshape(-1, 1)) == get_regression_metrics(y, z)
    assert get_regression_metrics(y, z, np.ones(4)) == get_regression_metrics(y, z)


def test_regression_metrics_integer_weights_repeat_rows_and_shape_checks():
    rng = np.random.default_rng(2)
    y = rng.integers(1, 6, 200).astype(np.float32)
    z = rng.normal(3.0, 1.5, 200)
    w = rng.integers(0, 4, 200).astype(np.float32)
    rep = np.repeat(np.arange(200), w.astype(int))
    mw, mr = get_regression_metrics(y, z, w), get_regression_metrics(y[rep], z[rep])
    for k in mr:
        assert abs(mw[k] - mr[k]) <= 1e-9 * max(1.0, abs(mr[k])), k
    with pytest.raises(ValueError):
        get_regression_metrics(y, z, w[:10])
    with pytest.raises(ValueError):
        get_regression_metrics(np.ones((200, 2)), z)      # label_dimension 2


# ---------------------------------------------------------------------------------------------------- argument checks
def test_model_fn_head_params_are_checked_before_the_engine_exists():
    from recommender_tensorflow_b200.trainers import deep_fm, ml_100k
    cols = ml_100k.get_feature_columns()["linear"]
    feats = {"user_id": np.zeros(2, np.int32)}
    for bad, msg in (({"head": "multi_class"}, "head"), ({"head": "regression", "label_dimension": 2}, "label_dimension"),
                     ({"head": "regression", "inverse_link_fn": np.exp}, "inverse_link_fn"),
                     ({"head": "regression", "loss_fn": lambda y, z: y}, "loss_fn")):
        params = {"categorical_columns": cols, **bad}
        with pytest.raises(ValueError, match=msg):
            deep_fm.model_fn(feats, np.zeros(2, np.float32), ml_100k.ModeKeys.TRAIN, params)
        assert deep_fm._ENGINE_KEY not in params


def test_canned_regressors_reject_label_dimension_and_engine_rejects_unknown_head():
    from recommender_tensorflow_b200.engine import DeepFMEngine
    from recommender_tensorflow_b200.trainers import deep, linear, linear_deep, ml_100k
    fcs = ml_100k.get_feature_columns()
    with pytest.raises(ValueError, match="label_dimension"):
        linear.LinearRegressor(fcs["linear"], label_dimension=2)
    with pytest.raises(ValueError, match="label_dimension"):
        deep.DNNRegressor([16], fcs["deep"], label_dimension=3)
    with pytest.raises(ValueError, match="label_dimension"):
        linear_deep.DNNLinearCombinedRegressor(linear_feature_columns=fcs["linear"], dnn_feature_columns=fcs["deep"],
                                               dnn_hidden_units=[16], label_dimension=2)
    with pytest.raises(ValueError, match="head"):
        DeepFMEngine(fcs["linear"], head="poisson")
    assert linear.LinearRegressor.HEAD == deep.DNNRegressor.HEAD == linear_deep.DNNLinearCombinedRegressor.HEAD == "regression"
    assert linear.LinearClassifier.HEAD == "binary"


def _struct_fields(name):
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "deepfm_b200.h")).read(), flags=re.S)
    body = re.search(r"typedef struct \{([^{}]*)\} %s;" % name, src).group(1)
    names = []
    for decl in (d.strip() for d in body.split(";")):
        if decl:
            names += [re.findall(r"(\w+)\s*$", part.strip())[0] for part in decl.split(",")]
    return names


def test_header_ctypes_layouts_and_zeroed_defaults():
    assert _struct_fields("dfm_config") == [f[0] for f in _lib.Config._fields_]
    assert _struct_fields("dfm_csv_config") == [f[0] for f in CsvConfig._fields_]
    assert _struct_fields("dfm_csv_config")[-1] == "label_raw"
    src = open(os.path.join(ROOT, "include", "deepfm_b200.h")).read()
    heads = dict(re.findall(r"#define DFM_HEAD_(\w+)\s+(\d+)", src))
    assert heads == {"LOGISTIC": "0", "SQUARED": "1"} and _lib.HEADS == {"logistic": 0, "squared": 1}
    # head sits in the alignment gap before dropout_seed: size and every other offset are unchanged
    assert _lib.Config.head.offset == _lib.Config.dropout.offset + 4
    assert _lib.Config.dropout_seed.offset == _lib.Config.dropout.offset + 8
    assert ctypes.sizeof(_lib.Config) == 168
    assert _lib.Config().head == 0 and CsvConfig().label_raw == 0       # zeroed structs keep today's behaviour


@pytest.mark.parametrize("head", [2, -1, 7])
def test_create_rejects_unknown_head_without_gpu(head):
    lib = _lib.load()
    cats = (_lib.Column * 1)()
    cats[0].name, cats[0].kind, cats[0].num_buckets = b"a", _lib.COL_KIND["hash"], 10
    cfg = _lib.Config()
    cfg.n_cat, cfg.cat = 1, ctypes.cast(cats, ctypes.POINTER(_lib.Column))
    cfg.embedding_size, cfg.use_linear, cfg.max_batch, cfg.head = 4, 1, 16, head
    h = ctypes.c_void_p()
    assert lib.dfm_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    assert b"head must be one of DFM_HEAD_*" in lib.dfm_last_error(None)


def _csv_create(kinds, label_field, label_raw):
    lib = _lib.load()
    n = len(kinds)
    kind = (ctypes.c_int32 * n)(*kinds)
    cfg = CsvConfig(n, ctypes.cast(kind, ctypes.POINTER(ctypes.c_int32)), None, None, label_field, 0, 16, 4096, 0, None, 0, None,
                    label_raw)
    h = ctypes.c_void_p()
    rc = lib.dfm_csv_create(ctypes.byref(cfg), ctypes.byref(h))
    return rc, (lib.dfm_csv_last_error(None) or b"").decode()


@pytest.mark.parametrize("kinds,label_field,label_raw", [([CSV_INT32, CSV_STRING], 1, 1), ([CSV_INT32, CSV_STRING], 1, 0),
                                                         ([CSV_INT32, CSV_FLOAT32], 1, 0), ([CSV_INT32], 3, 1)])
def test_csv_label_field_checks_without_gpu(kinds, label_field, label_raw):
    """the label field must be int32, or int32 / float32 with label_raw; checked before any CUDA call"""
    rc, err = _csv_create(kinds, label_field, label_raw)
    assert rc == -1 and "label_field must be an int32 field" in err, (rc, err)
