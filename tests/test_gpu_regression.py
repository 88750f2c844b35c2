"""GPU: the squared head (DFM_HEAD_SQUARED, regression on the float label) on every head path.

Each parity case checks, from the kernel names torch.profiler records, that the step ran the squared (SQ) instantiation
of the head it means to test, then compares loss, logits and every weight and slot after 3 steps with the squared-head
oracle (tests/regression_oracle.py) at the bars of test_gpu_parity.py.  The worst relative errors are printed."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from recommender_tensorflow_b200 import synth
from recommender_tensorflow_b200.engine import DeepFMEngine, default_optimizer
from recommender_tensorflow_b200.sharded import VirtualCluster
from tests.regression_oracle import head_pair
from tests.test_gpu_parity import _bag_setup, _ml_engine
from tests.util import assert_state_close, assert_step_close, make_pair

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _kernels(fn):
    """names of the CUDA kernels fn() launches"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _ran_squared(names, kernel):
    """an SQ instantiation of `kernel` ran: SQ is the template argument before the last one (WGT)"""
    pat = re.compile(r"\b%s<([^>]*)>\(" % kernel)
    for n in names:
        m = pat.search(n)
        if m and [a.strip() for a in m.group(1).split(",")][-2] in ("true", "(bool)1"):
            return True
    return False


def _ratings(rng, B):
    return rng.integers(1, 6, B).astype(np.float32)


def _ml_batches(n, B, rng):
    ml = synth.ML100K()
    return [(ml.batch(B, rng)[0], _ratings(rng, B)) for _ in range(n)]


def _criteo(max_batch, buckets=50000, k=16, hidden=(16, 16), **kw):
    cats, nums = synth.criteo_columns(buckets, n_cat=26, n_num=13)
    return DeepFMEngine(cats, nums, embedding_size=k, hidden_units=hidden, max_batch=max_batch, head="squared", **kw)


def _criteo_batches(n, B, rng, **kw):
    out = []
    for _ in range(n):
        feats, _ = synth.criteo_batch(B, rng, **kw)
        out.append((feats, rng.normal(0.5, 1.0, B).astype(np.float32)))
    return out


def _run(eng, ora, batches, what, kernel, noise=4.0, tc_noise=None, weights=None, tensor_bound=()):
    """tensor_bound: tensors checked element by element against rtol + the float32 oracle's own worst deviation from
    float64 on the whole tensor (assert_state_close's tensor-wide mode, factor 1) instead of per row"""
    for i, (feats, y) in enumerate(batches):
        w = None if weights is None else weights[i]
        (loss, logits), names = _kernels(lambda: eng.train_step(feats, y, return_logits=True, weights=w))
        assert _ran_squared(names, kernel), "%s: no squared %s among %s" % (what, kernel, sorted(n for n in names if "kernel" in n))
        rloss, rlogits = ora.train_step_raw(feats, y, w)
        assert_step_close(loss, logits, ora, rloss, rlogits, RTOL, "%s step %d" % (what, i), noise=noise)
    report = {}
    ref, ref64 = ora.state(), ora.state64()
    per_row = {k: v for k, v in ref.items() if k not in tensor_bound}
    assert_state_close(eng.state(), per_row, RTOL, 1e-7, what, ref64, report=report, tc_noise=tc_noise)
    if tensor_bound:
        assert_state_close(eng.state(), {k: ref[k] for k in tensor_bound}, RTOL, 1e-7, what, ref64, report=report, tc_noise=1.0)
    print("%s: worst relative error per tensor: %s" % (what, {k: "%.1e" % v for k, v in report.items()}))


# ------------------------------------------------------------------------------------------- parity per head path
@pytest.mark.parametrize("key_space", [None, 3000], ids=["mostly-once", "repeated"])
def test_fused_rows_criteo(key_space):
    """record-staged kernel, Criteo shape (k = 16, [16, 16], Adam: FAST), rows mostly looked up once or often repeated"""
    B = 8192
    eng = _criteo(B)
    ora = head_pair(eng, make_pair(eng, seed=101)[1])
    rng = np.random.default_rng(102)
    kw = {} if key_space is None else {"key_space": key_space}
    # Mostly-once rows: a table element whose gradient is tiny is moved by Adam's g / (sqrt(v) + eps) with its rounding
    # noise amplified, and that noise is not correlated row by row with the float32 oracle's (which, on these seeds,
    # itself misses float64 on 635 emb elements by more than rtol, by up to 27x).  So emb is held to the oracle's own
    # worst deviation on the table; every other tensor keeps the per-row allowance.
    _run(eng, ora, _criteo_batches(3, B, rng, **kw), "sq-fused-rows-%s" % key_space, "fused_rows_kernel",
         tensor_bound=("emb",) if key_space is None else ())


@pytest.mark.parametrize("red", ["mean", "sum"])
def test_fused_small(red):
    eng = _ml_engine(k=4, hidden=(16, 16), max_batch=2048, head="squared", loss_reduction=red)
    ora = head_pair(eng, make_pair(eng, seed=103)[1])
    _run(eng, ora, _ml_batches(3, 2048, np.random.default_rng(104)), "sq-fused-small-" + red, "fused_small_kernel")


@pytest.mark.parametrize("opt", ["Adam", "Adagrad", "Ftrl", "RMSProp", "SGD"])
def test_every_optimizer(opt):
    """ML-100K shape on the fused small tower with each optimizer on both sides"""
    eng = _ml_engine(k=4, hidden=(16, 16), max_batch=1024, head="squared", opt_deep=default_optimizer(opt, 0.01),
                     opt_linear=default_optimizer(opt, 0.01))
    ora = head_pair(eng, make_pair(eng, seed=105)[1])
    _run(eng, ora, _ml_batches(3, 1024, np.random.default_rng(106)), "sq-opt-" + opt, "fused_small_kernel")


def test_small_mlp():
    """k = 32 on 39 fields is too wide for the fused small-tower kernel: gather + small_mlp_fwd_bwd_top_kernel"""
    eng = _criteo(1024, buckets=2000, k=32)
    ora = head_pair(eng, make_pair(eng, seed=107)[1])
    _run(eng, ora, _criteo_batches(3, 1024, np.random.default_rng(108), key_space=8000), "sq-small-mlp",
         "small_mlp_fwd_bwd_top_kernel")


def test_general_tower_tanh():
    eng = _ml_engine(k=8, hidden=(16, 8), max_batch=1024, activation="tanh", head="squared")
    ora = head_pair(eng, make_pair(eng, seed=109)[1])
    _run(eng, ora, _ml_batches(3, 1024, np.random.default_rng(110)), "sq-tanh", "head_kernel")


def test_tensor_core_tower():
    """configs[2]-shaped tower (k = 16, [256, 128]) on the tcgen05 GEMMs with the fused head + backward kernel"""
    eng = _ml_engine(k=16, hidden=(256, 128), max_batch=4096, head="squared")
    ora = head_pair(eng, make_pair(eng, seed=111)[1])
    _run(eng, ora, _ml_batches(3, 4096, np.random.default_rng(112)), "sq-tc", "head_bwd_kernel", noise=8.0, tc_noise=8.0)


def test_multivalent_columns_weighted():
    from recommender_tensorflow_b200.trainers import ml_100k
    ml, rng = synth.ML100K(), np.random.default_rng(113)
    cols, _, _ = _bag_setup(4, rng, ml)
    eng = DeepFMEngine(cols, (), embedding_size=8, hidden_units=(16, 16), max_batch=600, feature_dtypes=ml_100k.FEATURE_DTYPES,
                       multivalent={"genres": 6, "tags": 3}, head="squared", weighted=True)
    ora = head_pair(eng, make_pair(eng, seed=114)[1])
    batches = [(_bag_setup(600, rng, ml)[1], _ratings(rng, 600)) for _ in range(3)]
    weights = [rng.uniform(0.0, 3.0, 600).astype(np.float32) for _ in range(3)]
    _run(eng, ora, batches, "sq-bags-weighted", "small_mlp_fwd_bwd_top_kernel", weights=weights)


def test_graph_path_small_batches():
    eng = _ml_engine(k=4, hidden=(16, 16), max_batch=64, head="squared")
    ora = head_pair(eng, make_pair(eng, seed=115)[1])
    _run(eng, ora, _ml_batches(6, 32, np.random.default_rng(116)), "sq-graph", "fused_small_kernel")
    assert eng.graph_steps == 6


# ------------------------------------------------------------------------------------------- bit identities
@pytest.mark.parametrize("shape", ["criteo_rows", "fused_small", "graph_small_batch"])
def test_all_ones_weights_and_rerun_bit_identical(shape):
    """a weighted squared handle fed all-ones weights, and a second unweighted squared handle, reproduce an unweighted
    squared handle bit for bit"""
    rng = np.random.default_rng(117)
    if shape == "criteo_rows":
        make = lambda **kw: _criteo(4096, **kw)
        batches = _criteo_batches(4, 4096, rng, key_space=60000)
    else:
        B = 1024 if shape == "fused_small" else 32
        make = lambda **kw: _ml_engine(k=4, hidden=(16, 16), max_batch=B, head="squared", **kw)
        batches = _ml_batches(4, B, rng)
    a, b, c = make(), make(weighted=True), make()
    _, w0 = make_pair(a, seed=118)
    b.set_weights(w0)
    c.set_weights(w0)
    for feats, y in batches:
        la, za = a.train_step(feats, y, return_logits=True)
        lb, zb = b.train_step(feats, y, return_logits=True, weights=np.ones(len(y), np.float32))
        lc, zc = c.train_step(feats, y, return_logits=True)
        for l2, z2 in ((lb, zb), (lc, zc)):
            assert np.float32(la).view(np.uint32) == np.float32(l2).view(np.uint32), (shape, la, l2)
            assert np.array_equal(za.view(np.uint32), z2.view(np.uint32)), shape
    assert a.state_checksum() == b.state_checksum() == c.state_checksum()


GRAPH_SCRIPT = r"""
import sys
sys.path.insert(0, %r)
import numpy as np
from recommender_tensorflow_b200 import synth
from tests.test_gpu_parity import _ml_engine
from tests.util import make_pair
eng = _ml_engine(k=4, hidden=(16, 16), max_batch=256, head="squared")
make_pair(eng, seed=119)
ml, rng = synth.ML100K(), np.random.default_rng(120)
losses = []
for i in range(6):
    f, _ = ml.batch(48, rng)
    losses.append(eng.train_step(f, rng.integers(1, 6, 48).astype(np.float32)))
print("RESULT %%s %%s %%d" %% (eng.state_checksum(), np.asarray(losses, np.float32).view(np.uint32).tolist(), eng.graph_steps))
""" % ROOT


def test_graph_and_plain_launches_bit_identical():
    """the small-batch CUDA graph captures the squared instantiation the step launches: with DFM_NO_GRAPH=1 (read once
    per process, hence the subprocesses) the same batches leave the same bits behind"""
    out = []
    for extra in ({}, {"DFM_NO_GRAPH": "1"}):
        env = dict(os.environ)
        env.pop("DFM_NO_GRAPH", None)
        env.update(extra)
        r = subprocess.run([sys.executable, "-c", GRAPH_SCRIPT], capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        out.append([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1].rsplit(" ", 1))
    assert out[0][0] == out[1][0]
    assert int(out[0][1]) == 6 and int(out[1][1]) == 0


# ------------------------------------------------------------------------------------------- row-sharded
def _names(eng):
    out = []
    for v in eng.variable_names():
        out.append(v)
        out += [v + "/" + s for s in eng.slot_names(v)]
    return out


@pytest.mark.parametrize("p2p", [False, True])
def test_row_sharded_world2(p2p):
    world, B = 2, 1024
    cats, nums = synth.criteo_columns(500, n_cat=26, n_num=13)
    kw = dict(embedding_size=16, hidden_units=(16, 16), head="squared")
    ref = DeepFMEngine(cats, nums, max_batch=B, **kw)
    _, w0 = make_pair(ref, seed=121)
    ora = head_pair(ref, w0)
    engs = [DeepFMEngine(cats, nums, max_batch=B // world, rank=r, world=world, **kw) for r in range(world)]
    for e in engs:
        e.set_weights_sharded(w0)
    vc = VirtualCluster(engs, p2p=p2p)
    rng = np.random.default_rng(122)
    per = B // world
    for step in range(3):
        feats, _ = synth.criteo_batch(B, rng, key_space=3000)
        y = rng.normal(0.5, 1.0, B).astype(np.float32)
        pbs = []
        for r, e in enumerate(engs):
            fr = {}
            for k, v in feats.items():
                if isinstance(v, tuple):
                    data, offs = v
                    o = offs[r * per:(r + 1) * per + 1]
                    fr[k] = (data[o[0]:o[-1]].copy(), (o - o[0]).astype(np.int32))
                else:
                    fr[k] = v[r * per:(r + 1) * per]
            pbs.append(e.pack(fr, y[r * per:(r + 1) * per], device=True))
        (loss, logits), names = _kernels(lambda: vc.train_step(pbs, return_logits=True))
        assert _ran_squared(names, "fused_rows_kernel")       # the row-buffer form of the record-staged kernel
        rloss, rlogits = ora.train_step_raw(feats, y)
        assert_step_close(loss, logits, ora, rloss, rlogits, RTOL, "sq-sharded p2p=%s step %d" % (p2p, step))
    report = {}
    assert_state_close(vc.state(_names(engs[0])), ora.state(), RTOL, 1e-7, "sq-sharded", ora.state64(), report=report)
    print("sq-sharded p2p=%s: worst relative error per tensor: %s" % (p2p, {k: "%.1e" % v for k, v in report.items()}))


# ------------------------------------------------------------------------------------------- input and estimators
def test_csv_label_raw_matches_python_decoder(tmp_path):
    """GPU CSV reader with cutoff=None: the labels are the ratings as float32, as get_input_fn(cutoff=None) gives them,
    and training on either input leaves the same state"""
    from recommender_tensorflow_b200.csv_reader import GpuCsvReader
    from recommender_tensorflow_b200.trainers import ml_100k
    path = str(tmp_path / "train.csv")
    ml_100k.write_synthetic_csv(path, 500)
    eng = _ml_engine(k=4, max_batch=500, head="squared")
    reader = GpuCsvReader(eng, ml_100k.COLUMNS, ml_100k.DEFAULTS, ml_100k.LABEL_COL, cutoff=None, max_records=500)
    pb = reader.decode(open(path, "rb").read().split(b"\n", 1)[1])
    feats, y = next(ml_100k.get_input_fn(path, ml_100k.ModeKeys.EVAL, batch_size=500, cutoff=None)())
    assert np.array_equal(reader.labels(), y) and set(np.unique(y)) <= {1.0, 2.0, 3.0, 4.0, 5.0} and y.max() > 1
    # the default stays the thresholded 0/1 label
    r5 = GpuCsvReader(eng, ml_100k.COLUMNS, ml_100k.DEFAULTS, ml_100k.LABEL_COL, max_records=500)
    r5.decode(open(path, "rb").read().split(b"\n", 1)[1])
    assert np.array_equal(r5.labels(), (y >= 5).astype(np.float32))
    other = _ml_engine(k=4, max_batch=500, head="squared")
    _, w0 = make_pair(eng, seed=123)
    other.set_weights(w0)
    la = eng.train_step_device(pb)
    lb = other.train_step(feats, y)
    eng.sync()
    assert float(la.item()) == lb and eng.state_checksum() == other.state_checksum()


def test_dnn_linear_combined_regressor_checkpoint_resume(tmp_path):
    """train -> checkpoint -> a new estimator resumes from model_dir -> evaluate -> predict; one step equals the
    squared-head oracle's SUM-reduced step"""
    from recommender_tensorflow_b200.trainers import linear_deep, ml_100k
    from recommender_tensorflow_b200.trainers.model_utils import get_regression_metrics
    fcs = ml_100k.get_feature_columns(embedding_size=4)
    make = lambda: linear_deep.DNNLinearCombinedRegressor(model_dir=str(tmp_path), linear_feature_columns=fcs["linear"],
                                                          dnn_feature_columns=fcs["deep"], dnn_hidden_units=[16, 16],
                                                          max_batch=256, tf_random_seed=1)
    est = make()
    eng = est.engine
    assert eng.head == "squared" and eng.loss_reduction == "sum"
    ora = head_pair(eng, make_pair(eng, seed=124)[1])
    rng = np.random.default_rng(125)
    (feats, y), = _ml_batches(1, 256, rng)
    est.train(lambda: iter([(feats, y)]), steps=1)
    ora.train_step_raw(feats, y)
    assert_state_close(eng.state(), ora.state(), RTOL, 1e-7, "DNNLinearCombinedRegressor", ora.state64())
    (f2, y2), = _ml_batches(1, 256, rng)
    est.train(lambda: iter([(f2, y2)]), steps=1)
    assert est.latest_checkpoint().endswith("model.ckpt-2.npz")
    est2 = make()
    m = est2.evaluate(lambda: iter([(feats, y)]))
    assert m["global_step"] == 2
    ref = get_regression_metrics(y, eng.predict_logits(feats))      # the resumed model predicts what the trained one does
    assert all(m[k] == ref[k] for k in ref) and set(m) == set(ref) | {"global_step"}
    preds = list(est2.predict(lambda: iter([feats])))
    assert len(preds) == 256 and set(preds[0]) == {"predictions"}
    assert np.array_equal(np.array([p["predictions"][0] for p in preds]), eng.predict_logits(feats))


def test_canned_regressors_one_step():
    from recommender_tensorflow_b200.trainers import deep, linear, ml_100k
    fcs = ml_100k.get_feature_columns(embedding_size=4)
    rng = np.random.default_rng(126)
    for est in (linear.LinearRegressor(fcs["linear"], max_batch=256, weight_column="wt"),
                deep.DNNRegressor([16, 16], fcs["deep"], max_batch=256, tf_random_seed=1)):
        eng = est.engine
        assert eng.head == "squared" and eng.loss_reduction == "sum"
        ora = head_pair(eng, make_pair(eng, seed=127)[1])
        (feats, y), = _ml_batches(1, 256, rng)
        w = None
        if est.weight_column:
            w = rng.uniform(0.0, 3.0, 256).astype(np.float32)
            feats["wt"] = w
        est.train(lambda: iter([(feats, y)]), steps=1)
        ora.train_step_raw(feats, y, w)
        assert_state_close(eng.state(), ora.state(), RTOL, 1e-7, type(est).__name__, ora.state64())


def test_model_fn_regression_three_modes():
    from recommender_tensorflow_b200.trainers import deep_fm, ml_100k
    from recommender_tensorflow_b200.trainers.model_utils import get_regression_metrics
    cols = ml_100k.get_feature_columns(embedding_size=4)["linear"]
    params = {"categorical_columns": cols, "embedding_size": 4, "hidden_units": [16, 16], "dropout": 0, "max_batch": 128,
              "tf_random_seed": 3, "head": "regression"}
    (feats, y), = _ml_batches(1, 128, np.random.default_rng(128))
    spec = deep_fm.model_fn(feats, y, ml_100k.ModeKeys.TRAIN, params)
    eng = params[deep_fm._ENGINE_KEY]
    assert eng.head == "squared" and eng.loss_reduction == "mean"
    assert set(spec.predictions) == {"predictions"} and spec.predictions["predictions"].shape == (128, 1)
    z = eng.predict_logits(feats)
    assert spec.loss > 0
    ev = deep_fm.model_fn(feats, y, ml_100k.ModeKeys.EVAL, params)
    assert ev.eval_metric_ops == get_regression_metrics(y, z) and ev.loss == ev.eval_metric_ops["average_loss"]
    pr = deep_fm.model_fn(feats, None, ml_100k.ModeKeys.PREDICT, params)
    assert np.array_equal(pr.predictions["predictions"][:, 0], z)
