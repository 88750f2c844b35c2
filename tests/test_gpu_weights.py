"""GPU: per-example weights (weight_column) applied on the device where dz and the loss term are formed.

A weighted handle fed all-ones weights is bit-identical to an unweighted one; with random weights in [0, 3] (zeros
included) every head path matches the oracle at the bars of test_gpu_parity.py.  Each case checks, from the kernel names
torch.profiler records, that the step ran the weighted instantiation of the head it means to test."""
import re

import numpy as np
import pytest

from recommender_tensorflow_b200 import synth
from recommender_tensorflow_b200.engine import DeepFMEngine
from recommender_tensorflow_b200.sharded import VirtualCluster
from tests.test_gpu_parity import _bag_setup, _ml_engine
from tests.util import assert_state_close, assert_step_close, make_pair
from tests.weighted_oracle import weighted_pair, weighted_step

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def _kernels(fn):
    """names of the CUDA kernels fn() launches"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _ran_weighted(names, kernel):
    """a weighted (last template argument true) instantiation of `kernel` ran"""
    pat = re.compile(r"\b%s<[^>]*(true|\(bool\)1)>\(" % kernel)
    return any(pat.search(n) for n in names)


def _weights(rng, B):
    w = rng.uniform(0.0, 3.0, B).astype(np.float32)
    w[rng.random(B) < 0.1] = 0.0
    return w


def _run_weighted(eng, ora, batches, what, kernel, noise=4.0, tc_noise=None, seed=0):
    rng = np.random.default_rng(seed)
    for i, (feats, y) in enumerate(batches):
        w = _weights(rng, len(y))
        (loss, logits), names = _kernels(lambda: eng.train_step(feats, y, return_logits=True, weights=w))
        assert _ran_weighted(names, kernel), "%s: no weighted %s among %s" % (what, kernel, sorted(n for n in names if "kernel" in n))
        rloss, rlogits = weighted_step(ora, feats, y, w)
        assert_step_close(loss, logits, ora, rloss, rlogits, RTOL, "%s step %d" % (what, i), noise=noise)
    report = {}
    assert_state_close(eng.state(), ora.state(), RTOL, 1e-7, what, ora.state64(), report=report, tc_noise=tc_noise)
    print("%s: worst relative error per tensor: %s" % (what, {k: "%.1e" % v for k, v in report.items()}))


# ------------------------------------------------------------------------------------------- all-ones = unweighted
def _criteo(max_batch, buckets=50000, k=16, hidden=(16, 16), **kw):
    cats, nums = synth.criteo_columns(buckets, n_cat=26, n_num=13)
    return DeepFMEngine(cats, nums, embedding_size=k, hidden_units=hidden, max_batch=max_batch, **kw)


@pytest.mark.parametrize("shape", ["criteo_rows", "fused_small", "graph_small_batch"])
def test_all_ones_weights_bit_identical(shape):
    if shape == "criteo_rows":
        make = lambda **kw: _criteo(4096, **kw)
        gen = lambda rng: synth.criteo_batch(4096, rng, key_space=60000)
        kernel = "fused_rows_kernel"
    else:
        B = 1024 if shape == "fused_small" else 32
        make = lambda **kw: _ml_engine(k=4, hidden=(16, 16), max_batch=B, **kw)
        ml = synth.ML100K()
        gen = lambda rng: ml.batch(B, rng)
        kernel = "fused_small_kernel"
    a, b = make(), make(weighted=True)
    _, w0 = make_pair(a, seed=41)
    b.set_weights(w0)
    rng = np.random.default_rng(42)
    for step in range(4):
        feats, y = gen(rng)
        la, za = a.train_step(feats, y, return_logits=True)
        (lb, zb), names = _kernels(lambda: b.train_step(feats, y, return_logits=True, weights=np.ones(len(y), np.float32)))
        assert _ran_weighted(names, kernel), sorted(n for n in names if "kernel" in n)
        assert np.float32(la).view(np.uint32) == np.float32(lb).view(np.uint32), (shape, step, la, lb)
        assert np.array_equal(za.view(np.uint32), zb.view(np.uint32)), (shape, step)
        assert a.last_step_launches == b.last_step_launches
    assert a.state_checksum() == b.state_checksum()
    assert a.graph_steps == b.graph_steps == 4      # every case here is at most 131072 samples: one graph per step
    sa, sb = a.state(), b.state()
    for n in sa:
        assert np.array_equal(sa[n].view(np.uint32), sb[n].view(np.uint32)), n


# ------------------------------------------------------------------------------------------- parity per head path
def test_fused_rows_large_batch():
    """record-staged kernel, Criteo shape, above the graph threshold (plain launches)"""
    B = 131073
    eng = _criteo(B, weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=51)[1])
    rng = np.random.default_rng(52)
    _run_weighted(eng, ora, [synth.criteo_batch(B, rng) for _ in range(2)], "w-fused-rows", "fused_rows_kernel", seed=53)
    assert eng.graph_steps == 0


def test_fused_small():
    eng = _ml_engine(k=4, hidden=(16, 16), max_batch=2048, weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=54)[1])
    ml, rng = synth.ML100K(), np.random.default_rng(55)
    _run_weighted(eng, ora, [ml.batch(2048, rng) for _ in range(3)], "w-fused-small", "fused_small_kernel", seed=56)


def test_small_mlp():
    """k = 32 on 39 fields is too wide for the fused small-tower kernel: gather + small_mlp_fwd_bwd_top_kernel"""
    eng = _criteo(1024, buckets=2000, k=32, weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=57)[1])
    rng = np.random.default_rng(58)
    _run_weighted(eng, ora, [synth.criteo_batch(1024, rng, key_space=8000) for _ in range(3)], "w-small-mlp",
                  "small_mlp_fwd_bwd_top_kernel", seed=59)


def test_general_tower_tanh():
    eng = _ml_engine(k=8, hidden=(16, 8), max_batch=1024, activation="tanh", weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=60)[1])
    ml, rng = synth.ML100K(), np.random.default_rng(61)
    _run_weighted(eng, ora, [ml.batch(1024, rng) for _ in range(3)], "w-tanh", "head_kernel", seed=62)


def test_tensor_core_tower():
    eng = _ml_engine(k=16, hidden=(256, 128), max_batch=4096, weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=63)[1])
    ml, rng = synth.ML100K(), np.random.default_rng(64)
    _run_weighted(eng, ora, [ml.batch(4096, rng) for _ in range(3)], "w-tc", "head_bwd_kernel", seed=65)


def test_linear_only_sum():
    eng = _ml_engine(k=4, max_batch=1024, use_mf=False, use_dnn=False, loss_reduction="sum", weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=66)[1])
    ml, rng = synth.ML100K(), np.random.default_rng(67)
    _run_weighted(eng, ora, [ml.batch(1024, rng) for _ in range(3)], "w-linear", "head_kernel", seed=68)


def test_multivalent_columns():
    from recommender_tensorflow_b200.trainers import ml_100k
    ml, rng = synth.ML100K(), np.random.default_rng(70)
    cols, _, _ = _bag_setup(4, rng, ml)
    eng = DeepFMEngine(cols, (), embedding_size=8, hidden_units=(16, 16), max_batch=600, feature_dtypes=ml_100k.FEATURE_DTYPES,
                       multivalent={"genres": 6, "tags": 3}, weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=71)[1])
    batches = [_bag_setup(600, rng, ml)[1:] for _ in range(3)]
    _run_weighted(eng, ora, batches, "w-bags", "small_mlp_fwd_bwd_top_kernel", seed=72)


def test_graph_path_new_weight_buffers_every_step():
    """small batches replay one CUDA graph per step: each step brings its own weights buffer (host and device batches
    alternate), and the graph must read this step's, never a stale one"""
    eng = _ml_engine(k=4, hidden=(16, 16), max_batch=64, weighted=True)
    ora = weighted_pair(eng, make_pair(eng, seed=73)[1])
    ml, rng = synth.ML100K(), np.random.default_rng(74)
    for i in range(6):
        feats, y = ml.batch(32, rng)
        w = _weights(rng, 32)
        if i % 2:
            loss, logits = eng.train_step(feats, y, return_logits=True, weights=w)
        else:
            loss, logits = eng.train_step_device(eng.pack(feats, y, device=True, weights=w), return_logits=True)
        rloss, rlogits = weighted_step(ora, feats, y, w)
        assert_step_close(loss, logits, ora, rloss, rlogits, RTOL, "w-graph step %d" % i)
    assert eng.graph_steps == 6
    assert_state_close(eng.state(), ora.state(), RTOL, 1e-7, "w-graph", ora.state64())


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
    kw = dict(embedding_size=16, hidden_units=(16, 16))
    ref = DeepFMEngine(cats, nums, max_batch=B, **kw)
    _, w0 = make_pair(ref, seed=75)
    ora = weighted_pair(ref, w0)
    engs = [DeepFMEngine(cats, nums, max_batch=B // world, rank=r, world=world, weighted=True, **kw) for r in range(world)]
    for e in engs:
        e.set_weights_sharded(w0)
    vc = VirtualCluster(engs, p2p=p2p)
    rng = np.random.default_rng(76)
    per = B // world
    for step in range(3):
        feats, y = synth.criteo_batch(B, rng, key_space=3000)
        w = _weights(rng, B)
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
            pbs.append(e.pack(fr, y[r * per:(r + 1) * per], device=True, weights=w[r * per:(r + 1) * per]))
        (loss, logits), names = _kernels(lambda: vc.train_step(pbs, return_logits=True))
        assert _ran_weighted(names, "fused_rows_kernel")       # the row-buffer form of the record-staged kernel
        rloss, rlogits = weighted_step(ora, feats, y, w)
        assert_step_close(loss, logits, ora, rloss, rlogits, RTOL, "w-sharded p2p=%s step %d" % (p2p, step))
    assert_state_close(vc.state(_names(engs[0])), ora.state(), RTOL, 1e-7, "w-sharded", ora.state64())


# ------------------------------------------------------------------------------------------- API edges
def test_weighted_engine_requires_weights_and_unweighted_ignores_them():
    from recommender_tensorflow_b200._lib import DfmError
    ml, rng = synth.ML100K(), np.random.default_rng(77)
    feats, y = ml.batch(64, rng)
    eng = _ml_engine(k=4, max_batch=64, weighted=True)
    with pytest.raises(ValueError):
        eng.train_step(feats, y)
    pb = eng.pack(feats, y, device=True, weights=np.ones(64, np.float32))
    pb.raw.weights = None
    with pytest.raises(DfmError):
        eng.train_step_device(pb)
    assert eng.global_step == 0
    z = eng.predict_logits(feats)                 # forward reads no weights
    assert z.shape == (64,)
    a, b = _ml_engine(k=4, max_batch=64), _ml_engine(k=4, max_batch=64)       # unweighted engines ignore weights
    make_pair(a, seed=0)
    make_pair(b, seed=0)
    assert a.train_step(feats, y) == b.train_step(feats, y, weights=np.full(64, 7.0, np.float32))
    assert a.state_checksum() == b.state_checksum()


# ------------------------------------------------------------------------------------------- end to end
def test_csv_weight_field_gpu_input_equals_host_input(tmp_path):
    """model_fn with params["weight_column"]: a weight field of the CSV (the int32 age, read as float)
    through the GPU CSV reader gives the same trained state and the same weighted EVAL metrics as host-parsed input."""
    from recommender_tensorflow_b200 import feature_column as fc
    from recommender_tensorflow_b200.trainers import deep_fm, ml_100k
    path = str(tmp_path / "train.csv")
    ml_100k.write_synthetic_csv(path, 700)
    cols = ml_100k.get_feature_columns(embedding_size=4)["linear"]
    results = []
    for gpu in (False, True):
        est = deep_fm.Estimator(model_fn=deep_fm.model_fn, model_dir=None, params={
            "categorical_columns": cols, "embedding_size": 4, "hidden_units": [16, 16], "dropout": 0, "max_batch": 64,
            "tf_random_seed": 3, "weight_column": fc.numeric_column("age", dtype="int32")})
        eng = est.build(64)
        assert eng.weighted
        if gpu:
            train = ml_100k.get_gpu_input_fn(path, eng, batch_size=64, seed=9, weight_column="age")
            evalf = ml_100k.get_gpu_input_fn(path, eng, ml_100k.ModeKeys.EVAL, batch_size=64, weight_column="age")
        else:
            train = ml_100k.get_input_fn(path, batch_size=64, seed=9)
            evalf = ml_100k.get_input_fn(path, ml_100k.ModeKeys.EVAL, batch_size=64)
        est.SAVE_SUMMARY_STEPS = 0
        est.train(train, max_steps=8, log_every=0)
        results.append((eng.state_checksum(), est.evaluate(evalf)))
    assert results[0][0] == results[1][0]
    assert results[0][1] == results[1][1]
    # the weights change the model: an unweighted run of the same batches ends elsewhere
    est = deep_fm.Estimator(model_fn=deep_fm.model_fn, model_dir=None, params={
        "categorical_columns": cols, "embedding_size": 4, "hidden_units": [16, 16], "dropout": 0, "max_batch": 64, "tf_random_seed": 3})
    est.SAVE_SUMMARY_STEPS = 0
    est.train(ml_100k.get_input_fn(path, batch_size=64, seed=9), max_steps=8, log_every=0)
    assert est.engine.state_checksum() != results[0][0]


def test_canned_estimators_weight_column_sum_reduction():
    """LinearClassifier / DNNClassifier / DNNLinearCombinedClassifier with weight_column: one step equals the oracle's
    SUM-reduced weighted step; a missing weight feature is a KeyError"""
    from recommender_tensorflow_b200.trainers import deep, linear, linear_deep, ml_100k
    fcs = ml_100k.get_feature_columns(embedding_size=4)
    ml, rng = synth.ML100K(), np.random.default_rng(80)
    for est in (linear.LinearClassifier(fcs["linear"], max_batch=256, weight_column="wt"),
                deep.DNNClassifier([16, 16], fcs["deep"], max_batch=256, weight_column="wt", tf_random_seed=1),
                linear_deep.DNNLinearCombinedClassifier(linear_feature_columns=fcs["linear"], dnn_feature_columns=fcs["deep"],
                                                        dnn_hidden_units=[16, 16], max_batch=256, weight_column="wt",
                                                        tf_random_seed=1)):
        eng = est.engine
        assert eng.weighted and eng.loss_reduction == "sum"
        ora = weighted_pair(eng, make_pair(eng, seed=81)[1])
        feats, y = ml.batch(256, rng)
        w = _weights(rng, 256)
        feats["wt"] = w
        est.train(lambda: iter([(feats, y)]), steps=1)
        weighted_step(ora, feats, y, w)
        assert_state_close(eng.state(), ora.state(), RTOL, 1e-7, type(est).__name__, ora.state64())
        m = est.evaluate(lambda: iter([(feats, y)]))
        from recommender_tensorflow_b200.trainers.model_utils import get_binary_metrics
        ref = get_binary_metrics(y, eng.predict_logits(feats), w)
        assert all(m[k] == ref[k] for k in ref)
        with pytest.raises(KeyError):
            est.evaluate(lambda: iter([({k: v for k, v in feats.items() if k != "wt"}, y)]))
