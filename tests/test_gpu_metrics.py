"""GPU: EVAL metrics streamed on the device (csrc/metrics.cuh, dfm_metrics_* / dfm_evaluate) against oracle/metrics.py fed the
SAME device logits.  Counts are exact except that a sample whose float32 p lies within a few ulps of a threshold may sit in
the neighbouring bin (the device's expf and numpy's exp may differ in the last bits): the number of such samples bounds
the bins that may differ.  Float64 sums agree to 1e-12 of the sum of their absolute terms."""
import numpy as np
import pytest

from oracle import metrics as om
from recommender_tensorflow_b200 import synth
from recommender_tensorflow_b200._lib import DfmError
from recommender_tensorflow_b200.engine import DeepFMEngine
from recommender_tensorflow_b200.sharded import VirtualCluster
from recommender_tensorflow_b200.trainers import ml_100k
from recommender_tensorflow_b200.trainers.model_utils import finish_metrics, get_binary_metrics
from tests.util import make_pair

pytestmark = pytest.mark.gpu
BIN_KEYS = {"accuracy", "accuracy_baseline", "auc", "auc_precision_recall", "average_loss", "loss", "label/mean",
            "precision", "prediction/mean", "recall"}
REG_KEYS = {"average_loss", "loss", "label/mean", "prediction/mean"}


def _engine(head="logistic", weighted=False, max_batch=4097, seed=0):
    eng = DeepFMEngine(ml_100k.get_feature_columns()["linear"], (), embedding_size=4, hidden_units=(16, 16),
                       max_batch=max_batch, feature_dtypes=ml_100k.FEATURE_DTYPES, head=head, weighted=weighted)
    eng.init_random(seed)
    return eng


def _labels(rng, n, head):
    return (rng.random(n) < 0.4).astype(np.float32) if head == "logistic" else rng.integers(1, 6, n).astype(np.float32)


def _weights(rng, n):
    """zero, fractional and negative weights"""
    return rng.choice([0.0, 0.25, 1.0, 1.5, 3.0, -0.5], size=n).astype(np.float32)


def _abs_sums(z, y, w, head):
    z, y = z.astype(np.float64), y.astype(np.float64)
    w = np.ones_like(z) if w is None else np.abs(w.astype(np.float64))
    if head == "squared":
        return np.array([w.sum(), (w * np.abs(y)).sum(), (w * np.abs(z)).sum(), (w * (y - z) ** 2).sum()])
    loss = np.maximum(z, 0) - z * y + np.log1p(np.exp(-np.abs(z)))
    return np.array([w.sum(), (w * np.abs(y)).sum(), (w / (1 + np.exp(-z))).sum(), (w * np.abs(loss)).sum()])


def assert_state_matches(dev, ora, z, y, w, what=""):
    """device state vs the oracle state of the same logits (z: all logits of the stream, concatenated)"""
    head = ora["head"]
    assert dev["head"] == head and dev["weighted"] == ora["weighted"]
    assert int(dev["n"]) == int(ora["n"]), what
    scale = _abs_sums(z, y, w, head)
    assert np.all(np.abs(dev["sums"] - ora["sums"]) <= 1e-12 * scale + 1e-300), (what, dev["sums"], ora["sums"])
    if head == "squared":
        assert not dev["bin_count"].any() and not dev["cls"].any() and not dev["bin_weight"].any() and not dev["w_cls"].any()
        return
    assert np.array_equal(dev["cls"], ora["cls"]), what
    wscale = scale[0]
    assert np.all(np.abs(dev["w_cls"] - ora["w_cls"]) <= 1e-12 * wscale), what
    near = int(om.near_threshold(z).sum())
    moved = int(np.abs(dev["bin_count"] - ora["bin_count"]).sum()) // 2
    assert moved <= near, (what, moved, near)
    for c in (0, 1):
        assert dev["bin_count"][c].sum() == ora["bin_count"][c].sum(), what
        assert abs(dev["bin_weight"][c].sum() - ora["bin_weight"][c].sum()) <= 1e-12 * wscale, what
    if near == 0:
        assert np.array_equal(dev["bin_count"], ora["bin_count"]), what
        assert np.all(np.abs(dev["bin_weight"] - ora["bin_weight"]) <= 1e-12 * wscale), what


def _accumulate(eng, batches):
    import torch
    eng.metrics_reset()
    for z, y, w in batches:
        t = [torch.from_numpy(a).cuda() if a is not None else None for a in (z, y, w)]
        eng.metrics_accumulate(t[0], t[1], t[2])
    return eng.metrics_state()


# ---------------------------------------------------------------------------------- the kernel on given logits
@pytest.mark.parametrize("head", ["logistic", "squared"])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("n", [1, 31, 512, 513, 4097, 65536, 200000])
def test_accumulate_matches_oracle(head, weighted, n):
    """ragged sizes, one tile (512), more than one, B = 65 536, and more tiles than CTAs (200 000)"""
    rng = np.random.default_rng(n)
    eng = _engine(head, weighted, max_batch=64)
    z = rng.normal(0, 3, n).astype(np.float32)
    z[:n // 10] = 0.0                                      # ties: class 0
    y = _labels(rng, n, head)
    w = _weights(rng, n) if weighted else None
    dev = _accumulate(eng, [(z, y, w)])
    ora = om.batch_state(z, y, w, head)
    assert_state_matches(dev, ora, z, y, w, "n=%d" % n)


@pytest.mark.parametrize("head", ["logistic", "squared"])
def test_stream_of_batches_and_bit_identical_rerun(head):
    rng = np.random.default_rng(7)
    eng = _engine(head, True, max_batch=64)
    batches = []
    for n in (1, 31, 4097, 700, 65536, 3):
        batches.append((rng.normal(0, 2, n).astype(np.float32), _labels(rng, n, head), _weights(rng, n)))
    dev = _accumulate(eng, batches)
    ora = om.stream_state(batches, head, True)
    cat = [np.concatenate([b[i] for b in batches]) for i in range(3)]
    assert_state_matches(dev, ora, *cat, what="stream")
    again = _accumulate(eng, batches)
    for k in ("n", "bin_count", "cls", "bin_weight", "w_cls", "sums"):
        assert np.array_equal(np.atleast_1d(dev[k]).view(np.uint8), np.atleast_1d(again[k]).view(np.uint8)), k
    # unweighted handle: weights are not read, the state counts unit weights
    eng_u = _engine(head, False, max_batch=64)
    du = _accumulate(eng_u, batches)
    ou = om.stream_state([(z, y, None) for z, y, _ in batches], head, False)
    assert_state_matches(du, ou, cat[0], cat[1], None, "unweighted")


# ---------------------------------------------------------------------------------- dfm_evaluate on a model
@pytest.mark.parametrize("head", ["logistic", "squared"])
@pytest.mark.parametrize("weighted", [False, True])
def test_evaluate_device_and_host_batches(head, weighted):
    """dfm_evaluate (device PackedBatch) and dfm_evaluate_host (host dict) against the oracle fed predict_logits of the same
    batches; both paths give the same bits"""
    rng = np.random.default_rng(11)
    eng = _engine(head, weighted, seed=12)
    make_pair(eng, seed=13)
    ml = synth.ML100K()
    batches = []
    for n in (1, 31, 4097):
        feats, _ = ml.batch(n, rng)
        batches.append((feats, _labels(rng, n, head), _weights(rng, n) if weighted else None))
    logits = [eng.predict_logits(f) for f, _, _ in batches]
    ora = om.stream_state([(z, y, w) for z, (_, y, w) in zip(logits, batches)], head, weighted)
    states = []
    for device in (True, False):
        eng.metrics_reset()
        for f, y, w in batches:
            eng.evaluate_batch(eng.pack(f, y, device=True, weights=w) if device else f, y, w)
        states.append(eng.metrics_state())
        cat = [np.concatenate(logits)] + [None if batches[0][i] is None else np.concatenate([b[i] for b in batches]) for i in (1, 2)]
        assert_state_matches(states[-1], ora, *cat, what="device" if device else "host")
    for k in ("n", "bin_count", "cls", "bin_weight", "w_cls", "sums"):
        assert np.array_equal(states[0][k], states[1][k]), k
    m = finish_metrics(states[0])
    assert set(m) == (BIN_KEYS if head == "logistic" else REG_KEYS)


def test_evaluate_errors():
    rng = np.random.default_rng(14)
    feats, y = synth.ML100K().batch(64, rng)
    eng = _engine("logistic", True, max_batch=64)
    w = _weights(rng, 64)
    pb = eng.pack(feats, y, device=True, weights=w)
    pb.raw.weights = None
    with pytest.raises(DfmError) as e:
        eng.evaluate_batch(pb)
    assert e.value.code == -1 and "weights" in str(e.value)
    pb = eng.pack(feats, y, device=True, weights=w)
    pb.raw.labels = None
    with pytest.raises(DfmError) as e:
        eng.evaluate_batch(pb)
    assert e.value.code == -1 and "labels" in str(e.value)
    with pytest.raises(DfmError):
        eng.evaluate_batch(feats)                         # host batch without labels
    import torch
    t = torch.zeros(64, device="cuda")
    with pytest.raises(DfmError):
        eng.metrics_accumulate(t, t, None)                # weighted handle, no weights
    eng.metrics_reset()
    assert int(eng.metrics_state()["n"]) == 0             # nothing was accumulated by the rejected calls


# ---------------------------------------------------------------------------------- estimators
def _straddle(z):
    """samples whose float32 and float64 p fall on different sides of a threshold (the host evaluate() uses float64)"""
    th = om.thresholds()
    z = np.asarray(z, np.float32)
    b32 = np.searchsorted(th, om.prob32(z))
    b64 = np.searchsorted(th.astype(np.float64), 1.0 / (1.0 + np.exp(-z.astype(np.float64))))
    return int((b32 != b64).sum())


def _compare_host(m, ref, z, what):
    assert set(m) == set(ref), what
    for k in ref:
        tol = 1e-9 if (k.startswith("auc") and _straddle(z) == 0) or not k.startswith("auc") else 5e-3
        assert abs(m[k] - ref[k]) <= tol * max(1.0, abs(ref[k])), (what, k, m[k], ref[k])


def test_estimator_evaluate_streaming_host_and_gpu_input(tmp_path):
    from recommender_tensorflow_b200 import feature_column as fc
    from recommender_tensorflow_b200.trainers import deep_fm
    path = str(tmp_path / "data.csv")
    ml_100k.write_synthetic_csv(path, 900)
    cols = ml_100k.get_feature_columns(embedding_size=4)["linear"]
    for weighted in (False, True):
        params = {"categorical_columns": cols, "embedding_size": 4, "hidden_units": [16, 16], "dropout": 0, "max_batch": 128,
                  "tf_random_seed": 3}
        if weighted:
            params["weight_column"] = fc.numeric_column("age", dtype="int32")
        est = deep_fm.Estimator(model_fn=deep_fm.model_fn, model_dir=None, params=params)
        est.SAVE_SUMMARY_STEPS = 0
        eng = est.build(128)
        est.train(ml_100k.get_input_fn(path, batch_size=128, seed=9), max_steps=12, log_every=0)
        host_fn = ml_100k.get_input_fn(path, ml_100k.ModeKeys.EVAL, batch_size=128)
        gpu_fn = ml_100k.get_gpu_input_fn(path, eng, ml_100k.ModeKeys.EVAL, batch_size=128, device_labels=True,
                                          weight_column="age" if weighted else None)
        assert all(lab is None for _, lab in gpu_fn())   # nothing read back
        ref = est.evaluate(host_fn)
        a, b = est.evaluate_streaming(host_fn), est.evaluate_streaming(gpu_fn)
        # the GPU reader's batches are decoded into the same buffers: each decode is ordered after the previous
        # batch's evaluation, so the streamed result equals the host-input one exactly
        assert a == b
        assert set(a) == BIN_KEYS | {"global_step"} and a["global_step"] == 12
        z = np.concatenate([eng.predict_logits(f) for f, _ in host_fn()])
        _compare_host(a, ref, z, "weighted=%s" % weighted)
        # steps: the first two batches only
        feats = list(host_fn())[:2]
        part = est.evaluate_streaming(host_fn, steps=2)
        y2 = np.concatenate([lab for _, lab in feats])
        w2 = np.concatenate([f["age"] for f, _ in feats]).astype(np.float32) if weighted else None
        z2 = np.concatenate([eng.predict_logits(f) for f, _ in feats])
        _compare_host({k: v for k, v in part.items() if k != "global_step"}, get_binary_metrics(y2, z2, w2), z2, "steps=2")


def test_canned_evaluate_streaming(tmp_path):
    from recommender_tensorflow_b200.trainers import linear_deep
    path = str(tmp_path / "data.csv")
    ml_100k.write_synthetic_csv(path, 600)
    fcs = ml_100k.get_feature_columns(embedding_size=4)
    for cls, cutoff in ((linear_deep.DNNLinearCombinedClassifier, 5), (linear_deep.DNNLinearCombinedRegressor, None)):
        est = cls(linear_feature_columns=fcs["linear"], dnn_feature_columns=fcs["deep"], dnn_hidden_units=[16, 16],
                  max_batch=100, tf_random_seed=1)
        est.train(ml_100k.get_input_fn(path, batch_size=100, seed=2, cutoff=cutoff), steps=5)
        host_fn = ml_100k.get_input_fn(path, ml_100k.ModeKeys.EVAL, batch_size=100, cutoff=cutoff)
        gpu_fn = ml_100k.get_gpu_input_fn(path, est.engine, ml_100k.ModeKeys.EVAL, batch_size=100, cutoff=cutoff,
                                          device_labels=True)
        ref = est.evaluate(host_fn)
        a, b = est.evaluate_streaming(host_fn), est.evaluate_streaming(gpu_fn)
        assert a == b
        z = np.concatenate([est.engine.predict_logits(f) for f, _ in host_fn()])
        _compare_host(a, ref, z, cls.__name__)
        assert set(a) == (BIN_KEYS if cutoff else REG_KEYS) | {"global_step"}


# ---------------------------------------------------------------------------------- row-sharded
@pytest.mark.parametrize("p2p", [False, True])
@pytest.mark.parametrize("weighted", [False, True])
def test_virtual_cluster_world2_equals_single_gpu(p2p, weighted):
    cats, nums = synth.criteo_columns(3000, n_cat=10, n_num=5)
    kw = dict(embedding_size=8, hidden_units=(32, 16), weighted=weighted)
    world, per = 2, 300
    ref = DeepFMEngine(cats, nums, max_batch=world * per, **kw)
    _, wts = make_pair(ref, seed=31)
    engs = [DeepFMEngine(cats, nums, max_batch=per, rank=r, world=world, **kw) for r in range(world)]
    for e in engs:
        e.set_weights_sharded(wts)
    vc = VirtualCluster(engs, p2p=p2p)
    rng = np.random.default_rng(32)

    def split(feats, y, w):
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
            sl = slice(r * per, (r + 1) * per)
            pbs.append(e.pack(fr, y[sl], device=True, weights=None if w is None else w[sl]))
        return pbs
    steps = []
    ref.metrics_reset()
    for _ in range(3):
        feats, y = synth.criteo_batch(world * per, rng, key_space=5000)
        w = _weights(rng, world * per) if weighted else None
        steps.append(split(feats, y, w))
        ref.evaluate_batch(feats, y, w)
    m = vc.evaluate(iter(steps))
    want = finish_metrics(ref.metrics_state())
    assert set(m) == BIN_KEYS
    for k in want:
        assert abs(m[k] - want[k]) <= 1e-10 * max(1.0, abs(want[k])), (k, m[k], want[k])
    assert vc.evaluate(iter(steps), steps=1) != m
