"""GPU: crossed_column end to end - crossed ids computed by transform_kernel equal the oracle's sparse_cross_hashed bit
for bit (upstream vectors, every constituent kind, large prime bucket counts, multivalent constituents), and models with
crosses train like the oracle through model_fn, the canned estimators, host buffers, the GPU CSV reader and row
sharding."""
import io

import numpy as np
import pytest

from oracle import cross
from recommender_tensorflow_b200 import feature_column as fc
from recommender_tensorflow_b200 import synth
from recommender_tensorflow_b200.engine import DeepFMEngine
from recommender_tensorflow_b200.sharded import VirtualCluster
from recommender_tensorflow_b200.trainers import ml_100k
from tests.util import assert_state_close, assert_step_close, make_pair

pytestmark = pytest.mark.gpu

D = cross.DEFAULT_HASH_KEY
DT = {"s": "string", "t": "string", "a": "int32", "n": "int32", "age": "int32", "g": "string", "i": "int32",
      "m": "int32", "ms": "string", "k1": "string", "k2": "string", "k3": "string"}


def _oracle_step(pair, specs, feats, y, x=None):
    ids = cross.transform(specs, feats)
    pair.last64 = pair.o64.train_step(ids, x, y)
    return pair.o32.train_step(ids, x, y)


def _names(eng):
    out = []
    for v in eng.variable_names():
        out.append(v)
        out += [v + "/" + s for s in eng.slot_names(v)]
    return out


# ---------------------------------------------------------------- ids
@pytest.mark.parametrize("hash_key,expected", [(None, 83), (D + 1, 31)])
def test_device_kat(hash_key, expected):
    col = fc.crossed_column(["k1", "k2", "k3"], 100, hash_key=hash_key)
    eng = DeepFMEngine([col], (), embedding_size=4, hidden_units=(8,), max_batch=64, feature_dtypes=DT)
    feats = {"k%d" % j: np.array([b"batch1-FC%d-F1" % j] * 3, dtype=object) for j in (1, 2, 3)}
    assert eng.transform(feats).tolist() == [[expected]] * 3


def _kind_columns(nb):
    age = fc.bucketized_column(fc.numeric_column("age"), [18, 25, 35, 50, 65])
    g0 = fc.categorical_column_with_vocabulary_list("g", ["F", "M"])
    g1 = fc.categorical_column_with_vocabulary_list("t", ["x", "yy", "zzz"], num_oov_buckets=3)
    ident = fc.categorical_column_with_identity("i", 7)
    return [fc.crossed_column(["s", "a"], nb),                       # raw string x raw int
            fc.crossed_column([age, g0, ident], nb, hash_key=12345),  # bucketized x vocab (no OOV) x identity
            fc.crossed_column([g1, "n", "s", age], nb)]              # vocab (OOV) x raw int x raw string x bucketized


def _kind_feats(B, rng):
    return {"s": np.array([b"", b"k", b"key-%d" % rng.integers(0, 50), b"a-longer-key-of-30-bytes-%05d" % rng.integers(0, 9)] * (B // 4)
                          + [b"x"] * (B % 4), dtype=object)[rng.permutation(B)],
            "a": rng.integers(-5, 200, B).astype(np.int32),
            "n": np.where(rng.random(B) < 0.2, -1, rng.integers(-2 ** 31, 2 ** 31 - 1, B)).astype(np.int32),
            "age": rng.integers(0, 90, B).astype(np.int32),
            "g": rng.choice(np.array([b"F", b"M", b"X", b""], dtype=object), B),
            "t": rng.choice(np.array([b"x", b"yy", b"zzz", b"w", b""], dtype=object), B),
            "i": np.where(rng.random(B) < 0.1, -1, rng.integers(0, 7, B)).astype(np.int32)}


@pytest.mark.parametrize("nb", [2, 100, 10 ** 7])
def test_ids_every_kind_equal_oracle(nb):
    cols = _kind_columns(nb) + [fc.categorical_column_with_hash_bucket("s", 1000)]
    eng = DeepFMEngine(cols, (), embedding_size=4, hidden_units=(8,), max_batch=1000, feature_dtypes=DT)
    rng = np.random.default_rng(nb)
    for B in (1000, 77):                                           # ragged last tiles
        feats = _kind_feats(B, rng)
        got = eng.transform(feats)
        want = cross.transform(eng.specs, feats)
        assert got.shape == (B, 4) and (got == want).all()


def test_ids_int32_max_buckets():
    """2^31 - 1 buckets: every bit of the 64-bit chain reaches the id (one cross per model: the table must fit)."""
    rng = np.random.default_rng(5)
    feats = _kind_feats(500, rng)
    for col in _kind_columns(2 ** 31 - 1):
        eng = DeepFMEngine([col], (), use_mf=False, use_dnn=False, max_batch=500, feature_dtypes=DT)
        got = eng.transform(feats)
        assert (got == cross.transform(eng.specs, feats)).all()
        assert (got >= 1 << 24).any()
        eng.close()


def _mv_feats(B, rng):
    m = rng.integers(0, 40, (B, 3)).astype(np.int32)
    m[rng.random((B, 3)) < 0.35] = -1
    m[: B // 10] = -1                                              # empty bags
    ms = rng.choice(np.array([b"p", b"q", b"rr", b""], dtype=object), (B, 2))
    return {"m": m, "ms": ms, "age": rng.integers(0, 90, B).astype(np.int32), "a": rng.integers(0, 9, B).astype(np.int32)}


def test_multivalent_constituents_ids_and_training():
    age = fc.bucketized_column(fc.numeric_column("age"), [30, 60])
    cols = [fc.crossed_column(["m", "ms"], 301), fc.crossed_column(["a", "m"], 97), fc.crossed_column([age, "a"], 53),
            fc.categorical_column_with_identity("a", 9)]
    eng = DeepFMEngine(cols, (), embedding_size=8, hidden_units=(16, 16), max_batch=512, feature_dtypes=DT,
                       multivalent={"m": 3, "ms": 2})
    # model order (sorted by "<name>_embedding"): a_X_age_bucketized, a_X_m (3 slots), a, m_X_ms (6 slots)
    assert [(s["name"], s["width"]) for s in eng.specs] == [("a_X_age_bucketized", 1), ("a_X_m", 3), ("a", 1), ("m_X_ms", 6)]
    pair, _ = make_pair(eng, seed=3)
    rng = np.random.default_rng(4)
    for step in range(3):
        feats, y = _mv_feats(512, rng), (rng.random(512) < 0.3).astype(np.float32)
        ids = eng.transform(feats)
        assert (ids == cross.transform(eng.specs, feats)).all()
        # an empty bag of m empties both of its crosses; the single-valued fields stay present
        assert (ids[:51, 1:4] == -1).all() and (ids[:51, 5:] == -1).all() and (ids[:51, [0, 4]] >= 0).all()
        loss, logits = eng.train_step(feats, y, return_logits=True)
        rloss, rlogits = _oracle_step(pair, eng.specs, feats, y)
        assert_step_close(loss, logits, pair, rloss, rlogits, 1e-5, "mv step %d" % step)
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "mv", pair.state64())


# ---------------------------------------------------------------- training parity
def ml100k_crossed(embedding_size=4):
    base = ml_100k.get_feature_columns(embedding_size)["linear"]
    by = {c.name: c for c in base}
    crosses = [fc.crossed_column(["user_id", "item_id"], 5000),
               fc.crossed_column([by["age_bucketized"], by["gender"]], 20),
               fc.crossed_column(["occupation", by["release_year_bucketized"]], 300)]
    return base + crosses


def test_ml100k_deepfm_with_crosses_equals_oracle():
    from recommender_tensorflow_b200.trainers.deep_fm import _ENGINE_KEY, model_fn
    cols = ml100k_crossed()
    params = {"categorical_columns": cols, "embedding_size": 4, "hidden_units": [16, 16], "optimizer": "Adam",
              "learning_rate": 0.01, "tf_random_seed": 1, "max_batch": 1024}
    ml, rng = synth.ML100K(), np.random.default_rng(7)
    feats, y = ml.batch(1024, rng)
    model_fn(feats, y, ml_100k.ModeKeys.PREDICT, params)            # builds the engine
    eng = params[_ENGINE_KEY]
    assert "age_bucketized_X_gender" in [s["name"] for s in eng.specs]
    pair, _ = make_pair(eng, seed=8)
    for step in range(4):
        feats, y = ml.batch(1024, rng)
        spec = model_fn(feats, y, ml_100k.ModeKeys.TRAIN, params)
        rloss, rlogits = _oracle_step(pair, eng.specs, feats, y)
        assert_step_close(spec.loss, spec.predictions["logits"].reshape(-1), pair, rloss, rlogits, 1e-5, "ml step %d" % step)
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "ml100k crossed", pair.state64())
    tf_names = eng.tf_variable_map()
    assert "linear/linear_model/age_bucketized_X_gender/weights" in tf_names
    assert "input_layer/input_layer/item_id_X_user_id_embedding/embedding_weights" in tf_names


def test_canned_wide_deep_with_crosses_equals_oracle():
    from recommender_tensorflow_b200.trainers.linear_deep import DNNLinearCombinedClassifier
    cols = ml100k_crossed()
    est = DNNLinearCombinedClassifier(linear_feature_columns=cols, dnn_feature_columns=[fc.embedding_column(c, 4) for c in cols],
                                      dnn_hidden_units=[16, 8], max_batch=512, tf_random_seed=2)
    eng = est.engine
    pair, _ = make_pair(eng, seed=9)
    ml, rng = synth.ML100K(), np.random.default_rng(10)
    for step in range(3):
        feats, y = ml.batch(512, rng)
        loss, logits = eng.train_step(feats, y, return_logits=True)
        rloss, rlogits = _oracle_step(pair, eng.specs, feats, y)
        assert_step_close(loss, logits, pair, rloss, rlogits, 1e-5, "wide&deep step %d" % step)
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "wide&deep crossed", pair.state64())
    names = eng.tf_variable_map("canned")
    assert "dnn/input_from_feature_columns/input_layer/item_id_X_user_id_embedding/embedding_weights" in names


def _criteo(n_hashed, crossed, buckets=500):
    cats, nums = synth.criteo_columns(buckets, n_cat=n_hashed)
    if crossed:
        cats = cats + [fc.crossed_column(["C%d" % a, "C%d" % b], 700) for a, b in ((1, 2), (3, 4), (5, 6))]
    dt = {"C%d" % (f + 1): "string" for f in range(26)}
    return DeepFMEngine(cats, nums, embedding_size=16, hidden_units=(16, 16), max_batch=2048, feature_dtypes=dt)


def test_crossed_fields_choose_the_tower_like_hashed_fields():
    """29 fields (26 hashed + 3 crossed) exceed the record-staged kernel's shared-memory tile exactly as 29 hashed
    fields do: both take the same step kernels."""
    a, b = _criteo(26, True), _criteo(29, False)
    rng = np.random.default_rng(18)
    feats, y = synth.criteo_batch(2048, rng, n_cat=29, key_space=3000)
    a.train_step(feats, y)
    b.train_step(feats, y)
    assert a.last_step_launches == b.last_step_launches


def test_criteo_with_crosses_record_staged_equals_oracle():
    """23 hashed + 3 crossed fields: the record-staged step of the 26-field Criteo model."""
    plain, eng = _criteo(26, False), _criteo(23, True)
    pair, _ = make_pair(eng, seed=11)
    make_pair(plain, seed=11)
    rng = np.random.default_rng(12)
    for step in range(5):
        feats, y = synth.criteo_batch(2048, rng, key_space=3000)
        x = np.stack([feats[c.key] for c in eng.num_columns], 1)
        loss, logits = eng.train_step(feats, y, return_logits=True)
        plain.train_step(feats, y)
        # the crossed model takes the same step kernels as the model without crosses (crosses of width 1 are fields)
        assert eng.last_step_launches == plain.last_step_launches
        rloss, rlogits = _oracle_step(pair, eng.specs, feats, y, x)
        assert_step_close(loss, logits, pair, rloss, rlogits, 1e-5, "criteo step %d" % step, noise=8.0)
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "criteo crossed", pair.state64(), tc_noise=8.0)


@pytest.mark.parametrize("p2p", [False, True])
def test_sharded_with_crosses_equals_oracle(p2p):
    cols = ml100k_crossed()
    kw = dict(embedding_size=4, hidden_units=(16, 16), feature_dtypes=ml_100k.FEATURE_DTYPES)
    ref = DeepFMEngine(cols, (), max_batch=1024, **kw)
    pair, w = make_pair(ref, seed=13)
    engs = [DeepFMEngine(cols, (), max_batch=512, rank=r, world=2, **kw) for r in range(2)]
    for e in engs:
        e.set_weights_sharded(w)
    vc = VirtualCluster(engs, p2p=p2p)
    ml, rng = synth.ML100K(), np.random.default_rng(14)
    for step in range(3):
        feats, y = ml.batch(1024, rng)
        pbs = [e.pack({k: v[r * 512:(r + 1) * 512] for k, v in feats.items()}, y[r * 512:(r + 1) * 512], device=True)
               for r, e in enumerate(engs)]
        loss, logits = vc.train_step(pbs, return_logits=True)
        rloss, rlogits = _oracle_step(pair, ref.specs, feats, y)
        assert_step_close(loss, logits, pair, rloss, rlogits, 1e-5, "sharded crossed step %d" % step)
    assert_state_close(vc.state(_names(engs[0])), pair.state(), 1e-5, 1e-7, "sharded crossed", pair.state64())


# ---------------------------------------------------------------- input paths, checkpoints, determinism
def _trained(path, seed=15):
    cols = ml100k_crossed()
    eng = DeepFMEngine(cols, (), embedding_size=4, hidden_units=(16, 16), max_batch=1024, feature_dtypes=ml_100k.FEATURE_DTYPES)
    eng.init_random(seed)
    ml, rng = synth.ML100K(), np.random.default_rng(16)
    for _ in range(3):
        feats, y = ml.fast_batch(1024, rng)
        if path == "host":
            eng.train_step(feats, y)
        else:
            eng.train_step_device(eng.pack(feats, y, device=True))
    eng.sync()
    return eng


def test_host_and_device_steps_bit_identical_and_deterministic():
    a, b, c = _trained("host"), _trained("device"), _trained("host")
    sa, sb, sc = a.state(), b.state(), c.state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
        assert np.array_equal(sa[k], sc[k]), k
    assert a.state_checksum() == b.state_checksum() == c.state_checksum()


def test_checkpoint_round_trip(tmp_path):
    eng = _trained("device")
    path = eng.save_checkpoint(str(tmp_path / "model.ckpt-3.npz"))
    data = np.load(path)
    assert data["linear/linear_model/occupation_X_release_year_bucketized/weights"].shape == (300, 1)
    assert data["input_layer/input_layer/item_id_X_user_id_embedding/embedding_weights"].shape == (5000, 4)
    assert "linear/linear_model/item_id_X_user_id/weights/Adam" in data
    other = _trained("device", seed=99)
    other.load_checkpoint(path)
    sa, sb = eng.state(), other.state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert other.global_step == 3


def test_gpu_csv_reader_with_crosses():
    from recommender_tensorflow_b200.csv_reader import GpuCsvReader
    cols = ml100k_crossed()
    eng = DeepFMEngine(cols, (), embedding_size=4, hidden_units=(16, 16), max_batch=600, feature_dtypes=ml_100k.FEATURE_DTYPES)
    ml, rng = synth.ML100K(), np.random.default_rng(17)
    feats, y = ml.batch(600, rng)
    buf = io.StringIO()
    buf.write(",".join(ml_100k.COLUMNS) + "\n")
    for r in range(600):
        row = []
        for name in ml_100k.COLUMNS:
            if name == "rating":
                row.append("5" if y[r] else "3")
            elif name in feats:
                v = feats[name][r]
                row.append(v.decode() if isinstance(v, bytes) else str(int(v)))
            else:
                row.append("0" if ml_100k.FEATURE_DTYPES[name] == "int32" else "x")
        buf.write(",".join(row) + "\n")
    text = buf.getvalue().encode()
    reader = GpuCsvReader(eng, ml_100k.COLUMNS, ml_100k.DEFAULTS, label_col="rating")
    body = text[text.index(b"\n") + 1:]
    pb = reader.decode(body)
    assert pb.batch_size == 600
    got = eng.transform(pb)
    assert (got == eng.transform(feats)).all()
    assert (got == cross.transform(eng.specs, feats)).all()
    assert np.array_equal(reader.labels(), y)
