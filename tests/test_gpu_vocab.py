"""GPU: vocabulary columns looked up through the device hash table - ids equal the oracle bit for bit for string and
integer vocabularies from 1 to 10^6 entries (hits, misses, empty values, long keys, OOV buckets, default values), with
the fingerprints truncated so that the byte comparison decides, on either forced path; as crossed-column constituents
and multivalent columns; and models with vocabulary columns train like the oracle through model_fn, the canned
estimators, the record-staged Criteo step, row sharding, the GPU CSV reader and checkpoints."""
import io

import numpy as np
import pytest

from oracle import vocab as ov
from recommender_tensorflow_b200 import feature_column as fc
from recommender_tensorflow_b200 import synth
from recommender_tensorflow_b200.engine import DeepFMEngine
from recommender_tensorflow_b200.sharded import VirtualCluster
from recommender_tensorflow_b200.trainers import ml_100k
from tests.util import assert_state_close, assert_step_close, make_pair

pytestmark = pytest.mark.gpu

DT = {"s": "string", "n": "int32", "i": "int32", "a": "int32"}


def _oracle_step(pair, specs, feats, y, x=None):
    ids = ov.transform(specs, feats)
    pair.last64 = pair.o64.train_step(ids, x, y)
    return pair.o32.train_step(ids, x, y)


def _str_vocab(V, rng):
    """V distinct keys of 1..80 bytes (a quarter over 16, some over 64)."""
    lens = rng.choice([1, 3, 8, 16, 17, 30, 40, 65, 80], V, p=[.05, .15, .2, .15, .15, .1, .1, .05, .05])
    return [(b"%d:" % j + b"k" * int(n))[:max(int(n), len(b"%d:" % j))] for j, n in enumerate(lens)]


def _str_inputs(vocab, B, rng):
    hit = [vocab[j] for j in rng.integers(0, len(vocab), B)]
    miss = [b"miss-%d" % j + b"m" * int(rng.integers(0, 70)) for j in range(B)]
    r = rng.random(B)
    vals = [b"" if r[b] < 0.1 else (hit[b] if r[b] < 0.55 else miss[b]) for b in range(B)]
    # a key sharing a prefix with a vocabulary entry, and one differing only in its last byte
    vals[0] = vocab[0][:-1] + b"#" if len(vocab[0]) > 1 else b"#"
    vals[-1] = vocab[-1] + b"x"
    return np.array(vals, dtype=object)


def _int_vocab(V, rng):
    v = rng.choice(np.arange(-2 ** 31 + 1, 2 ** 31 - 1, 997, dtype=np.int64), V, replace=False)
    return [int(x) for x in v] + [2 ** 40, -2 ** 40]       # entries outside int32 are never hit


def _int_inputs(vocab, B, rng):
    hits = np.array(vocab[:-2], np.int64)[rng.integers(0, len(vocab) - 2, B)]
    r = rng.random(B)
    out = np.where(r < 0.1, -1, np.where(r < 0.55, hits, rng.integers(-2 ** 31, 2 ** 31 - 1, B)))
    return out.astype(np.int32)


def _vocab_cols(dtype, V, rng):
    voc = _str_vocab(V, rng) if dtype == "string" else _int_vocab(V, rng)
    if dtype == "string":
        voc = [v.decode() for v in voc]
    cols = [fc.categorical_column_with_vocabulary_list("s" if dtype == "string" else "n", voc, num_oov_buckets=k)
            for k in (0, 1, 7)]
    cols += [fc.categorical_column_with_vocabulary_list("s" if dtype == "string" else "n", voc, default_value=len(voc) // 2)]
    return [fc.embedding_column(c, 4) for c in cols], voc


def _check_ids(dtype, V, seed):
    rng = np.random.default_rng(seed)
    cols, voc = _vocab_cols(dtype, V, rng)
    # four columns over the same feature would share a name: give each its own key
    keyed = []
    feats_keys = []
    for j, c in enumerate(cols):
        cc = c.categorical_column._replace(key="%s%d" % (c.categorical_column.key, j))
        keyed.append(cc)
        feats_keys.append(cc.key)
    eng = DeepFMEngine(keyed, (), embedding_size=4, hidden_units=(8,), max_batch=1000,
                       feature_dtypes={k: dtype for k in feats_keys})
    for B in (1000, 77):                                   # ragged last tile
        base = _str_inputs([v.encode() for v in voc], B, rng) if dtype == "string" else _int_inputs(voc, B, rng)
        feats = {k: base[rng.permutation(B)] for k in feats_keys}
        got = eng.transform(feats)
        want = ov.transform(eng.specs, feats)
        assert (got == want).all(), (dtype, V, B, np.argwhere(got != want)[:5])
        assert (got >= 0).any() and (got == -1).any()
    eng.close()


@pytest.mark.parametrize("dtype", ["string", "int32"])
@pytest.mark.parametrize("V", [1, 2, 9, 300, 20000, 10 ** 6])
def test_ids_equal_oracle(dtype, V):
    _check_ids(dtype, V, V)


@pytest.mark.parametrize("path,bits", [("table", 3), ("table", 64), ("scan", 64)])
@pytest.mark.parametrize("V", [1, 5, 300])
def test_ids_forced_path_and_truncated_fingerprints(monkeypatch, path, bits, V):
    """3-bit fingerprints make almost every probe meet equal fingerprints of other keys: the bytes decide."""
    monkeypatch.setenv("DFM_VOCAB_PATH", path)
    monkeypatch.setenv("DFM_VOCAB_FP_BITS", str(bits))
    _check_ids("string", V, 100 + V)
    if path == "table":
        _check_ids("int32", V, 200 + V)


def test_identity_default_value():
    cols = [fc.categorical_column_with_identity("i", 10, default_value=7), fc.categorical_column_with_identity("a", 5)]
    eng = DeepFMEngine(cols, (), embedding_size=4, hidden_units=(8,), max_batch=64, feature_dtypes=DT)
    feats = {"i": np.array([-1, 0, 9, 10, -5, 2 ** 31 - 1], np.int32), "a": np.array([0, 1, 2, 3, 4, -1], np.int32)}
    got = eng.transform(feats)
    assert got.tolist() == [[0, -1], [1, 0], [2, 9], [3, 7], [4, 7], [-1, 7]]      # model order: a, i
    assert (got == ov.transform(eng.specs, feats)).all()


def test_vocabulary_and_defaulted_identity_as_cross_constituents():
    rng = np.random.default_rng(3)
    svoc = [v.decode() for v in _str_vocab(50, rng)]
    ivoc = _int_vocab(40, rng)
    s0 = fc.categorical_column_with_vocabulary_list("s", svoc, default_value=3)
    s1 = fc.categorical_column_with_vocabulary_list("s", svoc, num_oov_buckets=5)
    n0 = fc.categorical_column_with_vocabulary_list("n", ivoc)
    n1 = fc.categorical_column_with_vocabulary_list("n", ivoc, default_value=0)
    i7 = fc.categorical_column_with_identity("i", 6, default_value=2)
    cols = [fc.crossed_column([s0, n0], 1000), fc.crossed_column([s1, n1, i7], 10 ** 6), fc.crossed_column([n1, "a"], 77),
            fc.crossed_column([i7, "s"], 300)]
    eng = DeepFMEngine(cols, (), embedding_size=4, hidden_units=(8,), max_batch=1000, feature_dtypes=DT)
    for B in (1000, 33):
        feats = {"s": _str_inputs([v.encode() for v in svoc], B, rng), "n": _int_inputs(ivoc, B, rng),
                 "i": rng.integers(-1, 9, B).astype(np.int32), "a": rng.integers(-3, 3, B).astype(np.int32)}
        got = eng.transform(feats)
        assert (got == ov.transform(eng.specs, feats)).all()
        assert (got == -1).any() and (got >= 0).any()


def test_multivalent_vocabulary_columns_ids_and_training():
    rng = np.random.default_rng(5)
    svoc = [v.decode() for v in _str_vocab(1000, rng)]
    ivoc = _int_vocab(500, rng)
    cols = [fc.categorical_column_with_vocabulary_list("s", svoc, num_oov_buckets=3),
            fc.categorical_column_with_vocabulary_list("n", ivoc, default_value=1),
            fc.categorical_column_with_identity("i", 6, default_value=0)]
    eng = DeepFMEngine(cols, (), embedding_size=8, hidden_units=(16, 16), max_batch=512, feature_dtypes=DT,
                       multivalent={"s": 3, "n": 2})
    pair, _ = make_pair(eng, seed=6)
    for step in range(3):
        B = 512
        feats = {"s": _str_inputs([v.encode() for v in svoc], B * 3, rng).reshape(B, 3),
                 "n": _int_inputs(ivoc, B * 2, rng).reshape(B, 2), "i": rng.integers(-1, 9, B).astype(np.int32)}
        y = (rng.random(B) < 0.3).astype(np.float32)
        assert (eng.transform(feats) == ov.transform(eng.specs, feats)).all()
        loss, logits = eng.train_step(feats, y, return_logits=True)
        rloss, rlogits = _oracle_step(pair, eng.specs, feats, y)
        assert_step_close(loss, logits, pair, rloss, rlogits, 1e-5, "mv vocab step %d" % step)
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "mv vocab", pair.state64())


# ---------------------------------------------------------------- training parity
def _zip_vocab_file(tmp_path, V=10 ** 5):
    """zipcode vocabulary file: V five/six-digit keys, '\\r\\n' line ends, the last line without a newline."""
    keys = [b"%05d" % j for j in range(0, 2 * V, 2)]
    p = tmp_path / "zipcode.txt"
    p.write_bytes(b"\r\n".join(keys))
    return str(p)


def ml100k_vocab(tmp_path):
    base = ml_100k.get_feature_columns(4)["linear"]
    keep = [c for c in base if c.name not in ("user_id", "item_id", "zipcode", "occupation")]
    return keep + [
        fc.categorical_column_with_vocabulary_file("zipcode", _zip_vocab_file(tmp_path), num_oov_buckets=3),
        fc.categorical_column_with_vocabulary_list("user_id", list(range(1, 944, 2)), default_value=0),
        fc.categorical_column_with_vocabulary_list("occupation", list(synth.OCCUPATIONS[:12])),
        fc.categorical_column_with_identity("item_id", 1200, default_value=5)]


def test_ml100k_deepfm_with_vocabularies_equals_oracle(tmp_path):
    from recommender_tensorflow_b200.trainers.deep_fm import _ENGINE_KEY, model_fn
    cols = ml100k_vocab(tmp_path)
    params = {"categorical_columns": cols, "embedding_size": 4, "hidden_units": [16, 16], "optimizer": "Adam",
              "learning_rate": 0.01, "tf_random_seed": 1, "max_batch": 1024}
    ml, rng = synth.ML100K(), np.random.default_rng(7)
    feats, y = ml.batch(1024, rng)
    model_fn(feats, y, ml_100k.ModeKeys.PREDICT, params)
    eng = params[_ENGINE_KEY]
    assert {s["name"]: s["num_buckets"] for s in eng.specs}["zipcode"] == 10 ** 5 + 3
    pair, _ = make_pair(eng, seed=8)
    for step in range(4):
        feats, y = ml.batch(1024, rng)
        spec = model_fn(feats, y, ml_100k.ModeKeys.TRAIN, params)
        rloss, rlogits = _oracle_step(pair, eng.specs, feats, y)
        assert_step_close(spec.loss, spec.predictions["logits"].reshape(-1), pair, rloss, rlogits, 1e-5, "ml step %d" % step)
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "ml100k vocab", pair.state64())
    names = eng.tf_variable_map()
    assert "input_layer/input_layer/zipcode_embedding/embedding_weights" in names
    assert "linear/linear_model/user_id/weights" in names


def test_canned_wide_deep_with_vocabularies_equals_oracle(tmp_path):
    from recommender_tensorflow_b200.trainers.linear_deep import DNNLinearCombinedClassifier
    cols = ml100k_vocab(tmp_path)
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
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "wide&deep vocab", pair.state64())


def _criteo(vocab, V=2000):
    cats, nums = synth.criteo_columns(500)
    if vocab:
        keys, _ = synth.hex8(np.arange(V, dtype=np.uint32) * np.uint32(3))
        voc = [bytes(keys[j * 8:(j + 1) * 8]).decode() for j in range(V)]
        cats = [fc.categorical_column_with_vocabulary_list(c.key, voc, num_oov_buckets=2) if f % 2 == 0 else c
                for f, c in enumerate(cats)]
    dt = {"C%d" % (f + 1): "string" for f in range(26)}
    return DeepFMEngine(cats, nums, embedding_size=16, hidden_units=(16, 16), max_batch=2048, feature_dtypes=dt)


def test_criteo_with_vocabularies_record_staged_equals_oracle():
    """13 of the 26 Criteo fields are vocabulary columns: the model keeps the record-staged step of the hashed model."""
    plain, eng = _criteo(False), _criteo(True)
    pair, _ = make_pair(eng, seed=11)
    make_pair(plain, seed=11)
    rng = np.random.default_rng(12)
    for step in range(5):
        feats, y = synth.criteo_batch(2048, rng, key_space=9000)
        x = np.stack([feats[c.key] for c in eng.num_columns], 1)
        loss, logits = eng.train_step(feats, y, return_logits=True)
        plain.train_step(feats, y)
        assert eng.last_step_launches == plain.last_step_launches
        rloss, rlogits = _oracle_step(pair, eng.specs, feats, y, x)
        assert_step_close(loss, logits, pair, rloss, rlogits, 1e-5, "criteo step %d" % step, noise=8.0)
    assert_state_close(eng.state(), pair.state(), 1e-5, 1e-7, "criteo vocab", pair.state64(), tc_noise=8.0)


def _names(eng):
    out = []
    for v in eng.variable_names():
        out.append(v)
        out += [v + "/" + s for s in eng.slot_names(v)]
    return out


@pytest.mark.parametrize("p2p", [False, True])
def test_sharded_with_vocabularies_equals_oracle(tmp_path, p2p):
    cols = ml100k_vocab(tmp_path)
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
        assert_step_close(loss, logits, pair, rloss, rlogits, 1e-5, "sharded vocab step %d" % step)
    assert_state_close(vc.state(_names(engs[0])), pair.state(), 1e-5, 1e-7, "sharded vocab", pair.state64())


# ---------------------------------------------------------------- input paths, checkpoints, determinism
def _trained(tmp_path, path, seed=15):
    eng = DeepFMEngine(ml100k_vocab(tmp_path), (), embedding_size=4, hidden_units=(16, 16), max_batch=1024,
                       feature_dtypes=ml_100k.FEATURE_DTYPES)
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


def test_host_and_device_steps_bit_identical_and_deterministic(tmp_path):
    a, b, c = _trained(tmp_path, "host"), _trained(tmp_path, "device"), _trained(tmp_path, "host")
    sa, sb, sc = a.state(), b.state(), c.state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
        assert np.array_equal(sa[k], sc[k]), k
    assert a.state_checksum() == b.state_checksum() == c.state_checksum()


def test_checkpoint_round_trip(tmp_path):
    eng = _trained(tmp_path, "device")
    path = eng.save_checkpoint(str(tmp_path / "model.ckpt-3.npz"))
    data = np.load(path)
    assert data["input_layer/input_layer/zipcode_embedding/embedding_weights"].shape == (10 ** 5 + 3, 4)
    assert data["linear/linear_model/user_id/weights"].shape == (472, 1)
    assert "linear/linear_model/occupation/weights/Adam" in data
    other = _trained(tmp_path, "device", seed=99)
    other.load_checkpoint(path)
    sa, sb = eng.state(), other.state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert other.global_step == 3


def test_gpu_csv_reader_with_vocabularies(tmp_path):
    from recommender_tensorflow_b200.csv_reader import GpuCsvReader
    eng = DeepFMEngine(ml100k_vocab(tmp_path), (), embedding_size=4, hidden_units=(16, 16), max_batch=600,
                       feature_dtypes=ml_100k.FEATURE_DTYPES)
    ml, rng = synth.ML100K(), np.random.default_rng(17)
    feats, y = ml.batch(600, rng)
    buf = io.StringIO()
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
    reader = GpuCsvReader(eng, ml_100k.COLUMNS, ml_100k.DEFAULTS, label_col="rating")
    pb = reader.decode(buf.getvalue().encode())
    got = eng.transform(pb)
    assert (got == eng.transform(feats)).all()
    assert (got == ov.transform(eng.specs, feats)).all()
    assert np.array_equal(reader.labels(), y)
