"""CPU: crossed_column semantics - the oracle's hash chain on the upstream TF vectors, the order / missing-value / OOV
rules on hand-built inputs, the column's name and TF's argument checks, and the C ABI's rejections (dfm_create validates
crossed columns before any CUDA call)."""
import ctypes

import numpy as np
import pytest

from oracle import cross
from oracle.farmhash import fingerprint64
from recommender_tensorflow_b200 import _lib
from recommender_tensorflow_b200 import feature_column as fc
from recommender_tensorflow_b200.engine import cross_spec

D = cross.DEFAULT_HASH_KEY
KAT_BAGS = [[b"batch1-FC1-F1"], [b"batch1-FC2-F1"], [b"batch1-FC3-F1"]]


# ---------------------------------------------------------------- upstream vectors (sparse_cross_op_test.py)
@pytest.mark.parametrize("hash_key,num_buckets,expected", [
    (None, 0, 1971693436396284976),
    (D + 1, 0, 4847552627144134031),
    (None, 100, 83),
    (D + 1, 100, 31),
])
def test_sparse_cross_hashed_kat(hash_key, num_buckets, expected):
    assert cross.sparse_cross_hashed(KAT_BAGS, num_buckets, hash_key) == [expected]


def test_product_order_last_key_fastest():
    ids = cross.sparse_cross_hashed([[b"a", b"b"], [1, 2, 3]], 0)
    assert ids == [cross.cross_one(v, 0) for v in ([b"a", 1], [b"a", 2], [b"a", 3], [b"b", 1], [b"b", 2], [b"b", 3])]
    assert len(set(ids)) == 6


# ---------------------------------------------------------------- rules on hand-built inputs
def _dtypes():
    return {"a": "int32", "s": "string", "m": "int32", "ms": "string", "age": "int32", "g": "string", "f": "float32",
            "i": "int32"}


def test_sparse_keys_hash_before_dense_keys():
    age = fc.bucketized_column(fc.numeric_column("age"), [20, 40])
    g = fc.categorical_column_with_vocabulary_list("g", ["F", "M"])
    col = fc.crossed_column(["a", age, "m", g, "s"], 1000)
    spec = cross_spec(col, _dtypes(), {"m": 3})
    # categorical and multivalent raw keys (sparse) first, single-valued raw keys (dense) after, key order kept
    assert [k["name"] for k in spec["keys"]] == ["age_bucketized", "m", "g", "a", "s"]
    assert [k["width"] for k in spec["keys"]] == [1, 3, 1, 1, 1]
    assert spec["width"] == 3 and spec["hash_key"] == D and spec["num_buckets"] == 1000
    feats = {"a": np.array([7], np.int32), "age": np.array([25], np.int32), "m": np.array([[4, -1, 5]], np.int32),
             "g": np.array([b"M"], dtype=object), "s": np.array([b"x"], dtype=object)}
    ids = cross.transform_crossed(spec, feats)
    assert ids.tolist() == [[cross.cross_one([1, 4, 1, 7, b"x"], 1000), -1, cross.cross_one([1, 5, 1, 7, b"x"], 1000)]]


def test_single_valued_raw_keys_drop_nothing():
    spec = cross_spec(fc.crossed_column(["a", "s"], 0x7FFFFFFF), _dtypes())
    feats = {"a": np.array([-1, -7, 3], np.int32), "s": np.array([b"", b"q", b""], dtype=object)}
    ids = cross.transform_crossed(spec, feats)[:, 0]
    m64 = (1 << 64) - 1
    chain = lambda v, s: cross.fingerprint_cat64(cross.fingerprint_cat64(D, v & m64), fingerprint64(s)) % 0x7FFFFFFF
    assert ids.tolist() == [chain(-1, b""), chain(-7, b"q"), chain(3, b"")]
    assert cross.feature_fp(-1) == 0xFFFFFFFFFFFFFFFF


def test_multivalent_raw_padding_is_absent():
    spec = cross_spec(fc.crossed_column(["ms", "m"], 50), _dtypes(), {"ms": 2, "m": 2})
    feats = {"ms": np.array([[b"u", b""], [b"", b""]], dtype=object), "m": np.array([[-1, 9], [1, 2]], np.int32)}
    ids = cross.transform_crossed(spec, feats)
    assert ids[0].tolist() == [-1, cross.cross_one([b"u", 9], 50), -1, -1]
    assert (ids[1] == -1).all()                       # an empty bag empties the cross


def test_vocab_oov_without_buckets_is_crossed_as_minus_one():
    g0 = fc.categorical_column_with_vocabulary_list("g", ["F", "M"])
    g1 = fc.categorical_column_with_vocabulary_list("g", ["F", "M"], num_oov_buckets=3)
    feats = {"g": np.array([b"M", b"X", b""], dtype=object), "i": np.array([2, 2, 2], np.int32)}
    i = fc.categorical_column_with_identity("i", 4)
    ids0 = cross.transform_crossed(cross_spec(fc.crossed_column([g0, i], 97), _dtypes()), feats)[:, 0]
    assert ids0.tolist() == [cross.cross_one([1, 2], 97), cross.cross_one([-1, 2], 97), -1]
    ids1 = cross.transform_crossed(cross_spec(fc.crossed_column([g1, i], 97), _dtypes()), feats)[:, 0]
    oov = 2 + fingerprint64(b"X") % 3
    assert ids1.tolist() == [cross.cross_one([1, 2], 97), cross.cross_one([oov, 2], 97), -1]


def test_empty_categorical_bag_empties_the_cross():
    i = fc.categorical_column_with_identity("i", 4)
    spec = cross_spec(fc.crossed_column([i, "a"], 10), _dtypes())
    ids = cross.transform_crossed(spec, {"i": np.array([-1, 3], np.int32), "a": np.array([5, 5], np.int32)})[:, 0]
    assert ids.tolist() == [-1, cross.cross_one([3, 5], 10)]


def test_nested_crosses_are_flattened_and_named():
    age = fc.bucketized_column(fc.numeric_column("age"), [20, 40])
    g = fc.categorical_column_with_vocabulary_list("g", ["F", "M"])
    inner = fc.crossed_column(["s", age], 10, hash_key=5)
    outer = fc.crossed_column([g, inner, "a"], 20)
    assert inner.name == "age_bucketized_X_s"
    assert outer.name == "a_X_age_bucketized_X_g_X_s"
    assert fc.crossed_column([age, g], 7).name == "age_bucketized_X_g"
    assert fc.embedding_column(fc.crossed_column([age, g], 7), 4).name == "age_bucketized_X_g_embedding"
    spec = cross_spec(outer, _dtypes())
    assert [k["name"] for k in spec["keys"]] == ["g", "age_bucketized", "s", "a"]
    assert spec["hash_key"] == D                      # only the outer column's hash_key is used


def test_crossed_column_value_errors():
    h = fc.categorical_column_with_hash_bucket("s", 10)
    with pytest.raises(ValueError, match="hash_bucket_size must be > 1"):
        fc.crossed_column(["a", "s"], 0)
    with pytest.raises(ValueError, match="keys must be a list with length > 1"):
        fc.crossed_column(["a"], 10)
    with pytest.raises(ValueError, match="categorical_column_with_hash_bucket is not supported for crossing"):
        fc.crossed_column(["a", h], 10)
    with pytest.raises(ValueError, match="Unsupported key type"):
        fc.crossed_column(["a", fc.numeric_column("f")], 10)
    with pytest.raises(ValueError, match="sparse_cross takes only int64 and string"):
        cross_spec(fc.crossed_column(["a", "f"], 10), _dtypes())
    with pytest.raises(ValueError, match="at most 8"):
        cross_spec(fc.crossed_column(["a"] * 9, 10), _dtypes())


# ---------------------------------------------------------------- C ABI rejections (before any CUDA call)
def _create(cat, src, n_cat=None, n_src=None):
    lib = _lib.load()
    cats = (_lib.Column * max(len(cat), 1))(*cat)
    srcs = (_lib.Column * max(len(src), 1))(*src)
    cfg = _lib.Config()
    cfg.n_cat, cfg.cat = len(cat) if n_cat is None else n_cat, ctypes.cast(cats, ctypes.POINTER(_lib.Column))
    cfg.n_src, cfg.src = len(src) if n_src is None else n_src, ctypes.cast(srcs, ctypes.POINTER(_lib.Column))
    cfg.embedding_size, cfg.use_linear, cfg.max_batch = 4, 1, 16
    h = ctypes.c_void_p()
    rc = lib.dfm_create(ctypes.byref(cfg), ctypes.byref(h))
    return rc, (lib.dfm_last_error(None) or b"").decode()


def _col(kind, dtype="int32", nb=0, width=1, keys=None):
    c = _lib.Column()
    c.name, c.kind, c.dtype, c.num_buckets, c.width = b"c", _lib.COL_KIND[kind], _lib.DTYPE[dtype], nb, width
    if keys is not None:
        arr = (ctypes.c_int32 * len(keys))(*keys)
        _col.keep.append(arr)
        c.n_keys, c.keys = len(keys), ctypes.cast(arr, ctypes.POINTER(ctypes.c_int32))
    return c


_col.keep = []


@pytest.mark.parametrize("what,cat,src,code,msg", [
    ("hashed key", [("crossed", 10, [0, 1])], [("hash", "string", 5, 1), ("raw", "int32", 0, 1)], -1,
     "categorical_column_with_hash_bucket is not supported for crossing"),
    ("float raw key", [("crossed", 10, [0, 1])], [("raw", "float32", 0, 1), ("raw", "int32", 0, 1)], -1, "int32 or string"),
    ("key out of range", [("crossed", 10, [0, 2])], [("raw", "int32", 0, 1), ("raw", "int32", 0, 1)], -1, "outside [0, n_src)"),
    ("one key", [("crossed", 10, [0])], [("raw", "int32", 0, 1)], -1, "keys must be a list with length > 1"),
    ("no buckets", [("crossed", 0, [0, 1])], [("raw", "int32", 0, 1), ("raw", "int32", 0, 1)], -1, "hash_bucket_size"),
    ("too many keys", [("crossed", 10, list(range(9)))], [("raw", "int32", 0, 1)] * 9, -4, "at most 8 keys"),
    ("width over the limit", [("crossed", 10, [0, 1])], [("raw", "int32", 0, 17), ("raw", "int32", 0, 16)], -4,
     "too many value slots"),
    ("too many columns", [("crossed", 10, [0, 1])] * 33, [("raw", "int32", 0, 1)] * 32, -1, "too many feature columns"),
    ("raw model column", [("raw", 0, None)], [], -1, "allowed only as a source column"),
    ("crossed source", [("crossed", 10, [0, 1])], [("crossed", "int32", 5, 1), ("raw", "int32", 0, 1)], -1,
     "Unsupported key type"),
])
def test_abi_rejects(what, cat, src, code, msg):
    cats = [_col(k, "int32", nb, keys=keys) for k, nb, keys in cat]
    srcs = [_col(k, d, nb, width=w) for k, d, nb, w in src]
    rc, err = _create(cats, srcs)
    assert rc == code and msg in err, (what, rc, err)
