"""CPU: vocabulary columns - TF-1.12's argument checks and messages, the vocabulary-file rules (product reader and the
oracle's independent reader), oracle ids for integer vocabularies, OOV buckets and default values, and the C ABI's
rejections (dfm_create validates vocabulary and identity columns before any CUDA call)."""
import ctypes
import json
import os

import numpy as np
import pytest

from oracle import vocab as ov
from oracle.farmhash import fingerprint64
from recommender_tensorflow_b200 import _lib
from recommender_tensorflow_b200 import feature_column as fc
from recommender_tensorflow_b200.engine import pack_vocabulary

KAT = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "hash_kat.json")))


def _write(tmp_path, data, name="vocab.txt"):
    p = tmp_path / name
    p.write_bytes(data)
    return str(p)


# ---------------------------------------------------------------- argument checks
def test_vocabulary_file_value_errors(tmp_path):
    path = _write(tmp_path, b"a\nb\nc\n")
    with pytest.raises(ValueError, match=r"^Missing vocabulary_file in k\.$"):
        fc.categorical_column_with_vocabulary_file("k", "")
    with pytest.raises(ValueError, match=r"^vocabulary_file in k does not exist\.$"):
        fc.categorical_column_with_vocabulary_file("k", str(tmp_path / "nope.txt"))
    # a given size skips the existence check (the file is read when the engine resolves the column)
    col = fc.categorical_column_with_vocabulary_file("k", str(tmp_path / "nope.txt"), vocabulary_size=3)
    assert col.num_buckets == 3
    with pytest.raises(ValueError, match=r"^Invalid vocabulary_size in k\.$"):
        fc.categorical_column_with_vocabulary_file("k", path, vocabulary_size=0)
    with pytest.raises(ValueError, match=r"^Can't specify both num_oov_buckets and default_value in k\.$"):
        fc.categorical_column_with_vocabulary_file("k", path, num_oov_buckets=2, default_value=0)
    with pytest.raises(ValueError, match=r"^Invalid num_oov_buckets -2 in k\.$"):
        fc.categorical_column_with_vocabulary_file("k", path, num_oov_buckets=-2)
    with pytest.raises(ValueError, match="dtype must be string or integer"):
        fc.categorical_column_with_vocabulary_file("k", path, dtype="float32")
    with pytest.raises(ValueError, match="must be -1 or in"):
        fc.categorical_column_with_vocabulary_file("k", path, default_value=3)


def test_vocabulary_file_column_shape(tmp_path):
    path = _write(tmp_path, b"a\nb\nc")
    col = fc.categorical_column_with_vocabulary_file("k", path, num_oov_buckets=4)
    assert col.name == "k" and col.vocabulary_size == 3 and col.num_buckets == 7 and col.default_value == -1
    assert fc.embedding_column(col, 4).name == "k_embedding"
    s = col.spec()
    assert s["vocab"] == [b"a", b"b", b"c"] and s["num_oov"] == 4 and s["dtype"] == "string"


def test_vocabulary_list_value_errors():
    with pytest.raises(ValueError, match="must be non-empty"):
        fc.categorical_column_with_vocabulary_list("k", [])
    with pytest.raises(ValueError, match=r"^Can't specify both num_oov_buckets and default_value in k\.$"):
        fc.categorical_column_with_vocabulary_list("k", ["a"], num_oov_buckets=1, default_value=0)
    with pytest.raises(ValueError, match=r"^Invalid num_oov_buckets -1 in k\.$"):
        fc.categorical_column_with_vocabulary_list("k", ["a"], num_oov_buckets=-1)
    with pytest.raises(ValueError, match="dtype string and vocabulary dtype int64 do not match, column_name: k"):
        fc.categorical_column_with_vocabulary_list("k", [1, 2], dtype="string")
    with pytest.raises(ValueError, match="do not match, column_name: k"):
        fc.categorical_column_with_vocabulary_list("k", ["a"], dtype="int64")
    with pytest.raises(ValueError, match="must be -1 or in"):
        fc.categorical_column_with_vocabulary_list("k", ["a", "b"], default_value=2)
    with pytest.raises(ValueError, match="must be -1 or in"):
        fc.categorical_column_with_vocabulary_list("k", ["a", "b"], default_value=-2)


def test_vocabulary_list_dtype_inference_and_default():
    c = fc.categorical_column_with_vocabulary_list("k", [10, -3, 2 ** 40])
    assert c.dtype == "int32" and c.vocabulary_list == (10, -3, 2 ** 40) and c.default_value == -1
    assert c.spec()["dtype"] == "int32"
    c = fc.categorical_column_with_vocabulary_list("k", ["a", "b"], default_value=1)
    assert c.dtype == "string" and c.default_value == 1 and c.num_buckets == 2
    c = fc.categorical_column_with_vocabulary_list("k", [b"x"], dtype="string")
    assert c.vocabulary_list == ("x",)


def test_identity_default_value_check():
    with pytest.raises(ValueError, match=r"^default_value 4 not in range \[0, 4\), column_name i$"):
        fc.categorical_column_with_identity("i", 4, default_value=4)
    with pytest.raises(ValueError, match=r"^default_value -1 not in range \[0, 4\), column_name i$"):
        fc.categorical_column_with_identity("i", 4, default_value=-1)
    assert fc.categorical_column_with_identity("i", 4, default_value=3).spec()["default_value"] == 3
    assert fc.categorical_column_with_identity("i", 4).spec()["default_value"] is None


# ---------------------------------------------------------------- file rules
READERS = [lambda p, n, d: fc.read_vocabulary_file(p, n, d, "k"), lambda p, n, d: ov.read_vocabulary_file(p, n, d)]


@pytest.mark.parametrize("read", READERS, ids=["product", "oracle"])
def test_file_line_rules(tmp_path, read):
    path = _write(tmp_path, b"a\r\nb\n\nc\r\r\nlast")
    assert read(path, 5, "string") == [b"a", b"b", b"", b"c\r", b"last"]
    assert read(path, 2, "string") == [b"a", b"b"]                  # vocabulary_size truncates
    with pytest.raises(ValueError, match="Invalid vocab_size"):
        read(path, 6, "string")
    assert read(_write(tmp_path, b"x\ny\n", "t.txt"), 2, "string") == [b"x", b"y"]   # nothing after a final newline
    with pytest.raises(ValueError, match="same key"):
        read(_write(tmp_path, b"x\ny\nx\n", "d.txt"), 3, "string")
    assert read(_write(tmp_path, b"x\ny\nx\n", "d2.txt"), 2, "string") == [b"x", b"y"]   # duplicate beyond the size


def test_file_line_count_default(tmp_path):
    assert fc.categorical_column_with_vocabulary_file("k", _write(tmp_path, b"a\nb\nc\n")).vocabulary_size == 3
    assert fc.categorical_column_with_vocabulary_file("k", _write(tmp_path, b"a\nb\nc", "u.txt")).vocabulary_size == 3
    assert fc.categorical_column_with_vocabulary_file("k", _write(tmp_path, b"a\n\n\n", "e.txt")).vocabulary_size == 3


@pytest.mark.parametrize("read", READERS, ids=["product", "oracle"])
def test_file_int_rules(tmp_path, read):
    # safe_strto64: surrounding whitespace is allowed, a '+' sign, inner spaces, hex and overflow are not
    path = _write(tmp_path, b"7\n -12 \n\t3\r\n9223372036854775807\n-9223372036854775808\n")
    assert read(path, 5, "int32") == [7, -12, 3, 2 ** 63 - 1, -2 ** 63]
    for bad in (b"+5", b"1 2", b"", b"0x10", b"9223372036854775808", b"- 5", b"1.0", b"a"):
        p = _write(tmp_path, b"1\n" + bad + b"\n3\n", "bad.txt")
        with pytest.raises(ValueError, match="line 1"):
            read(p, 3, "int32")
    with pytest.raises(ValueError, match="same key"):
        read(_write(tmp_path, b"5\n 5\n", "dup.txt"), 2, "int32")


def test_safe_strto64_agree():
    cases = [b"0", b"-0", b"  42", b"42  ", b"\v42\f", b"--1", b"-", b" ", b"12a", b"007", b"-9223372036854775809"]
    for c in cases:
        assert fc._strto64(c) == ov.safe_strto64(c), c


# ---------------------------------------------------------------- oracle ids
def test_oracle_string_ids():
    voc = ["F", "M", "a-key-longer-than-16-bytes"]
    vals = np.array([b"M", b"", b"X", b"a-key-longer-than-16-bytes", b"F"], dtype=object)
    assert ov.vocab_lookup(vals, voc).tolist() == [1, -1, -1, 2, 0]
    assert ov.vocab_lookup(vals, voc, default_value=2).tolist() == [1, -1, 2, 2, 0]
    assert ov.vocab_lookup(vals, voc, num_oov=5).tolist() == [1, -1, 3 + fingerprint64(b"X") % 5, 2, 0]


def test_oracle_oov_pinned_by_fingerprint_vectors():
    kat = KAT["fingerprint64"]
    assert len(kat) >= 4
    vals = np.array([k.encode() for k in kat], dtype=object)
    want = [1 + fp % 7 for fp in kat.values()]
    assert ov.vocab_lookup(vals, ["zz-not-a-kat-key"], num_oov=7).tolist() == want
    # an int key's OOV bucket is that of its decimal string (AsString), pinned by TF's hashed int vectors
    for v in KAT["hash_bucket_int32"]:
        got = ov.vocab_lookup(np.array(v["keys"], np.int32), [-99], num_oov=v["num_buckets"], dtype="int32")
        assert (got - 1).tolist() == v["ids"]


def test_oracle_int_ids():
    voc = [5, -7, 2 ** 40, 0]
    vals = np.array([5, -1, 0, 3, -7, 123456], np.int32)
    assert ov.vocab_lookup(vals, voc, dtype="int32").tolist() == [0, -1, 3, -1, 1, -1]
    assert ov.vocab_lookup(vals, voc, default_value=2, dtype="int32").tolist() == [0, -1, 3, 2, 1, 2]
    got = ov.vocab_lookup(vals, voc, num_oov=3, dtype="int32").tolist()
    assert got == [0, -1, 3, 4 + fingerprint64(b"3") % 3, 1, 4 + fingerprint64(b"123456") % 3]


def test_oracle_first_occurrence_wins_and_defaults_unchanged():
    assert ov.vocab_lookup(np.array([b"a"], dtype=object), ["a", "b", "a"]).tolist() == [0]
    from oracle import transforms
    vals = np.array([b"F", b"M", b"X", b""], dtype=object)
    assert ov.vocab_lookup(vals, ["F", "M"], 1).tolist() == transforms.vocab_lookup(vals, ["F", "M"], 1).tolist()


def test_oracle_identity_default():
    x = np.array([-1, 0, 3, 4, -5, 100], np.int32)
    assert ov.identity(x, 4, 2).tolist() == [-1, 0, 3, 2, 2, 2]
    with pytest.raises(ValueError):
        ov.identity(x, 4)


# ---------------------------------------------------------------- C ABI rejections (before any CUDA call)
_keep = []


def _vcol(dtype="string", vocab=("a", "b"), ints=None, num_oov=0, default=None, kind="vocab", nb=0, offsets=None,
          size=None):
    c = _lib.Column()
    c.name, c.kind, c.dtype, c.num_buckets = b"v", _lib.COL_KIND[kind], _lib.DTYPE[dtype], nb
    if kind == "vocab":
        if vocab is not None:
            data, offs = pack_vocabulary(list(vocab), "string")
            if offsets is not None:
                offs = np.array(offsets, np.int64)
            _keep.append((data, offs))
            c.vocab_data, c.vocab_offsets = data.ctypes.data, offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
        if ints is not None:
            arr = np.array(ints, np.int64)
            _keep.append(arr)
            c.vocab_int = arr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
        c.vocab_size = len(vocab if vocab is not None else ints) if size is None else size
        c.num_oov = num_oov
    if default is not None:
        c.default_value, c.has_default = default, 1
    return c


def _create(cat, src=()):
    lib = _lib.load()
    cats = (_lib.Column * max(len(cat), 1))(*cat)
    srcs = (_lib.Column * max(len(src), 1))(*src)
    cfg = _lib.Config()
    cfg.n_cat, cfg.cat = len(cat), ctypes.cast(cats, ctypes.POINTER(_lib.Column))
    cfg.n_src, cfg.src = len(src), ctypes.cast(srcs, ctypes.POINTER(_lib.Column))
    cfg.embedding_size, cfg.use_linear, cfg.max_batch = 4, 1, 16
    h = ctypes.c_void_p()
    rc = lib.dfm_create(ctypes.byref(cfg), ctypes.byref(h))
    err = (lib.dfm_last_error(None) or b"").decode()
    if rc == 0:
        lib.dfm_destroy(h)
    return rc, err


@pytest.mark.parametrize("what,col,code,msg", [
    ("int raw, string vocab", dict(dtype="int32"), -1, "dtype int32 and vocabulary dtype string do not match"),
    ("string raw, int vocab", dict(vocab=None, ints=[1, 2]), -1, "dtype string and vocabulary dtype int64 do not match"),
    ("int raw, no vocab", dict(dtype="int32", vocab=None, ints=None, size=2), -1, "needs vocab_int"),
    ("float raw", dict(dtype="float32"), -4, "needs string or int32 input"),
    ("empty vocab", dict(size=0), -1, "vocab_size >= 1"),
    ("default out of range", dict(default=2), -1, "must be -1 or in [0, vocab_size)"),
    ("default below -1", dict(default=-2), -1, "must be -1 or in [0, vocab_size)"),
    ("default and oov", dict(default=0, num_oov=2), -1, "Can't specify both num_oov_buckets and default_value"),
    ("negative oov", dict(num_oov=-1), -1, "Invalid num_oov_buckets"),
    ("offsets not monotone", dict(vocab=("ab", "c"), offsets=[0, 2, 1]), -1, "not monotone"),
    ("offsets below zero", dict(vocab=("ab", "c"), offsets=[-1, 2, 3]), -1, "start at >= 0"),
    ("identity default out of range", dict(kind="identity", dtype="int32", nb=4, default=4), -1,
     "default_value 4 not in range [0, 4)"),
    ("identity negative default", dict(kind="identity", dtype="int32", nb=4, default=-1), -1,
     "default_value -1 not in range [0, 4)"),
])
def test_abi_rejects(what, col, code, msg):
    rc, err = _create([_vcol(**col)])
    assert rc == code and msg in err, (what, rc, err)
    rc, err = _create([_vcol(kind="identity", dtype="int32", nb=3)], [_vcol(**col)])        # as a cross constituent
    assert rc == code and msg in err, (what, rc, err)


def test_abi_rejects_vocabulary_bytes_beyond_int32_offsets():
    data = np.zeros(16, np.uint8)
    offs = np.array([0, 2 ** 30, 2 ** 31], np.int64)      # never read: the sizes alone are rejected
    c = _vcol()
    c.vocab_data, c.vocab_offsets, c.vocab_size = data.ctypes.data, offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), 2
    rc, err = _create([c])
    assert rc == -4 and "2^31 - 1 bytes" in err


def test_abi_accepts_valid_vocabularies_up_to_the_device():
    # a valid configuration passes the vocabulary checks and fails (without a GPU) or succeeds only at the device
    rc, err = _create([_vcol(), _vcol(dtype="int32", vocab=None, ints=[3, 4], default=1),
                       _vcol(kind="identity", dtype="int32", nb=4, default=0)])
    assert "vocab" not in err and "default_value" not in err, err
