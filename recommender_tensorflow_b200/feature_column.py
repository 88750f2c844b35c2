"""Feature-column descriptors with the names and argument meaning of `tf.feature_column.*` as the
reference uses them (trainers/ml_100k.py:18-39).  They are plain descriptors: all arithmetic
(hashing, bucketizing, vocabulary lookup, embedding) happens in the CUDA library.
"""
import os
from collections import namedtuple

import numpy as np


class _Cat:
    kind = None

    def spec(self):
        raise NotImplementedError

    @property
    def source(self):
        return self.key


class NumericColumn(namedtuple("NumericColumn", ["key", "dtype"])):
    @property
    def name(self):
        return self.key


class HashedCategoricalColumn(namedtuple("HashedCategoricalColumn", ["key", "hash_bucket_size", "dtype"]), _Cat):
    kind = "hash"

    @property
    def name(self):
        return self.key

    @property
    def num_buckets(self):
        return self.hash_bucket_size

    def spec(self):
        return dict(name=self.name, source=self.key, kind="hash", dtype=self.dtype, num_buckets=self.hash_bucket_size)


class BucketizedColumn(namedtuple("BucketizedColumn", ["source_column", "boundaries"]), _Cat):
    kind = "bucketized"

    @property
    def name(self):
        return self.source_column.name + "_bucketized"

    @property
    def key(self):
        return self.source_column.key

    @property
    def num_buckets(self):
        return len(self.boundaries) + 1

    def spec(self):
        return dict(name=self.name, source=self.key, kind="bucketized", dtype=None, boundaries=list(self.boundaries),
                    num_buckets=self.num_buckets)


class VocabularyListCategoricalColumn(
        namedtuple("VocabularyListCategoricalColumn", ["key", "vocabulary_list", "num_oov_buckets", "dtype", "default_value"],
                   defaults=("string", -1)), _Cat):
    """dtype "string": vocabulary_list holds str; "int32": int keys (int64 range).  default_value -1 = dropped."""
    kind = "vocab"

    @property
    def name(self):
        return self.key

    @property
    def num_buckets(self):
        return len(self.vocabulary_list) + self.num_oov_buckets

    def spec(self):
        return dict(name=self.name, source=self.key, kind="vocab", dtype=self.dtype, vocab=list(self.vocabulary_list),
                    num_oov=self.num_oov_buckets, default_value=self.default_value, num_buckets=self.num_buckets)


class VocabularyFileCategoricalColumn(
        namedtuple("VocabularyFileCategoricalColumn",
                   ["key", "vocabulary_file", "vocabulary_size", "num_oov_buckets", "default_value", "dtype"]), _Cat):
    """The file is read when the engine resolves the column (spec()), as TF reads it at table initialisation."""
    kind = "vocab"

    @property
    def name(self):
        return self.key

    @property
    def num_buckets(self):
        return self.vocabulary_size + self.num_oov_buckets

    def spec(self):
        vocab = read_vocabulary_file(self.vocabulary_file, self.vocabulary_size, self.dtype, self.key)
        return dict(name=self.name, source=self.key, kind="vocab", dtype=self.dtype, vocab=vocab,
                    num_oov=self.num_oov_buckets, default_value=self.default_value, num_buckets=self.num_buckets)


class IdentityCategoricalColumn(namedtuple("IdentityCategoricalColumn", ["key", "num_buckets", "default_value"],
                                           defaults=(None,)), _Cat):
    kind = "identity"

    @property
    def name(self):
        return self.key

    def spec(self):
        return dict(name=self.name, source=self.key, kind="identity", dtype="int32", num_buckets=self.num_buckets,
                    default_value=self.default_value)


class CrossedColumn(namedtuple("CrossedColumn", ["keys", "hash_bucket_size", "hash_key"]), _Cat):
    """tf.feature_column.crossed_column (TF-1.12 feature_column.py `_CrossedColumn`).  Its ids are
    sparse_cross_hashed(inputs, num_buckets=hash_bucket_size, hash_key=hash_key or DEFAULT_HASH_KEY) over the
    Cartesian product of the constituents' bags; the engine resolves the keys into source columns
    (engine.cross_spec) and the transform runs on the device."""
    kind = "crossed"

    def leaf_keys(self):
        """`_collect_leaf_level_keys`: nested crosses flattened, key order kept."""
        out = []
        for k in self.keys:
            out += k.leaf_keys() if isinstance(k, CrossedColumn) else [k]
        return out

    @property
    def name(self):
        return "_X_".join(sorted(k if isinstance(k, str) else k.name for k in self.leaf_keys()))

    @property
    def num_buckets(self):
        return self.hash_bucket_size

    @property
    def source(self):
        return None

    def spec(self):
        raise TypeError("a crossed column is resolved against the raw feature dtypes: use engine.cross_spec")


# sparse_ops.sparse_cross_hashed's default hash_key (TF-1.12 python/ops/sparse_ops.py `_DEFAULT_HASH_KEY`)
DEFAULT_HASH_KEY = 0xDECAFCAFFE


class EmbeddingColumn(namedtuple("EmbeddingColumn", ["categorical_column", "dimension"])):
    @property
    def name(self):
        return self.categorical_column.name + "_embedding"


def _dtype_name(dtype):
    if dtype is None:
        return "string"
    s = getattr(dtype, "name", None) or str(dtype)
    s = s.replace("tf.", "").replace("<dtype: '", "").replace("'>", "")
    if s in ("string", "str", "bytes", "object"):
        return "string"
    if s.startswith("int"):
        return "int32"
    if s.startswith("float"):
        return "float32"
    raise ValueError("unsupported dtype %r" % (dtype,))


def categorical_column_with_hash_bucket(key, hash_bucket_size, dtype="string"):
    if hash_bucket_size is None or hash_bucket_size < 1:
        raise ValueError("hash_bucket_size must be at least 1. hash_bucket_size: {}, key: {}".format(hash_bucket_size, key))
    d = _dtype_name(dtype)
    if d == "float32":
        raise ValueError("dtype must be string or integer. dtype: {}, column_name: {}".format(dtype, key))
    return HashedCategoricalColumn(key, int(hash_bucket_size), d)


def numeric_column(key, dtype="float32"):
    return NumericColumn(key, _dtype_name(dtype))


def bucketized_column(source_column, boundaries):
    if not isinstance(source_column, NumericColumn):
        raise ValueError("source_column must be a column generated with numeric_column(). Given: {}".format(source_column))
    b = list(boundaries)
    if not b or any(b[i] >= b[i + 1] for i in range(len(b) - 1)):
        raise ValueError("boundaries must be a sorted list.")
    return BucketizedColumn(source_column, tuple(float(x) for x in b))


def _vocab_default(default_value, vocabulary_size, key):
    """default_value of a vocabulary column: -1 (dropped) or a vocabulary index.  TF does not check it and would gather
    outside the table; here anything else is rejected."""
    d = -1 if default_value is None else int(default_value)
    if d != -1 and not 0 <= d < vocabulary_size:
        raise ValueError("default_value {} must be -1 or in [0, {}), column_name: {}".format(default_value, vocabulary_size, key))
    return d


def _vocab_dtype_name(dtype, prefix):
    """fc_utils.assert_string_or_int: string or integer, integer raw features are int32 here."""
    try:
        d = _dtype_name(dtype)
    except ValueError:
        d = None
    if d not in ("string", "int32"):
        raise ValueError("{} dtype must be string or integer. dtype: {}.".format(prefix, dtype))
    return d


def categorical_column_with_vocabulary_list(key, vocabulary_list, dtype=None, default_value=-1, num_oov_buckets=0):
    """TF-1.12 tf.feature_column.categorical_column_with_vocabulary_list.  The vocabulary dtype is inferred from the
    list as np.array(vocabulary_list).dtype does; a repeated entry keeps its first index (TF's duplicate check is not
    reproduced)."""
    if vocabulary_list is None or len(vocabulary_list) < 1:
        raise ValueError("vocabulary_list {} must be non-empty, column_name: {}".format(vocabulary_list, key))
    if num_oov_buckets:
        if default_value != -1:
            raise ValueError("Can't specify both num_oov_buckets and default_value in {}.".format(key))
    if num_oov_buckets < 0:
        raise ValueError("Invalid num_oov_buckets {} in {}.".format(num_oov_buckets, key))
    # np.array(vocabulary_list).dtype without materialising the array: all integers -> int64, all str / bytes -> string
    if all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in vocabulary_list):
        vocab_dtype, vocab_np = "int32", "int64"
    elif all(isinstance(v, (str, bytes, np.str_, np.bytes_)) for v in vocabulary_list):
        vocab_dtype, vocab_np = "string", "string"
    else:
        raise ValueError("column_name: {} vocabulary dtype must be string or integer. dtype: {}.".format(
            key, np.array(vocabulary_list).dtype))
    if dtype is None:
        d = vocab_dtype
    else:
        d = _vocab_dtype_name(dtype, "column_name: {}".format(key))
        if d != vocab_dtype:
            raise ValueError("dtype {} and vocabulary dtype {} do not match, column_name: {}".format(dtype, vocab_np, key))
    if d == "string":
        vocab = tuple(v.decode() if isinstance(v, bytes) else str(v) for v in vocabulary_list)
    else:
        vocab = tuple(int(v) for v in vocabulary_list)
        if any(not -(1 << 63) <= v < 1 << 63 for v in vocab):
            raise ValueError("column_name: {} vocabulary holds a value outside int64".format(key))
    return VocabularyListCategoricalColumn(key, vocab, int(num_oov_buckets), d,
                                           _vocab_default(default_value, len(vocab), key))


def categorical_column_with_vocabulary_file(key, vocabulary_file, vocabulary_size=None, num_oov_buckets=0,
                                            default_value=None, dtype="string"):
    """TF-1.12 tf.feature_column.categorical_column_with_vocabulary_file: one key per line (read_vocabulary_file)."""
    if not vocabulary_file:
        raise ValueError("Missing vocabulary_file in {}.".format(key))
    if vocabulary_size is None:
        if not os.path.exists(vocabulary_file):
            raise ValueError("vocabulary_file in {} does not exist.".format(key))
        with open(vocabulary_file, "rb") as f:
            data = f.read()
        vocabulary_size = len(_split_lines(data))
    if vocabulary_size < 1:
        raise ValueError("Invalid vocabulary_size in {}.".format(key))
    if num_oov_buckets:
        if default_value is not None:
            raise ValueError("Can't specify both num_oov_buckets and default_value in {}.".format(key))
        if num_oov_buckets < 0:
            raise ValueError("Invalid num_oov_buckets {} in {}.".format(num_oov_buckets, key))
    d = _vocab_dtype_name(dtype, "column_name: {} vocabulary".format(key))
    return VocabularyFileCategoricalColumn(key, vocabulary_file, int(vocabulary_size),
                                           0 if num_oov_buckets is None else int(num_oov_buckets),
                                           _vocab_default(default_value, int(vocabulary_size), key), d)


def _split_lines(data):
    """io::InputBuffer::ReadLine over a whole file: lines end at '\n' (not part of the line), a trailing '\r' is
    removed, a last line without '\n' counts, nothing follows a final '\n'."""
    lines = data.split(b"\n")
    if lines[-1] == b"":
        lines.pop()
    return [ln[:-1] if ln.endswith(b"\r") else ln for ln in lines]


_SPACE = b" \t\n\v\f\r"


def _strto64(b):
    """strings::safe_strto64: surrounding whitespace allowed, an optional '-', decimal digits only, int64 range."""
    s = b.strip(_SPACE)
    digits = s[1:] if s.startswith(b"-") else s
    if not digits or not digits.isdigit():
        return None
    v = int(s)
    return v if -(1 << 63) <= v < (1 << 63) else None


def read_vocabulary_file(path, vocabulary_size, dtype, key):
    """The first vocabulary_size keys of a vocabulary file, as index_table_from_file / TextFileLineIterator reads them
    (TF-1.12): bytes for dtype "string", int for "int32" (each line parsed as int64).  Fewer lines than vocabulary_size,
    a repeated key or an unparsable integer line is a ValueError, as the table initialisation fails in TF."""
    with open(path, "rb") as f:
        lines = _split_lines(f.read())
    if len(lines) < vocabulary_size:
        raise ValueError("Invalid vocab_size in {}: vocabulary_size = {} but file {} has {} lines.".format(
            key, vocabulary_size, path, len(lines)))
    lines = lines[:vocabulary_size]
    if dtype == "string":
        vocab = lines
    else:
        vocab = []
        for i, ln in enumerate(lines):
            v = _strto64(ln)
            if v is None:
                raise ValueError("Field {!r} in line {} of {} is not a valid int64 (column {}).".format(ln, i, path, key))
            vocab.append(v)
    seen = set()
    for i, v in enumerate(vocab):
        if v in seen:
            raise ValueError("HashTable has different value for same key. Key {!r} (line {} of {}, column {}) repeats an "
                             "earlier line.".format(v, i, path, key))
        seen.add(v)
    return vocab


def categorical_column_with_identity(key, num_buckets, default_value=None):
    if num_buckets < 1:
        raise ValueError("num_buckets {} < 1, column_name {}".format(num_buckets, key))
    if default_value is not None and (default_value < 0 or default_value >= num_buckets):
        raise ValueError("default_value {} not in range [0, {}), column_name {}".format(default_value, num_buckets, key))
    return IdentityCategoricalColumn(key, int(num_buckets), None if default_value is None else int(default_value))


def crossed_column(keys, hash_bucket_size, hash_key=None):
    """TF-1.12 tf.feature_column.crossed_column, with its argument checks and messages."""
    if not hash_bucket_size or hash_bucket_size < 1:
        raise ValueError("hash_bucket_size must be > 1. hash_bucket_size: {}".format(hash_bucket_size))
    if not keys or len(keys) < 2:
        raise ValueError("keys must be a list with length > 1. Given: {}".format(keys))
    for key in keys:
        if not isinstance(key, (str, _Cat)):
            raise ValueError("Unsupported key type. All keys must be either string, or categorical column except "
                             "_HashedCategoricalColumn. Given: {}".format(key))
        if isinstance(key, HashedCategoricalColumn):
            raise ValueError("categorical_column_with_hash_bucket is not supported for crossing. Hashing before crossing "
                             "will increase probability of collision. Instead, use the feature name as a string. "
                             "Given: {}".format(key))
    if hash_key is not None and not 0 <= int(hash_key) < 1 << 64:
        raise ValueError("hash_key must be a uint64. Given: {}".format(hash_key))
    return CrossedColumn(tuple(keys), int(hash_bucket_size), None if hash_key is None else int(hash_key))


def embedding_column(categorical_column, dimension):
    if dimension is None or dimension < 1:
        raise ValueError("Invalid dimension {}.".format(dimension))
    return EmbeddingColumn(categorical_column, int(dimension))
