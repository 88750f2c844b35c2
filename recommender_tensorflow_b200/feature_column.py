"""Feature-column descriptors with the names and argument meaning of `tf.feature_column.*` as the
reference uses them (trainers/ml_100k.py:18-39).  They are plain descriptors: all arithmetic
(hashing, bucketizing, vocabulary lookup, embedding) happens in the CUDA library.
"""
from collections import namedtuple


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
        namedtuple("VocabularyListCategoricalColumn", ["key", "vocabulary_list", "num_oov_buckets"]), _Cat):
    kind = "vocab"

    @property
    def name(self):
        return self.key

    @property
    def num_buckets(self):
        return len(self.vocabulary_list) + self.num_oov_buckets

    def spec(self):
        return dict(name=self.name, source=self.key, kind="vocab", dtype="string", vocab=list(self.vocabulary_list),
                    num_oov=self.num_oov_buckets, num_buckets=self.num_buckets)


class IdentityCategoricalColumn(namedtuple("IdentityCategoricalColumn", ["key", "num_buckets"]), _Cat):
    kind = "identity"

    @property
    def name(self):
        return self.key

    def spec(self):
        return dict(name=self.name, source=self.key, kind="identity", dtype="int32", num_buckets=self.num_buckets)


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


def categorical_column_with_vocabulary_list(key, vocabulary_list, dtype=None, default_value=-1, num_oov_buckets=0):
    if not vocabulary_list:
        raise ValueError("vocabulary_list {} must be non-empty, column_name: {}".format(vocabulary_list, key))
    if num_oov_buckets < 0:
        raise ValueError("Invalid num_oov_buckets {} in {}.".format(num_oov_buckets, key))
    vocab = tuple(v.decode() if isinstance(v, bytes) else str(v) for v in vocabulary_list)
    return VocabularyListCategoricalColumn(key, vocab, int(num_oov_buckets))


def categorical_column_with_identity(key, num_buckets, default_value=None):
    if num_buckets < 1:
        raise ValueError("num_buckets {} < 1, column_name {}".format(num_buckets, key))
    return IdentityCategoricalColumn(key, int(num_buckets))


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
