"""ORACLE (test infrastructure): tf.feature_column.crossed_column ids.

Restates TF-1.12 `_CrossedColumn._transform_feature` -> `sparse_ops.sparse_cross_hashed` (core/kernels/sparse_cross_op.cc,
HashCrosser): for every combination of one value from each constituent's bag (Cartesian product),

  h = hash_key;  for each constituent value v, in key order:  h = FingerprintCat64(h, f(v))
  id = h % num_buckets                       (num_buckets == 0: h % INT64_MAX)
  f(v): string -> Fingerprint64(bytes);  int -> (uint64)(int64)v;  categorical column -> (uint64)(int64)id

The hash chain is pinned by the upstream vectors of python/kernel_tests/sparse_cross_op_test.py
(tests/test_oracle_cross.py).  Which values are present (restated from TF 1.12, not pinned by an upstream vector):
padding of a multivalent raw key is absent, a single-valued raw key drops nothing, a categorical key drops what its
column drops except a vocabulary key's unknown-string id -1.

A crossed spec (engine.cross_spec) is {"kind": "crossed", "num_buckets", "hash_key", "keys": [source specs in hashing
order], "width"}; a source spec has kind "raw" | "bucketized" | "vocab" | "identity", "source", "dtype", "width".
"""
import itertools

import numpy as np

from . import transforms
from .farmhash import fingerprint64

M64 = (1 << 64) - 1
K_MUL = 0xC6A4A7935BD1E995
INT64_MAX = (1 << 63) - 1
DEFAULT_HASH_KEY = 0xDECAFCAFFE


def _shift_mix(x):
    return x ^ (x >> 47)


def fingerprint_cat64(fp1, fp2):
    """TF core/lib/hash/hash.h FingerprintCat64."""
    r = fp1 ^ K_MUL
    r ^= (_shift_mix((fp2 * K_MUL) & M64) * K_MUL) & M64
    r = (r * K_MUL) & M64
    r = (_shift_mix(r) * K_MUL) & M64
    return _shift_mix(r)


def feature_fp(v):
    """f(v) of one constituent value: bytes are fingerprinted, ints sign-extended to 64 bits."""
    if isinstance(v, (bytes, str)):
        return fingerprint64(v if isinstance(v, bytes) else v.encode())
    return int(v) & M64


def cross_one(values, num_buckets, hash_key=DEFAULT_HASH_KEY):
    """One crossed id of one combination (values in hashing order)."""
    h = hash_key
    for v in values:
        h = fingerprint_cat64(h, feature_fp(v))
    return h % num_buckets if num_buckets > 0 else h % INT64_MAX


def sparse_cross_hashed(bags, num_buckets=0, hash_key=None):
    """bags: one list of values per constituent (already without absent values) -> crossed ids, Cartesian-product order
    (last constituent fastest)."""
    hk = DEFAULT_HASH_KEY if hash_key is None else hash_key
    return [cross_one(c, num_buckets, hk) for c in itertools.product(*bags)]


def _slots(spec, features):
    """-> [B, width] object array of the constituent's values, None where absent."""
    w = int(spec.get("width", 1))
    raw = features[spec["source"]]
    if spec["kind"] == "raw":
        if spec["dtype"] == "string":
            vals = np.array(transforms.unpack_strings(raw) if isinstance(raw, tuple) else
                            [v if isinstance(v, bytes) else str(v).encode() for v in np.asarray(raw, dtype=object).reshape(-1)],
                            dtype=object).reshape(-1, w)
            if w > 1:
                vals = np.where(np.vectorize(len, otypes=[np.int64])(vals) == 0, None, vals)
            return vals
        vals = np.asarray(raw).astype(np.int64).reshape(-1, w).astype(object)
        if w > 1:
            vals = np.where(vals == -1, None, vals)
        return vals
    flat = dict(spec, width=1)
    if isinstance(raw, tuple):
        src = raw
    else:
        src = np.asarray(raw, dtype=object if spec["kind"] == "vocab" else None).reshape(-1)
    ids = transforms.transform_column(flat, {spec["source"]: src}).astype(np.int64).reshape(-1, w).astype(object)
    if spec["kind"] == "vocab":
        # '' is dropped before the lookup; an unknown string without OOV buckets keeps the id -1 (default_value)
        strs = transforms.unpack_strings(src)
        empty = np.array([len(v) == 0 for v in strs]).reshape(-1, w)
        return np.where(empty, None, ids)
    return np.where(ids == -1, None, ids)


def transform_crossed(spec, features):
    """ids [B, width] int32 of a crossed spec; -1 = absent combination."""
    keys = spec["keys"]
    cols = [_slots(k, features) for k in keys]
    B = cols[0].shape[0]
    widths = [int(k.get("width", 1)) for k in keys]
    nb, hk = int(spec["num_buckets"]), int(spec.get("hash_key") or DEFAULT_HASH_KEY)
    out = np.full((B, int(np.prod(widths))), -1, dtype=np.int64)
    for b in range(B):
        for j, combo in enumerate(itertools.product(*[range(w) for w in widths])):
            vals = [cols[i][b, d] for i, d in enumerate(combo)]
            if any(v is None for v in vals):
                continue
            out[b, j] = cross_one(vals, nb, hk)
    return out.astype(np.int32)


def transform(cat_specs, features, use_c=True):
    """oracle.transforms.transform with crossed columns: ids [B, n_slots] in the order of cat_specs."""
    cols = []
    for s in cat_specs:
        if s["kind"] == "crossed":
            cols.append(transform_crossed(s, features))
        else:
            cols.append(transforms.transform([s], features, use_c))
    return np.concatenate(cols, axis=1)
