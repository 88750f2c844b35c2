"""ORACLE (test infrastructure): vocabulary columns with integer keys, vocabulary files and default values.

Extends oracle.transforms / oracle.cross (whose results for string lists without a default are unchanged):

  vocab     index of the key in the vocabulary (first occurrence), else
            vocab_size + Fingerprint64(key or AsString(key)) mod num_oov   when num_oov > 0
            default_value (-1 = dropped)                                  otherwise
            '' (string) / -1 (int) -> empty bag before the lookup
  identity  id = value; -1 -> empty; outside [0, N) -> default_value, or a runtime error without one

The vocabulary-file reader restates TF-1.12 index_table_from_file (TextFileLineIterator over io::InputBuffer::ReadLine,
keys parsed with strings::safe_strto64 for integer columns) independently of the product's reader.

A vocabulary spec may carry "dtype": "string" | "int32" and "default_value"; an identity spec "default_value".
"""
import numpy as np

from . import cross, transforms
from .farmhash import fingerprint64

_WHITESPACE = frozenset(b" \t\n\v\f\r")        # isspace() in the C locale


def read_lines(data):
    """Lines of a file as ReadLine yields them: up to '\\n', one trailing '\\r' dropped, a last unterminated line kept."""
    out, start = [], 0
    while start < len(data):
        end = data.find(b"\n", start)
        if end < 0:
            end = len(data)
        line = data[start:end]
        if line[-1:] == b"\r":
            line = line[:-1]
        out.append(line)
        start = end + 1
    return out


def safe_strto64(b):
    """strings::safe_strto64: skip spaces, optional '-', at least one digit, skip spaces, nothing else; int64 range."""
    i, n = 0, len(b)
    while i < n and b[i] in _WHITESPACE:
        i += 1
    sign = 1
    if i < n and b[i] == ord("-"):
        sign, i = -1, i + 1
    if i >= n or not 48 <= b[i] <= 57:
        return None
    v = 0
    while i < n and 48 <= b[i] <= 57:
        v = v * 10 + (b[i] - 48)
        i += 1
    while i < n and b[i] in _WHITESPACE:
        i += 1
    if i != n:
        return None
    v *= sign
    return v if -(1 << 63) <= v < (1 << 63) else None


def read_vocabulary_file(path, vocabulary_size=None, dtype="string"):
    """-> list of keys (bytes or int).  Too few lines, a repeated key or an unparsable int line -> ValueError."""
    with open(path, "rb") as f:
        lines = read_lines(f.read())
    if vocabulary_size is None:
        vocabulary_size = len(lines)
    if len(lines) < vocabulary_size:
        raise ValueError("Invalid vocab_size: %d lines < %d" % (len(lines), vocabulary_size))
    keys = lines[:vocabulary_size]
    if dtype != "string":
        parsed = [safe_strto64(k) for k in keys]
        for i, v in enumerate(parsed):
            if v is None:
                raise ValueError("line %d (%r) is not a valid int64" % (i, keys[i]))
        keys = parsed
    if len(set(keys)) != len(keys):
        raise ValueError("HashTable has different value for same key")
    return keys


def _key(v):
    return v if isinstance(v, (bytes, int)) else (v.encode() if isinstance(v, str) else int(v))


def vocab_lookup(values, vocab, num_oov=0, default_value=-1, dtype="string"):
    """ids of a flat column (object array of bytes / (data, offsets) for strings, int32 array for ints)."""
    table = {}
    for i, v in enumerate(vocab):
        table.setdefault(_key(v), i)
    dflt = -1 if default_value is None else int(default_value)
    if dtype == "string":
        vals = transforms.unpack_strings(values)
        empty = [len(v) == 0 for v in vals]
        as_bytes = vals
    else:
        vals = [int(v) for v in np.asarray(values).reshape(-1)]
        empty = [v == -1 for v in vals]
        as_bytes = [str(v).encode() for v in vals]
    out = np.empty(len(vals), dtype=np.int32)
    for i, v in enumerate(vals):
        if empty[i]:
            out[i] = -1
        elif v in table:
            out[i] = table[v]
        elif num_oov > 0:
            out[i] = len(vocab) + fingerprint64(as_bytes[i]) % num_oov
        else:
            out[i] = dflt
    return out


def identity(x, num_buckets, default_value=None):
    if default_value is None:
        return transforms.identity(x, num_buckets)
    x = np.asarray(x).astype(np.int64)
    out = np.where((x != -1) & ((x < 0) | (x >= num_buckets)), int(default_value), x)
    return out.astype(np.int32)


def transform_column(spec, features, use_c=True):
    raw = features[spec.get("source", spec["name"])]
    if spec["kind"] == "vocab":
        return vocab_lookup(raw, spec["vocab"], spec.get("num_oov", 0), spec.get("default_value", -1),
                            spec.get("dtype", "string"))
    if spec["kind"] == "identity":
        return identity(raw, spec["num_buckets"], spec.get("default_value"))
    return transforms.transform_column(spec, features, use_c)


def _slots(spec, features):
    """cross._slots with integer vocabularies and default values: -> [B, width] object array, None where absent."""
    if spec["kind"] == "raw":
        return cross._slots(spec, features)
    w = int(spec.get("width", 1))
    raw = features[spec["source"]]
    is_str = spec["kind"] == "vocab" and spec.get("dtype", "string") == "string"
    src = raw if isinstance(raw, tuple) else np.asarray(raw, dtype=object if is_str else None).reshape(-1)
    ids = transform_column(dict(spec, width=1), {spec["source"]: src}).astype(np.int64).reshape(-1, w).astype(object)
    if spec["kind"] == "vocab":
        # the empty value is dropped before the lookup; an unknown key without OOV buckets crosses as default_value
        if is_str:
            empty = np.array([len(v) == 0 for v in transforms.unpack_strings(src)])
        else:
            empty = np.asarray(src).astype(np.int64) == -1
        return np.where(empty.reshape(-1, w), None, ids)
    return np.where(ids == -1, None, ids)


def transform_crossed(spec, features):
    cols = [_slots(k, features) for k in spec["keys"]]
    B = cols[0].shape[0]
    widths = [int(k.get("width", 1)) for k in spec["keys"]]
    nb, hk = int(spec["num_buckets"]), int(spec.get("hash_key") or cross.DEFAULT_HASH_KEY)
    out = np.full((B, int(np.prod(widths))), -1, dtype=np.int64)
    for b in range(B):
        for j, combo in enumerate(np.ndindex(*widths)):
            vals = [cols[i][b, d] for i, d in enumerate(combo)]
            if any(v is None for v in vals):
                continue
            out[b, j] = cross.cross_one(vals, nb, hk)
    return out.astype(np.int32)


def transform(cat_specs, features, use_c=True):
    """ids [B, n_slots] int32 in the order of cat_specs, every column kind."""
    cols = []
    for s in cat_specs:
        if s["kind"] == "crossed":
            cols.append(transform_crossed(s, features))
            continue
        w = int(s.get("width", 1))
        src = s.get("source", s["name"])
        feats = features if w == 1 else {src: transforms._flat(features[src])}
        cols.append(transform_column(s, feats, use_c).reshape(-1, w))
    return np.concatenate(cols, axis=1)
