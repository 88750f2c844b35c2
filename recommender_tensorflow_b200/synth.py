"""Synthetic inputs with the shape of the reference's data (SURVEY.md §8d).  numpy only.

ML-100K-shaped: the 42-column schema of trainers/ml_100k.py:3-15 as written by
src/data/ml_100k.py:58-96,152-157 (user attributes are functions of user_id, item attributes of
item_id).  Criteo-shaped: 26 categorical 8-hex-char keys + 13 float32 numerics + label.
"""
import numpy as np

OCCUPATIONS = ["administrator", "artist", "doctor", "educator", "engineer", "entertainment", "executive",
               "healthcare", "homemaker", "lawyer", "librarian", "marketing", "none", "other", "programmer",
               "retired", "salesman", "scientist", "student", "technician", "writer"]
GENRE = ("unknown,action,adventure,animation,children,comedy,crime,documentary,drama,fantasy,"
         "filmnoir,horror,musical,mystery,romance,scifi,thriller,war,western").split(",")
SEED = 20260101


class ML100K:
    """Deterministic user / item attribute tables + a sampler of interaction rows."""

    def __init__(self, seed=SEED, n_users=943, n_items=1682):
        rng = np.random.default_rng(seed)
        self.n_users, self.n_items = n_users, n_items
        self.age = rng.integers(7, 74, n_users + 1).astype(np.int32)
        self.gender = np.where(rng.random(n_users + 1) < 0.29, b"F", b"M").astype(object)
        self.occupation = np.array([OCCUPATIONS[i].encode() for i in rng.integers(0, len(OCCUPATIONS), n_users + 1)], dtype=object)
        self.zipcode = np.array([b"%05d" % z for z in rng.integers(0, 100000, n_users + 1)], dtype=object)
        self.release_year = rng.integers(1922, 1999, n_items + 1).astype(np.int32)
        g = (rng.random((n_items + 1, len(GENRE))) < 0.09)
        none = ~g.any(axis=1)
        g[none, rng.integers(1, len(GENRE), int(none.sum()))] = True
        self.genres = g.astype(np.int32)

    def batch(self, batch_size, rng, cutoff=5):
        """-> (features dict consumed by get_feature_columns(), labels float32 [B])."""
        u = rng.integers(1, self.n_users + 1, batch_size).astype(np.int32)
        i = rng.integers(1, self.n_items + 1, batch_size).astype(np.int32)
        rating = rng.choice(np.arange(1, 6), size=batch_size, p=[.061, .114, .271, .342, .212]).astype(np.int32)
        feats = {"user_id": u, "item_id": i, "age": self.age[u], "gender": self.gender[u],
                 "occupation": self.occupation[u], "zipcode": self.zipcode[u], "release_year": self.release_year[i]}
        for j, gname in enumerate(GENRE):
            feats[gname] = np.ascontiguousarray(self.genres[i, j])
        return feats, (rating >= cutoff).astype(np.float32)

    def fast_batch(self, batch_size, rng, cutoff=5):
        """Same as batch() but string columns come pre-packed as (uint8 bytes, int32 offsets)."""
        feats, y = self.batch(batch_size, rng, cutoff)
        for key in ("gender", "occupation", "zipcode"):
            feats[key] = pack_strings(feats[key])
        return feats, y


def pack_strings(values):
    lens = np.fromiter((len(v) for v in values), dtype=np.int64, count=len(values))
    offs = np.zeros(len(values) + 1, dtype=np.int32)
    np.cumsum(lens, out=offs[1:])
    data = np.frombuffer(b"".join(values) or b"\0", dtype=np.uint8).copy()
    return data, offs


HEX = np.frombuffer(b"0123456789abcdef", dtype=np.uint8)


def hex8(keys_u32):
    """uint32 keys -> packed 8-hex-char ASCII strings (bytes [n*8], offsets [n+1])."""
    k = np.asarray(keys_u32, dtype=np.uint32)
    out = np.empty((k.shape[0], 8), dtype=np.uint8)
    for j in range(8):
        out[:, j] = HEX[(k >> np.uint32(4 * (7 - j))) & np.uint32(15)]
    return out.reshape(-1), (np.arange(k.shape[0] + 1, dtype=np.int64) * 8).astype(np.int32)


def criteo_batch(batch_size, rng, n_cat=26, n_num=13, zipf_alpha=None, key_space=1 << 32):
    """Criteo-shaped batch: C1..C26 8-hex keys (uniform over key_space or Zipf), I1..I13 = log1p(counts)."""
    feats = {}
    for f in range(n_cat):
        if zipf_alpha:
            k = (rng.zipf(zipf_alpha, batch_size).astype(np.uint64) * np.uint64(2654435761 + 2 * f)) % np.uint64(key_space)
        else:
            k = rng.integers(0, key_space, batch_size, dtype=np.uint64)
        feats["C%d" % (f + 1)] = hex8(k.astype(np.uint32))
    for j in range(n_num):
        feats["I%d" % (j + 1)] = np.log1p(rng.poisson(3.0 + j, batch_size)).astype(np.float32)
    y = (rng.random(batch_size) < 0.25).astype(np.float32)
    return feats, y


def _float_text(x, form):
    """float32 x printed in one of several forms that all read back as x (form 0..4)"""
    if form == 0:
        return np.format_float_positional(x, unique=True, trim="-")       # shortest repr: 1.0986123, 0
    if form == 1:
        return "%.9g" % x
    if form == 2:
        return "%d" % x if float(x).is_integer() else "%.9g" % x
    if form == 3:
        return "%.8e" % x                                                   # 1.09861231e+00
    return np.format_float_scientific(x, unique=True, exp_digits=1)         # 1.0986123e+0


def criteo_tsv_schema(n_cat=26, n_num=13):
    """(columns, record_defaults) of a Criteo TSV line: label, I1..I13 ([0.0]), C1..C26 ([""])"""
    cols = ["label"] + ["I%d" % (j + 1) for j in range(n_num)] + ["C%d" % (f + 1) for f in range(n_cat)]
    return cols, [[0]] + [[0.0]] * n_num + [[""]] * n_cat


def write_criteo_tsv(path, n_rows, seed, empty_frac=0.05, n_cat=26, n_num=13):
    """Criteo-style raw text: per line the 0/1 label, I1..I13, C1..C26, tab-separated, no header.  The numerics are the
    float32 values criteo_batch draws, printed in a mix of forms (shortest repr, %.9g, integers, exponent forms); the
    categoricals are its 8-hex-char keys.  A share empty_frac of the numeric and categorical fields is left empty."""
    rng = np.random.default_rng(seed)
    feats, y = criteo_batch(n_rows, rng, n_cat, n_num)
    forms = rng.integers(0, 5, (n_rows, n_num))
    empty = rng.random((n_rows, n_num + n_cat)) < empty_frac
    cats = [feats["C%d" % (f + 1)][0].reshape(n_rows, 8).tobytes() for f in range(n_cat)]
    lines = []
    for i in range(n_rows):
        row = ["%d" % y[i]]
        for j in range(n_num):
            row.append("" if empty[i, j] else _float_text(feats["I%d" % (j + 1)][i], forms[i, j]))
        for f in range(n_cat):
            row.append("" if empty[i, n_num + f] else cats[f][8 * i:8 * i + 8].decode())
        lines.append("\t".join(row))
    with open(path, "w", newline="") as fh:
        fh.write("\n".join(lines) + "\n")


def criteo_columns(buckets_per_field, n_cat=26, n_num=13):
    from . import feature_column as fc
    cats = [fc.categorical_column_with_hash_bucket("C%d" % (f + 1), buckets_per_field) for f in range(n_cat)]
    nums = [fc.numeric_column("I%d" % (j + 1)) for j in range(n_num)]
    return cats, nums


def criteo_device_batches(engine, batch_size, n_batches, seed, n_cat=26, n_num=13):
    """n_batches Criteo-shaped PackedBatches generated ON THE DEVICE (torch ops: uniform 32-bit keys rendered as
    8-hex-char strings, log1p(Poisson) numerics, Bernoulli(0.25) labels), every one with fresh ids.  The arena layout
    is the one engine.pack() produces for a host batch of the same shape; only the key bytes, the numeric columns and
    the labels differ from batch to batch (the string offsets are the same arange * 8)."""
    import torch
    rng = np.random.default_rng(seed)
    feats, y = criteo_batch(batch_size, rng, n_cat, n_num)
    tmpl = engine.pack(feats, y, device=True)
    dev = tmpl.arena.device
    g = torch.Generator(device=dev)
    g.manual_seed(int(seed))
    hexlut = torch.tensor(list(b"0123456789abcdef"), dtype=torch.uint8, device=dev)
    shifts = torch.arange(7, -1, -1, device=dev, dtype=torch.int64) * 4
    out = [tmpl]
    for _ in range(n_batches - 1):
        arena = tmpl.arena.clone()
        for kind, idx, off, nbytes in tmpl.layout:
            if kind == "cat":
                keys = torch.randint(0, 1 << 32, (batch_size,), generator=g, device=dev, dtype=torch.int64)
                arena[off:off + nbytes] = hexlut[((keys[:, None] >> shifts[None, :]) & 15)].reshape(-1)
            elif kind == "num":
                lam = torch.full((batch_size,), 3.0 + idx, device=dev)
                arena[off:off + nbytes] = torch.log1p(torch.poisson(lam, generator=g)).to(torch.float32).view(torch.uint8).reshape(-1)
            elif kind == "lab":
                arena[off:off + nbytes] = (torch.rand(batch_size, generator=g, device=dev) < 0.25).to(torch.float32).view(torch.uint8).reshape(-1)
        out.append(engine.repack_like(tmpl, arena))
    return out
