"""Mirror of the reference's trainers/ml_100k.py: CSV schema, feature columns, input_fn."""
import csv

import numpy as np

from .. import feature_column as fc

# trainers/ml_100k.py:3-15
COLUMNS = ("user_id,item_id,rating,timestamp,datetime,year,month,day,week,dayofweek,"
           "age,gender,occupation,zipcode,zipcode1,zipcode2,zipcode3,"
           "title,release,video_release,imdb,unknown,action,adventure,animation,children,"
           "comedy,crime,documentary,drama,fantasy,filmnoir,horror,musical,mystery,romance,"
           "scifi,thriller,war,western,release_date,release_year").split(",")
GENRE = ("unknown,action,adventure,animation,children,comedy,crime,documentary,drama,fantasy,"
         "filmnoir,horror,musical,mystery,romance,scifi,thriller,war,western").split(",")
LABEL_COL = "rating"
DEFAULTS = [[0], [0], [0], [0], ["null"], [0], [0], [0], [0], [0],
            [0], ["null"], ["null"], ["null"], ["null"], ["null"], ["null"],
            ["null"], ["null"], ["null"], ["null"], [0], [0], [0], [0], [0],
            [0], [0], [0], [0], [0], [0], [0], [0], [0], [0],
            [0], [0], [0], [0], ["null"], [0]]
# dtype tf.decode_csv yields per column (int32 for [0] defaults, string for ["null"])
FEATURE_DTYPES = {c: ("int32" if isinstance(d[0], int) else "string") for c, d in zip(COLUMNS, DEFAULTS)}


def get_feature_columns(embedding_size=4):
    """trainers/ml_100k.py:18-39 — same columns, same order, same bucket counts."""
    user_fc = fc.categorical_column_with_hash_bucket("user_id", 1000, "int32")
    item_fc = fc.categorical_column_with_hash_bucket("item_id", 2000, "int32")
    age_fc = fc.numeric_column("age")
    age_buckets = fc.bucketized_column(age_fc, list(range(15, 66, 10)))
    gender_fc = fc.categorical_column_with_vocabulary_list("gender", ["F", "M"], num_oov_buckets=1)
    occupation_fc = fc.categorical_column_with_hash_bucket("occupation", 50)
    zipcode_fc = fc.categorical_column_with_hash_bucket("zipcode", 1000)
    release_year_fc = fc.numeric_column("release_year")
    release_year_buckets = fc.bucketized_column(release_year_fc, list(range(1930, 1991, 10)))
    genre_fc = [fc.categorical_column_with_identity(col, 2) for col in GENRE]
    linear_columns = [user_fc, item_fc, age_buckets, gender_fc, occupation_fc, zipcode_fc, release_year_buckets] + genre_fc
    deep_columns = [fc.embedding_column(c, embedding_size) for c in linear_columns]
    return {"linear": linear_columns, "deep": deep_columns}


class ModeKeys:
    """tf.estimator.ModeKeys"""
    TRAIN, EVAL, PREDICT = "train", "eval", "infer"


def _parse_rows(csv_path):
    """tf.data.TextLineDataset(csv).skip(1) + tf.decode_csv(value, DEFAULTS) (trainers/ml_100k.py:44-52):
    RFC-4180 quoting, empty fields take the column default."""
    with open(csv_path, newline="") as fh:
        reader = csv.reader(fh)
        next(reader, None)   # header
        for row in reader:
            if len(row) != len(COLUMNS):
                raise ValueError("Expect %d fields but have %d in record" % (len(COLUMNS), len(row)))
            yield row


def _to_batch(rows, cutoff):
    feats = {}
    for j, (name, default) in enumerate(zip(COLUMNS, DEFAULTS)):
        col = [r[j] for r in rows]
        if isinstance(default[0], int):
            feats[name] = np.array([int(v) if v != "" else default[0] for v in col], dtype=np.int32)
        else:
            feats[name] = np.array([(v if v != "" else default[0]).encode() for v in col], dtype=object)
    label = feats.pop(LABEL_COL)
    if cutoff is None:                                    # the rating itself: the regression head's tf.to_float(label)
        return feats, label.astype(np.float32)
    return feats, (label >= cutoff).astype(np.float32)   # tf.math.greater_equal(label, cutoff)


def get_input_fn(csv_path, mode=ModeKeys.TRAIN, batch_size=32, cutoff=5, seed=None):
    """trainers/ml_100k.py:42-61: skip header; TRAIN: shuffle(16*batch_size).repeat(); batch(batch_size).
    Returns a callable producing an iterator of (features dict, label float32 [B]).  The label is rating >= cutoff;
    cutoff=None makes it the rating itself (the regressors' label)."""
    def input_fn():
        rng = np.random.default_rng(seed)
        if mode == ModeKeys.TRAIN:
            buf, cap = [], 16 * batch_size
            batch = []
            while True:                                   # repeat()
                n_rows = 0
                for row in _parse_rows(csv_path):
                    n_rows += 1
                    if len(buf) < cap:                    # shuffle buffer
                        buf.append(row)
                        continue
                    j = int(rng.integers(0, cap))
                    batch.append(buf[j])
                    buf[j] = row
                    if len(batch) == batch_size:
                        yield _to_batch(batch, cutoff)
                        batch = []
                if n_rows == 0:
                    return
                # the shuffle buffer drains at the end of each epoch (shuffle precedes repeat)
                rng.shuffle(buf)
                for row in buf:
                    batch.append(row)
                    if len(batch) == batch_size:
                        yield _to_batch(batch, cutoff)
                        batch = []
                buf = []
        else:
            batch = []
            for row in _parse_rows(csv_path):
                batch.append(row)
                if len(batch) == batch_size:
                    yield _to_batch(batch, cutoff)
                    batch = []
            if batch:
                yield _to_batch(batch, cutoff)
    return input_fn


def write_synthetic_csv(path, n_rows, seed=20260101):
    """ML-100K-shaped CSV with the exact 42-column header of COLUMNS (SURVEY.md §8d)."""
    from .. import synth
    ml = synth.ML100K(seed)
    rng = np.random.default_rng(seed + 1)
    feats, _ = ml.batch(n_rows, rng)
    rating = rng.choice(np.arange(1, 6), size=n_rows, p=[.061, .114, .271, .342, .212])
    with open(path, "w", newline="") as fh:
        wr = csv.writer(fh)
        wr.writerow(COLUMNS)
        for i in range(n_rows):
            row = []
            for name, default in zip(COLUMNS, DEFAULTS):
                if name == LABEL_COL:
                    row.append(int(rating[i]))
                elif name in feats:
                    v = feats[name][i]
                    row.append(v.decode() if isinstance(v, bytes) else int(v))
                elif name == "title":
                    row.append("Movie, The (%d)" % (1900 + i % 100))      # exercises quoting
                else:
                    row.append(0 if isinstance(default[0], int) else "null")
            wr.writerow(row)


def _train_index_stream(n_rows, cap, rng):
    """Row indices in the order get_input_fn's shuffle(16*batch_size).repeat() emits rows (same RNG calls)."""
    while True:
        buf = []
        for i in range(n_rows):
            if len(buf) < cap:
                buf.append(i)
                continue
            j = int(rng.integers(0, cap))
            yield buf[j]
            buf[j] = i
        if n_rows == 0:
            return
        rng.shuffle(buf)
        yield from buf


def get_gpu_input_fn(csv_path, engine, mode=ModeKeys.TRAIN, batch_size=32, cutoff=5, seed=None, weight_column=None,
                     device_labels=False):
    """get_input_fn with tf.decode_csv moved to the GPU (SURVEY.md §8f rank 2): the host only selects whole records
    (same shuffle algorithm and RNG stream as get_input_fn, so the same seed gives the same batches); the file itself
    is uploaded once and stays in HBM, a batch travels as 4 bytes per record (its line number); `GpuCsvReader` splits,
    unquotes, parses and thresholds on the device (cutoff=None: the label is the rating itself, as in get_input_fn).  Yields
    (PackedBatch on the device, labels): in TRAIN mode labels is None (they are inside the batch), otherwise the
    float32 labels are read back for the metrics.  A record is one text line, as with tf.data.TextLineDataset (a
    quoted field cannot contain a line break).  weight_column (a field key or numeric_column of a weighted engine): the
    batches carry that field as their per-example weights; outside TRAIN its host copy is the batch's `weights`
    attribute, for the weighted metrics.  device_labels=True: yield (PackedBatch, None) in every mode, with nothing read
    back - for evaluate_streaming, which takes the labels and weights from the batch on the device."""
    from ..csv_reader import GpuCsvReader
    from .model_utils import weight_column_key
    wkey = weight_column_key(weight_column)

    def input_fn():
        data = np.fromfile(csv_path, dtype=np.uint8)
        nl = np.flatnonzero(data == 10)
        n_lines = int(nl.size) + (1 if data.size and data[-1] != 10 else 0)
        n_rows = max(n_lines - 1, 0)                                      # skip(1): the header
        ends = np.concatenate([nl + 1, [data.size]])[:n_lines]
        lens = np.diff(np.concatenate([[0], ends]))[1:]
        max_bytes = int(np.sort(lens)[-batch_size:].sum()) + 16 if n_rows else 16    # bound on one batch's string bytes
        reader = GpuCsvReader(engine, COLUMNS, DEFAULTS, LABEL_COL, cutoff, max_records=batch_size, max_bytes=max_bytes, weight_col=wkey)
        if n_rows:
            assert reader.load_file(csv_path) == n_lines                  # the file now lives in HBM, split into lines

        def emit(idx):
            pb = reader.decode_lines(np.asarray(idx, dtype=np.int32) + 1)    # +1: line 0 is the header
            if mode == ModeKeys.TRAIN or device_labels:
                return pb, None
            if wkey is not None:
                pb.weights = reader.weights()
            return pb, reader.labels()

        if mode == ModeKeys.TRAIN:
            rng = np.random.default_rng(seed)
            batch = []
            for i in _train_index_stream(n_rows, 16 * batch_size, rng):
                batch.append(i)
                if len(batch) == batch_size:
                    yield emit(batch)
                    batch = []
        else:
            for b0 in range(0, n_rows, batch_size):
                yield emit(np.arange(b0, min(b0 + batch_size, n_rows)))
    return input_fn
