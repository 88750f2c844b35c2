"""GPU: float32 fields of the CSV record decoder (DFM_CSV_FLOAT32), tab-separated records and int32 fields read as
float32.  The device column equals oracle/strtof.py bit for bit (NaN bit patterns included) over a corpus of 10^6
fields built to hit every branch of the parse; errors name the first offending record like the int32 ones; a Criteo
TSV file decodes to the host parse (csv with a tab delimiter plus the oracle) and trains to the same bits; bucketized
columns over float fields and numeric columns over int fields see what the host parse gives them."""
import csv
import io
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np
import pytest

from oracle.strtof import strtof_bits
from recommender_tensorflow_b200 import feature_column as fc
from recommender_tensorflow_b200 import synth
from recommender_tensorflow_b200.csv_reader import GpuCsvReader
from recommender_tensorflow_b200.engine import DeepFMEngine
from recommender_tensorflow_b200.trainers import ml_100k

pytestmark = pytest.mark.gpu

N_NUM = 8


def _float_engine(max_batch, boundaries=None, n_num=N_NUM):
    """one hashed column C plus numeric columns F1..Fn (F1 also bucketized when boundaries are given)"""
    cats = [fc.categorical_column_with_hash_bucket("C", 100)]
    if boundaries:
        cats.append(fc.bucketized_column(fc.numeric_column("F1"), boundaries))
    nums = [fc.numeric_column("F%d" % (j + 1)) for j in range(n_num)]
    return DeepFMEngine(cats, nums, embedding_size=4, hidden_units=(16, 16), max_batch=max_batch)


def _midpoint_text(bits, rng):
    """the exact halfway point above positive float32 `bits`, or it nudged by one unit in its 20th-40th digit"""
    ef = bits >> 23
    m = Fraction(2 * ((bits & 0x7FFFFF) | (0x800000 if ef else 0)) + 1) * Fraction(2) ** (max(ef, 1) - 151)
    getcontext().prec = 200
    d = Decimal(m.numerator) / Decimal(m.denominator)
    pick = int(rng.integers(0, 3))
    if pick == 0:
        return str(d)
    digits = int(rng.integers(20, 41))
    s = ("%." + str(digits - 1) + "e") % d       # rounded to 20-40 digits: just above or below the midpoint
    return s if pick == 1 else s.replace("e", "1e", 1) if "." in s else s


def _long_text(bits, rng):
    """forms past the 19 digits of the fast paths and the 120 of the slow one, and exponents of 20+ digits: the
    halfway point above `bits` padded to 121-160 digits with zeros and a final 1 (just above it) or 0 (on it), the
    same shifted behind zeros or in front of a long exponent, and 150 nines"""
    ef = bits >> 23
    mid = Fraction(2 * ((bits & 0x7FFFFF) | (0x800000 if ef else 0)) + 1) * Fraction(2) ** (max(ef, 1) - 151)
    digits, exp = _sci_digits(mid)
    pad = int(rng.integers(121, 161)) - len(digits)
    tail = "0" * max(pad, 1) + ("1" if rng.integers(0, 2) else "0")
    mant = digits[0] + "." + digits[1:] + tail
    pick = int(rng.integers(0, 4))
    if pick == 0:
        return "%se%d" % (mant, exp)
    if pick == 1:
        return "0." + "0" * 30 + digits + tail + "e%d" % (exp + 31)
    if pick == 2:
        return "%se%s%s" % (mant, "-" if exp < 0 else "+", "0" * 20 + str(abs(exp)))
    return "9" * 150 + "e-%d" % int(rng.integers(100, 190))


def _sci_digits(v):
    """positive Fraction with a terminating decimal expansion -> (all significant digits, decimal exponent)"""
    e = 0
    while v >= 10:
        v /= 10
        e += 1
    while v < 1:
        v *= 10
        e -= 1
    out = ""
    while v:
        d = v.numerator // v.denominator
        out += str(d)
        v = (v - d) * 10
    return out, e


def float_corpus(n, rng):
    """n field texts (as written in the record, quotes included) mixing every form the parse distinguishes"""
    u = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    u[: n // 8] &= np.uint32(0x807FFFFF)                       # subnormals and zeros
    f = u.view(np.float32)
    specials = ["inf", "-Infinity", "NaN", "-nan", "+INF", " nan ", "infinity", "-NAN"]
    out = []
    for i in range(n):
        x, b = f[i], int(u[i])
        r = i % 12
        if not np.isfinite(x) or r == 11:
            s = specials[i % len(specials)]
        elif r == 0:
            s = np.format_float_scientific(x, unique=True)
        elif r == 1:
            s = "%.9g" % x
        elif r == 2:
            s = "%.*e" % (int(rng.integers(19, 40)), x)          # 20-40 significant digits
        elif r == 3:
            s = np.format_float_positional(x, unique=True)
        elif r == 4 and (b & 0x7FFFFFFF) < 0x7F7FFFFF:
            s = ("-" if b >> 31 else "") + _midpoint_text(b & 0x7FFFFFFF, rng)
        elif r == 5:
            s = "%d" % int(rng.integers(-10 ** 9, 10 ** 9))
        elif r == 6:
            s = " %.6g\t" % x
        elif r == 7:
            s = "%.8E" % x
        elif r == 8:
            s = ["", "0", "-0", "5.", ".5", "1e39", "-1e-50", "7.1e-46", "0.000001e6", "1E+2"][i % 10]
        elif r == 10 and i % 24 == 10 and (b & 0x7FFFFFFF) < 0x7F7FFFFF:
            s = _long_text(b & 0x7FFFFFFF, rng)
        elif r == 9:
            s = '"%.9g"' % x                                         # quoted
        else:
            s = "%.17g" % x
        out.append(s)
    return out


def _expected_bits(text, default_bits=0):
    if text.startswith('"'):
        text = text[1:-1]
    if text == "":
        return default_bits
    b = strtof_bits(text.encode())
    assert b is not None, text
    return b


def test_float_parse_matches_oracle_bit_for_bit():
    """10^6 float fields (8 per record) through the device parse against oracle.strtof, NaN bit patterns included"""
    n_rec = 131072
    rng = np.random.default_rng(2026)
    fields = float_corpus(n_rec * N_NUM, rng)
    lines = ["k%d,%s" % (i, ",".join(fields[i * N_NUM:(i + 1) * N_NUM])) for i in range(n_rec)]
    text = ("\n".join(lines) + "\n").encode()
    eng = _float_engine(n_rec)
    cols = ["C"] + ["F%d" % (j + 1) for j in range(N_NUM)]
    rd = GpuCsvReader(eng, cols, [[""]] + [[0.0]] * N_NUM, max_records=n_rec, max_bytes=len(text) + 64)
    assert rd.decode(text).batch_size == n_rec
    want = np.array([_expected_bits(s) for s in fields], dtype=np.uint32).reshape(n_rec, N_NUM)
    for j in range(N_NUM):
        got = rd.column("F%d" % (j + 1))
        assert got.dtype == np.float32
        bad = np.flatnonzero(got.view(np.uint32) != want[:, j])
        assert bad.size == 0, [(fields[i * N_NUM + j], hex(int(got.view(np.uint32)[i])), hex(int(want[i, j]))) for i in bad[:10]]


def test_float_defaults_and_quoting():
    eng = _float_engine(16, n_num=2)
    rd = GpuCsvReader(eng, ["C", "F1", "F2"], [["x"], [-1.5], [0.0]], max_records=16)
    rd.decode(b'a,,\n"b",  2.5 ,""\nc,"-3e0",1e-45\n,"",nan\n')
    assert rd.column("F1").tolist() == [-1.5, 2.5, -3.0, -1.5]
    assert rd.column("F2").view(np.uint32).tolist() == [0, 0, 1, 0x7FC00000]
    assert list(rd.column("C")) == [b"a", b"b", b"c", b"x"]


@pytest.mark.parametrize("bad", ["1e", "1e5x", ".", "--1", "1 2", "infx", '"1""5"', "0x10", " ", '" "', "1,5"])
def test_float_errors_like_decode_csv(bad):
    eng = _float_engine(16, n_num=2)
    rd = GpuCsvReader(eng, ["C", "F1", "F2"], [[""], [0.0], [0.0]], max_records=16)
    rows = ["a,1,2"] * 6
    rows[2] = "a,%s,2" % bad
    rows[4] = "a,1,%s" % bad
    with pytest.raises(ValueError) as ei:
        rd.decode(("\n".join(rows) + "\n").encode())
    msg = str(ei.value)
    assert "record 2" in msg and ("wrong number of fields" if bad == "1,5" else "not a valid float") in msg, msg


def _host_criteo(text, n_num=13, n_cat=26):
    """csv with a tab delimiter plus oracle.strtof: the reference parse of a Criteo TSV text"""
    rows = list(csv.reader(io.StringIO(text, newline=""), delimiter="\t"))
    feats = {}
    for j in range(n_num):
        bits = np.array([_expected_bits(r[1 + j]) for r in rows], dtype=np.uint32)
        feats["I%d" % (j + 1)] = bits.view(np.float32)
    for f in range(n_cat):
        feats["C%d" % (f + 1)] = np.array([r[1 + n_num + f].encode() for r in rows], dtype=object)
    y = np.array([int(r[0]) >= 1 for r in rows], dtype=np.float32)
    return feats, y


def _criteo_engine(max_batch):
    cats, nums = synth.criteo_columns(1000)
    return DeepFMEngine(cats, nums, embedding_size=4, hidden_units=(16, 16), max_batch=max_batch)


def _assert_columns(rd, feats, y):
    for name, want in feats.items():
        got = rd.column(name)
        if want.dtype == object:
            assert list(got) == list(want), name
        else:
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), name
    assert np.array_equal(rd.labels(), y)


def test_criteo_tsv_end_to_end(tmp_path):
    path = str(tmp_path / "criteo.tsv")
    synth.write_criteo_tsv(path, 2048, seed=5, empty_frac=0.1)
    text = open(path, newline="").read()
    feats, y = _host_criteo(text)
    cols, defaults = synth.criteo_tsv_schema()
    B = 256
    a, b = _criteo_engine(B), _criteo_engine(B)
    rd = GpuCsvReader(b, cols, defaults, label_col="label", cutoff=1, max_records=2048, max_bytes=len(text) + 64, field_delim="\t")
    assert rd.decode(text.encode()).batch_size == 2048
    _assert_columns(rd, feats, y)
    assert rd.load_file(path) == 2048
    idx = np.random.default_rng(1).permutation(2048)
    a.init_random(3)
    b.init_random(3)
    for step in range(6):
        sel = idx[step * B:(step + 1) * B]
        pb = rd.decode_lines(sel)
        if step == 0:
            _assert_columns(rd, {k: v[sel] for k, v in feats.items()}, y[sel])
            assert np.array_equal(b.transform(pb), a.transform({k: v[sel] for k, v in feats.items()}))
        la, lga = a.train_step({k: v[sel] for k, v in feats.items()}, y[sel], return_logits=True)
        lb, lgb = b.train_step_device(pb, return_logits=True)
        assert la == lb and np.array_equal(lga, lgb), step
    assert a.state_checksum() == b.state_checksum()


def test_bucketized_over_float_field():
    bounds = [-1.0, 0.0, 0.5, 1.0, 1e30]
    n = 4096
    rng = np.random.default_rng(8)
    vals = float_corpus(n, rng)
    vals = [v if "nan" not in v.lower() else "2.5" for v in vals]
    text = "".join("k%d,%s,%s\n" % (i, vals[i], "%.9g" % rng.standard_normal()) for i in range(n))
    eng = _float_engine(n, boundaries=bounds, n_num=2)
    rd = GpuCsvReader(eng, ["C", "F1", "F2"], [[""], [0.25], [0.0]], max_records=n, max_bytes=len(text) + 64)
    pb = rd.decode(text.encode())
    rows = list(csv.reader(io.StringIO(text, newline="")))
    feats = {"C": np.array([r[0].encode() for r in rows], dtype=object),
             "F1": np.array([_expected_bits(r[1], 0x3E800000) for r in rows], dtype=np.uint32).view(np.float32),
             "F2": np.array([_expected_bits(r[2]) for r in rows], dtype=np.uint32).view(np.float32)}
    assert np.array_equal(rd.column("F1").view(np.uint32), feats["F1"].view(np.uint32))
    assert np.array_equal(eng.transform(pb), eng.transform(feats))


def test_numeric_column_over_int_field_trains_like_host_input():
    """numeric_column("age") over ML-100K's int32 field: the reader writes tf.to_float of it (as_float)"""
    cols = ml_100k.get_feature_columns(4)["linear"]
    mk = lambda: DeepFMEngine(cols, [fc.numeric_column("age")], embedding_size=4, hidden_units=(16, 16), max_batch=256,
                              feature_dtypes=ml_100k.FEATURE_DTYPES)
    a, b = mk(), mk()
    a.init_random(4)
    b.init_random(4)
    ml = synth.ML100K()
    rd = GpuCsvReader(b, ml_100k.COLUMNS, ml_100k.DEFAULTS, ml_100k.LABEL_COL, max_records=256)
    rng = np.random.default_rng(6)
    for step in range(5):
        lines = []
        for _ in range(256):
            u, it = int(rng.integers(1, ml.n_users + 1)), int(rng.integers(1, ml.n_items + 1))
            row = []
            for name, d in zip(ml_100k.COLUMNS, ml_100k.DEFAULTS):
                if name == "age":
                    row.append(["%d" % ml.age[u], "", " %d " % (ml.age[u] + 100000)][int(rng.integers(0, 3))])
                elif name == "user_id":
                    row.append("%d" % u)
                elif name == "item_id":
                    row.append("%d" % it)
                elif name == "rating":
                    row.append("%d" % rng.integers(1, 6))
                else:
                    row.append("%d" % rng.integers(0, 2) if isinstance(d[0], int) else "v%d" % rng.integers(0, 5))
            lines.append(",".join(row))
        text = "\n".join(lines) + "\n"
        feats, y = ml_100k._to_batch(list(csv.reader(io.StringIO(text, newline=""))), 5)
        pb = rd.decode(text.encode())
        assert np.array_equal(rd.float_column("age"), feats["age"].astype(np.float32))
        la, lga = a.train_step(feats, y, return_logits=True)
        lb, lgb = b.train_step_device(pb, return_logits=True)
        assert la == lb and np.array_equal(lga, lgb), step
    assert a.state_checksum() == b.state_checksum()


def test_int_to_float_rounds_to_nearest():
    """int32 values above 2^24 take __int2float_rn, i.e. np.float32 of the int"""
    eng = DeepFMEngine([fc.categorical_column_with_identity("i", 10)], [fc.numeric_column("i")], embedding_size=4,
                       hidden_units=(16, 16), max_batch=16)
    rd = GpuCsvReader(eng, ["i"], [[0]], max_records=16)
    vals = [16777217, 16777219, -16777219, 2147483647, -2147483648, 0, 3]
    rd.decode(("\n".join(str(v) for v in vals) + "\n").encode())
    assert np.array_equal(rd.float_column("i"), np.array(vals, dtype=np.int64).astype(np.float32))
