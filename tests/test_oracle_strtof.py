"""CPU: oracle/strtof.py, the statement of TF 1.12's safe_strtof grammar that the device float32 parse is checked
against: known answers, every accepted and rejected form, round trips of random float32 values, the cases where a
double-rounding parse (np.float32(float(s))) is wrong, and the C ABI's rejections of bad float / delimiter settings
(dfm_csv_create checks them before any CUDA call)."""
import ctypes
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np
import pytest

from oracle.strtof import strtof_bits
from recommender_tensorflow_b200 import _lib
from recommender_tensorflow_b200.csv_reader import CSV_FLOAT32, CSV_INT32, CSV_STRING, CsvConfig


def _double_rounded(s):
    with np.errstate(over="ignore"):
        return int(np.array([np.float32(float(s))]).view(np.uint32)[0])


KAT = [
    (b"1.000000059604644775390625", 0x3F800000),        # exact tie between 1 and 1 + 2^-23: even
    (b"1.0000000596046447753906251", 0x3F800001),
    (b"1.00000005960464477539062501", 0x3F800001),
    (b"3.4028235677973366e38", 0x7F7FFFFF),
    (b"3.40282357e38", 0x7F800000),
    (b"7e-46", 0x0), (b"7.1e-46", 0x1), (b"1e-45", 0x1),
    (b"0.1", 0x3DCCCCCD),
    (b"0", 0x0), (b"-0", 0x80000000), (b"-0.0e7", 0x80000000),
    (b"inf", 0x7F800000), (b"-inf", 0xFF800000),
    (b"nan", 0x7FC00000), (b"-nan", 0xFFC00000),
    (b"1.1754942e-38", 0x007FFFFF),                     # largest subnormal
    (b"1.17549435e-38", 0x00800000),                    # smallest normal
    (b"3.4028235e38", 0x7F7FFFFF),                      # FLT_MAX
    (b"1.4e-45", 0x1),                                  # smallest subnormal
]


@pytest.mark.parametrize("field,bits", KAT)
def test_known_answers(field, bits):
    assert strtof_bits(field) == bits, (field, hex(strtof_bits(field) or 0))


def test_known_answers_where_double_rounding_is_wrong():
    assert _double_rounded("1.0000000596046447753906251") == 0x3F800000
    assert _double_rounded("3.4028235677973366e38") == 0x7F800000


ACCEPTED = [
    (b"5.", 0x40A00000), (b".5", 0x3F000000), (b"+1", 0x3F800000), (b"-2.5", 0xC0200000),
    (b"1e3", 0x447A0000), (b"1E3", 0x447A0000), (b"1e+3", 0x447A0000), (b"1000e-3", 0x3F800000), (b"0.e+0", 0x0),
    (b" 1.5", 0x3FC00000), (b"1.5 ", 0x3FC00000), (b"\t\n\v\f\r 1.5 \r\n", 0x3FC00000),
    (b"007", 0x40E00000), (b"1e0000000000000000000000001", 0x41200000),
    (b"1e99999999999999999999", 0x7F800000), (b"-1e99999999999999999999", 0xFF800000),
    (b"1e-99999999999999999999", 0x0), (b"0e99999999999999999999", 0x0),
    (b"0." + b"0" * 80 + b"1e81", 0x3F800000),
    (b"Inf", 0x7F800000), (b"INFINITY", 0x7F800000), (b"+infinity", 0x7F800000), (b"-InFiNiTy", 0xFF800000),
    (b"NaN", 0x7FC00000), (b"+nan", 0x7FC00000), (b"-NAN", 0xFFC00000), (b" nan ", 0x7FC00000),
]

REJECTED = [b"", b" ", b" \t ", b"1e", b"1e+", b"1e5x", b".", b"-", b"+.", b"--1", b"+-1", b"1 2", b"1.2.3", b"infx",
            b"in", b"infinit", b"nana", b"-nanx", b"e5", b".e5", b"0x10", b"0X1p3", b"1,5", b'1""', b'""', b"1f",
            b"1d", b"\x001", b"1_000", b"\xef\xbc\x91"]


@pytest.mark.parametrize("field,bits", ACCEPTED)
def test_grammar_accepts(field, bits):
    assert strtof_bits(field) == bits, (field, hex(strtof_bits(field) or 0))


@pytest.mark.parametrize("field", REJECTED)
def test_grammar_rejects(field):
    assert strtof_bits(field) is None, field


def random_float32_bits(n, rng):
    """finite float32 bit patterns with every exponent field equally likely (0: subnormals and zeros)"""
    exp = rng.integers(0, 255, n, dtype=np.uint32)
    man = rng.integers(0, 1 << 23, n, dtype=np.uint32)
    sign = rng.integers(0, 2, n, dtype=np.uint32)
    return (sign << np.uint32(31)) | (exp << np.uint32(23)) | man


def test_round_trip_shortest_and_9_digits():
    u = random_float32_bits(100_000, np.random.default_rng(7))
    assert len(set((u >> np.uint32(23)) & np.uint32(255))) == 255
    for b, x in zip(u.tolist(), u.view(np.float32)):
        for s in (np.format_float_scientific(x, unique=True), np.format_float_positional(x, unique=True), "%.9g" % x):
            assert strtof_bits(s.encode()) == b, (s, hex(b))


def _midpoint(bits):
    """exact value of the point halfway between positive finite float32 `bits` and the next one up"""
    ef = bits >> 23
    sig = (bits & 0x7FFFFF) | (0x800000 if ef else 0)
    return Fraction(2 * sig + 1) * Fraction(2) ** (max(ef, 1) - 151)


def _decimal(v, digits=None):
    getcontext().prec = 200
    d = Decimal(v.numerator) / Decimal(v.denominator)
    return str(d) if digits is None else ("%." + str(digits - 1) + "e") % d


def test_midpoints_and_nearby_values_round_once():
    """exact midpoints go to the even neighbour; a unit in the 20th-30th significant digit above or below decides the
    direction, which np.float32(float(s)) (two roundings) gets wrong on many of them"""
    rng = np.random.default_rng(3)
    u = random_float32_bits(3000, rng) & np.uint32(0x7FFFFFFF)
    u = u[u < 0x7F7FFFFF]
    differ = 0
    for b in u.tolist():
        m = _midpoint(b)
        exact = _decimal(m)
        assert Fraction(exact) == m
        want = b + (b & 1)
        assert strtof_bits(exact.encode()) == want, (exact, hex(b))
        differ += _double_rounded(exact) != want
        digits = int(rng.integers(20, 31))
        e = len(str(m.numerator // m.denominator)) - 1 if m >= 1 else 0
        while Fraction(10) ** e > m:
            e -= 1                                       # m in [10^e, 10^(e+1))
        unit = Fraction(10) ** (e - digits + 1)          # one unit in the `digits`-th significant digit
        for delta, want in ((unit, b + 1), (-unit, b)):
            s = _decimal(m + delta)
            v = Fraction(Decimal(s))
            assert (v > m) == (delta > 0) and v != m
            assert strtof_bits(s.encode()) == want, (s, hex(b))
            differ += _double_rounded(s) != want
    assert differ > 100, differ


# ---------------------------------------------------------------- C ABI rejections (before any CUDA call)
def _create(kinds, field_delim=0, as_float=None):
    lib = _lib.load()
    n = len(kinds)
    kind = (ctypes.c_int32 * n)(*kinds)
    af = (ctypes.c_int32 * n)(*as_float) if as_float else None
    cfg = CsvConfig(n, ctypes.cast(kind, ctypes.POINTER(ctypes.c_int32)), None, None, -1, 0, 16, 4096, 0, None, field_delim,
                    ctypes.cast(af, ctypes.POINTER(ctypes.c_int32)) if af else None)
    h = ctypes.c_void_p()
    rc = lib.dfm_csv_create(ctypes.byref(cfg), ctypes.byref(h))
    return rc, (lib.dfm_csv_last_error(None) or b"").decode()


@pytest.mark.parametrize("delim", [ord('"'), ord("\n"), ord("\r"), 256, -1, -9])
def test_abi_rejects_bad_field_delim(delim):
    rc, err = _create([CSV_INT32, CSV_FLOAT32], field_delim=delim)
    assert rc == -1 and "field_delim" in err, (rc, err)


@pytest.mark.parametrize("kind", [CSV_STRING, CSV_FLOAT32, 0])
def test_abi_rejects_as_float_on_a_non_int_field(kind):
    rc, err = _create([CSV_INT32, kind], as_float=[0, 1])
    assert rc == -1 and "as_float is set on field 1" in err, (rc, err)


def test_abi_rejects_unknown_kind():
    rc, err = _create([CSV_INT32, 4])
    assert rc == -1 and "unknown kind 4" in err, (rc, err)
