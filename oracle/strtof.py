"""Reference parse of a float32 field of tf.decode_csv (record_defaults [0.0]), TF 1.12.

A non-empty field goes through strings::safe_strtof, i.e. locale_independent_strtonum<float>: a stream extraction
that ends in glibc strtof, plus a table of special names.  This module is the single statement of that grammar as
the project implements it (csrc/csv.cu), with exact rational arithmetic, so that the device parse can be checked
bit for bit:

- leading and trailing ASCII whitespace (isspace) is ignored; a field of blanks only is an error;
- decimal: [+-] digits [. digits] or [+-] . digits, then optionally [eE] [+-] digits; correctly rounded to float32
  (round half to even, any number of digits), subnormals kept, underflow to +-0, overflow to +-inf;
- case-insensitive inf / infinity / nan with an optional sign; -nan keeps the sign bit;
- anything else is an error.  TF 1.12 sends 0x... to strtol(.., 16); this project rejects hex.

The empty field (default substitution) and the unquoting of a quoted field are the caller's business.
"""
from fractions import Fraction

SPACE = b" \t\n\v\f\r"
_SPECIAL = {b"inf": 0x7F800000, b"infinity": 0x7F800000, b"nan": 0x7FC00000}


def _round_bits(v):
    """|v| (a non-negative Fraction) -> float32 bits, round half to even."""
    if v == 0:
        return 0
    # exponent of the unit in the last place: 2^(e - 23) for v in [2^e, 2^(e+1)), never below 2^-149
    e = v.numerator.bit_length() - v.denominator.bit_length()
    if Fraction(2) ** e > v:
        e -= 1
    ulp_exp = max(e - 23, -149)
    scaled = v / Fraction(2) ** ulp_exp
    m, rem = divmod(scaled.numerator, scaled.denominator)
    twice = 2 * rem
    if twice > scaled.denominator or (twice == scaled.denominator and m & 1):
        m += 1
    # m * 2^ulp_exp with m < 2^24 (or == 2^24 after rounding up): encode
    if ulp_exp == -149 and m < (1 << 23):
        return m                                          # subnormal (m == 2^23 is the smallest normal, encoded below)
    while m >= (1 << 24):
        m >>= 1
        ulp_exp += 1
    biased = ulp_exp + 23 + 127
    if biased >= 255:
        return 0x7F800000
    return (biased << 23) | (m & 0x7FFFFF)


def strtof_bits(field):
    """bytes of one (unquoted, non-empty) field -> float32 bit pattern (int), or None if it is not a valid float."""
    s = bytes(field).strip(SPACE)
    if not s:
        return None
    sign = 0
    if s[:1] in (b"+", b"-"):
        sign = 0x80000000 if s[:1] == b"-" else 0
        s = s[1:]
    special = _SPECIAL.get(s.lower())
    if special is not None:
        return special | sign
    mant, exp = s, 0
    for i, c in enumerate(s):
        if c in b"eE":
            mant, tail = s[:i], s[i + 1:]
            digits = tail[1:] if tail[:1] in (b"+", b"-") else tail
            if not digits or not digits.isdigit() or not digits.isascii():
                return None
            exp = int(tail)
            break
    intp, dot, frac = mant.partition(b".")
    if not (intp + frac) or any(c not in b"0123456789" for c in intp + frac):
        return None
    digits = (intp + frac).lstrip(b"0")
    k = exp - len(frac)
    if not digits:
        return sign
    lead = len(digits) - 1 + k            # the value lies in [10^lead, 10^(lead+1))
    if lead > 38:
        return 0x7F800000 | sign          # >= 1e39, beyond FLT_MAX + ulp/2
    if lead < -46:
        return sign                       # < 1e-46, below half the smallest subnormal (7.0e-46)
    return _round_bits(Fraction(int(digits)) * Fraction(10) ** k) | sign


def strtof(field):
    """-> numpy float32 scalar, or None (convenience for host parses)."""
    import numpy as np
    b = strtof_bits(field)
    return None if b is None else np.array([b], dtype=np.uint32).view(np.float32)[0]
