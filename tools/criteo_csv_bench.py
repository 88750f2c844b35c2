"""GPU CSV decoder on Criteo-shaped text: 65 536 tab-separated records (label, I1..I13 float32, C1..C26 hex keys, as
synth.write_criteo_tsv writes them), decoded from device-resident text and from pinned host memory; the share of
float fields whose rounding the fast paths of csv.cu cannot decide (counted on the host with the same rule); and the
ML-100K decode of tools/csv_bench.py for comparison.  Prints one JSON line with the card's name and power limit."""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from recommender_tensorflow_b200 import synth  # noqa: E402
from recommender_tensorflow_b200.csv_reader import GpuCsvReader  # noqa: E402
from recommender_tensorflow_b200.engine import DeepFMEngine  # noqa: E402
from recommender_tensorflow_b200.trainers import ml_100k  # noqa: E402

N = 65536


def _pow5(q):
    """(m, e): 5^q = m * 2^e rounded down, m in [2^63, 2^64) (the table of csv.cu)"""
    from fractions import Fraction
    v = Fraction(5) ** q
    k = v.numerator.bit_length() - v.denominator.bit_length()
    if Fraction(2) ** k > v:
        k -= 1
    return int(v * Fraction(2) ** (63 - k)), k - 63


def needs_slow_path(field):
    """True when csv_decimal_to_float hands this (valid, decimal) field to csv_float_slow.  A host restatement of the
    device rule (keep the two in step when either changes); the kernel itself counts nothing."""
    s = field.strip(b" \t\n\v\f\r").lstrip(b"+-")
    mant = s.split(b"e")[0].split(b"E")[0]
    ex = int(s[len(mant) + 1:]) if len(mant) < len(s) else 0
    w, nsig, q, sticky, dot = 0, 0, 0, False, False
    for c in mant:
        if c == ord("."):
            dot = True
            continue
        d = c - 48
        if nsig < 19:
            if nsig or d:
                w, nsig = w * 10 + d, nsig + 1
            q -= dot
        else:
            sticky |= d != 0
            q += not dot
    q += ex
    if w == 0 or q + nsig - 1 > 38 or q + nsig <= -46 or (not sticky and w <= 1 << 24 and -10 <= q <= 10):
        return False
    m, e = _pow5(q)
    lz = 64 - w.bit_length()
    n = (w << lz) * m
    t = 127 if n >> 127 else 126
    sh = max(t - 23, -(e + q - lz + 149))
    if sh >= 130:
        return False
    if sh == 129:
        return n >= (1 << 128) - (1 << 70)
    below = (1 << (sh - 1)) - 1
    f = n & below
    return (f >> 70) == (below >> 70) or ((n >> (sh - 1)) & 1 and f == 0)


def _time_decode(rd, src, reps=20):
    for _ in range(3):
        rd.decode(src)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        rd.decode(src)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def _sources(body):
    pad = (body.size + 15) // 16 * 16
    dev = torch.zeros(pad, dtype=torch.uint8, device="cuda")
    dev[:body.size] = torch.from_numpy(body.copy()).cuda()
    return (("device", dev[:body.size]), ("pinned_host", torch.from_numpy(body.copy()).pin_memory()))


def _rates(dt, n_bytes):
    return {"ms": round(dt * 1e3, 4), "M_records_per_s": round(N / dt / 1e6, 2), "GB_per_s_of_text": round(n_bytes / dt / 1e9, 2)}


def criteo(tmp):
    path = os.path.join(tmp, "criteo.tsv")
    synth.write_criteo_tsv(path, N, seed=1)
    body = np.fromfile(path, dtype=np.uint8)
    cats, nums = synth.criteo_columns(1 << 20)
    eng = DeepFMEngine(cats, nums, embedding_size=16, hidden_units=(16, 16), max_batch=N)
    cols, defaults = synth.criteo_tsv_schema()
    rd = GpuCsvReader(eng, cols, defaults, label_col="label", cutoff=1, max_records=N, max_bytes=body.size + 64, field_delim="\t")
    out = {"records": N, "bytes": int(body.size)}
    for name, src in _sources(body):
        out[name] = _rates(_time_decode(rd, src), body.size)
    floats = [f for line in body.tobytes().split(b"\n") if line for f in line.split(b"\t")[1:14] if f]
    out["float_fields"] = len(floats)
    # not a device counter: the share is counted on the host with needs_slow_path, a restatement of the kernel's rule
    out["slow_path_share_host_count"] = sum(map(needs_slow_path, floats)) / len(floats)
    return out


def ml100k(tmp):
    fc = ml_100k.get_feature_columns(16)
    eng = DeepFMEngine(fc["linear"], (), embedding_size=16, hidden_units=(256, 128), feature_dtypes=ml_100k.FEATURE_DTYPES, max_batch=N)
    path = os.path.join(tmp, "t.csv")
    ml_100k.write_synthetic_csv(path, N)
    data = np.fromfile(path, dtype=np.uint8)
    body = data[int(np.flatnonzero(data == 10)[0]) + 1:]
    rd = GpuCsvReader(eng, ml_100k.COLUMNS, ml_100k.DEFAULTS, ml_100k.LABEL_COL, max_records=N, max_bytes=body.size + 64)
    out = {"records": N, "bytes": int(body.size)}
    for name, src in _sources(body):
        out[name] = _rates(_time_decode(rd, src), body.size)
    return out


def main():
    if not torch.cuda.is_available():
        sys.exit("criteo_csv_bench: no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    with tempfile.TemporaryDirectory() as tmp:
        line = {"gpu": q.stdout.strip(), "criteo_tsv": criteo(tmp), "ml_100k_csv": ml100k(tmp)}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
