"""Cost of vocabulary lookups on the device (K1, transform_kernel): the hash table against the linear scan.

Part 1, transform alone: one vocabulary column, B = 65 536, V in {2, 16, 256, 4096, 10^5, 10^6, 10^7}; string keys
(1-40 bytes, a third over 16) and int keys; all hits, 50 % misses without OOV buckets and 50 % misses with 7 OOV buckets;
uniform and Zipf(1.05) choice of the hit keys.  Time per dfm_transform call from CUDA events around 50 back-to-back calls
(after 5 warm-up calls) on 4 alternating input batches; the table of V = 10^7 (512 MiB) is larger than the 126 MB L2,
smaller ones are L2-resident as they would be in training.  The scan (DFM_VOCAB_PATH=scan, string keys only: integer
vocabularies are always looked up through the table) is measured up to V = 4096; beyond that it costs O(V) compares
per lookup and is not run.

Part 2, step time: the headline-shaped model (26 string columns, 13 numerics, k = 16, hidden [16, 16], Adam,
B = 65 536) with every categorical column a vocabulary of 10^6 8-hex-char keys (inputs drawn from 2 x 10^6 keys: half
miss), against the same model with 26 hashed columns of 10^6 buckets.  Median of 60 device-resident steps (CUDA events
around each), 8 alternating input batches; and dfm_create's time for one string vocabulary of 10^7 entries.

The GPU name and power limit are read in the same run.

    python tools/vocab_bench.py [--out FILE] [--quick]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

B = 65536


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["clocks_max_sm"] = [v.strip() for v in q.split(",")]
    except Exception as e:
        info["power_limit"] = "unknown (%s)" % e
    return info


def str_vocab(V):
    lens = (np.arange(V) * 7919) % 40 + 1
    return [(b"%x" % j + b"-" * int(n))[:max(int(n), len(b"%x" % j))] for j, n in enumerate(lens)]


def pick(V, n, dist, rng):
    if dist == "zipf":
        return (rng.zipf(1.05, n) - 1) % V
    return rng.integers(0, V, n)


def inputs(dtype, vocab, miss, dist, rng):
    V = len(vocab)
    idx = pick(V, B, dist, rng)
    is_miss = rng.random(B) < miss
    if dtype == "string":
        vals = [b"~%x" % rng.integers(0, 1 << 40) if is_miss[b] else vocab[idx[b]] for b in range(B)]
        return np.array(vals, dtype=object)
    v = np.asarray(vocab, np.int64)[idx]
    return np.where(is_miss, -(rng.integers(1, 1 << 30, B) + 7), v).astype(np.int32)


def transform_time(eng, batches, reps=50, warm=5):
    import torch
    out = torch.empty((B, eng.n_slots), dtype=torch.int32, device="cuda")
    stream = torch.cuda.Stream()
    call = lambda pb: eng._check(eng.lib.dfm_transform(eng.h, C.byref(pb.raw), C.c_void_p(out.data_ptr()),
                                                       C.c_void_p(stream.cuda_stream)))
    for i in range(warm):
        call(batches[i % len(batches)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(reps):
        call(batches[i % len(batches)])
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1000.0 / reps


def part1(out, quick):
    from recommender_tensorflow_b200 import feature_column as fc
    from recommender_tensorflow_b200.engine import DeepFMEngine
    Vs = [2, 16, 256, 4096, 10 ** 5] if quick else [2, 16, 256, 4096, 10 ** 5, 10 ** 6, 10 ** 7]
    for dtype in ("string", "int32"):
        for V in Vs:
            vocab = str_vocab(V) if dtype == "string" else [int(x) for x in (np.arange(V, dtype=np.int64) * 2654435761) % (1 << 31)]
            lst = [v.decode() for v in vocab] if dtype == "string" else vocab
            rng = np.random.default_rng(V)
            for miss, oov in ((0.0, 0), (0.5, 0), (0.5, 7)):
                col = fc.categorical_column_with_vocabulary_list("k", lst, num_oov_buckets=oov)
                for path in ("table", "scan"):
                    if path == "scan" and (dtype != "string" or V > 4096):
                        continue
                    os.environ["DFM_VOCAB_PATH"] = path
                    eng = DeepFMEngine([col], (), embedding_size=4, hidden_units=(8,), max_batch=B,
                                       feature_dtypes={"k": dtype})
                    for dist in ("uniform", "zipf"):
                        batches = [eng.pack({"k": inputs(dtype, vocab, miss, dist, rng)}, None, device=True) for _ in range(4)]
                        us = transform_time(eng, batches)
                        rec = dict(part="transform", dtype=dtype, V=V, miss=miss, num_oov=oov, dist=dist, path=path,
                                   us_per_call=round(us, 2), ns_per_lookup=round(us * 1000 / B, 3))
                        print(json.dumps(rec), flush=True)
                        out.write(json.dumps(rec) + "\n")
                    eng.close()
    os.environ.pop("DFM_VOCAB_PATH", None)


def step_time(eng, batches, steps=60, warm=10):
    import torch
    stream = torch.cuda.Stream()
    loss = torch.zeros(1, dtype=torch.float32, device="cuda")
    with torch.cuda.stream(stream):
        for i in range(warm):
            eng.train_step_device(batches[i % len(batches)], loss_out=loss, stream=stream.cuda_stream)
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    with torch.cuda.stream(stream):
        evs[0].record(stream)
        for i in range(steps):
            eng.train_step_device(batches[i % len(batches)], loss_out=loss, stream=stream.cuda_stream)
            evs[i + 1].record(stream)
    torch.cuda.synchronize()
    ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
    return float(np.median(ms))


def part2(out, quick):
    import torch
    from recommender_tensorflow_b200 import feature_column as fc
    from recommender_tensorflow_b200 import synth
    from recommender_tensorflow_b200.engine import DeepFMEngine
    V = 10 ** 5 if quick else 10 ** 6
    keys, _ = synth.hex8(np.arange(V, dtype=np.uint32))
    voc = [bytes(keys[j * 8:(j + 1) * 8]).decode() for j in range(V)]
    dt = {"C%d" % (f + 1): "string" for f in range(26)}
    rng = np.random.default_rng(5)
    host = [synth.criteo_batch(B, rng, key_space=2 * V) for _ in range(8)]
    res = {}
    for variant in ("hashed", "vocab", "hashed", "vocab"):
        cats, nums = synth.criteo_columns(V)
        if variant == "vocab":
            cats = [fc.categorical_column_with_vocabulary_list(c.key, voc) for c in cats]
        t0 = time.time()
        eng = DeepFMEngine(cats, nums, embedding_size=16, hidden_units=(16, 16), max_batch=B, feature_dtypes=dt)
        t_create = time.time() - t0
        eng.init_random(1234)
        batches = [eng.pack(f, y, device=True) for f, y in host]
        ms = step_time(eng, batches)
        tr = transform_time(eng, batches)
        res.setdefault(variant, []).append(ms)
        rec = dict(part="step", variant=variant, V=V, fields=26, step_ms=round(ms, 4), transform_us=round(tr, 2),
                   create_s=round(t_create, 2), launches=eng.last_step_launches)
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")
        eng.close()
        del batches
        torch.cuda.empty_cache()
    # dfm_create of one string vocabulary of 10^7 entries (Python packing excluded)
    if not quick:
        big = [v.decode() for v in str_vocab(10 ** 7)]
        col = fc.categorical_column_with_vocabulary_list("k", big)
        t0 = time.time()
        eng = DeepFMEngine([col], (), embedding_size=4, hidden_units=(8,), max_batch=B, feature_dtypes={"k": "string"})
        rec = dict(part="create", V=10 ** 7, dtype="string", create_s_incl_python_packing=round(time.time() - t0, 2),
                   table_bytes=(1 << 25) * 16, vocab_bytes=sum(map(len, big)))
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")
        eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="vocab_bench.jsonl")
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--part", choices=["1", "2", "all"], default="all")
    a = ap.parse_args()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as out:
        info = gpu_info()
        print(json.dumps(info), flush=True)
        out.write(json.dumps(dict(part="env", **info)) + "\n")
        if a.part in ("1", "all"):
            part1(out, a.quick)
        if a.part in ("2", "all"):
            part2(out, a.quick)


if __name__ == "__main__":
    main()
