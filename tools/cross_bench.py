"""Cost of crossed columns on the Criteo-shaped headline workload (bench.py's deepfm_criteo_1e7_k16_h16x16_b65536:
B = 65 536, 26 hashed 8-hex-char columns of 10^7 buckets, 13 numerics, k = 16, hidden [16, 16], Adam), with 0, 3 and 6
extra crossed columns, each a cross of two raw hex keys (C1 x C2, C3 x C4, ...) at 10^7 buckets, and as a control for
each the same number of fields without crosses (26 + n hashed columns).

Per variant: the median step time from CUDA events around every step of the device-resident train step (after warm-up),
and, in a separate profiled run, the device time of transform_kernel per step from torch.profiler.  The inputs are 32
fresh seeded batches generated on the device (synth.criteo_device_batches, ~0.5 GB in all: larger than the 126 MB L2).
The GPU name and power limit are read in the same run.

    python tools/cross_bench.py [--steps 50] [--warmup 10] [--crosses 0 3 6] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["clocks_max_sm"] = [v.strip() for v in q.split(",")]
    except Exception as e:       # the numbers are still reported, marked as lacking the power limit
        info["power_limit"] = "unknown (%s)" % e
    return info


def run(n_cross, steps, warmup, B=65536, buckets=10 ** 7, n_hashed=26):
    import torch
    from recommender_tensorflow_b200 import feature_column as fc
    from recommender_tensorflow_b200 import synth
    from recommender_tensorflow_b200.engine import DeepFMEngine

    cats, nums = synth.criteo_columns(buckets, n_cat=n_hashed)
    cats += [fc.crossed_column(["C%d" % (2 * j + 1), "C%d" % (2 * j + 2)], buckets) for j in range(n_cross)]
    dtypes = {"C%d" % (f + 1): "string" for f in range(n_hashed)}
    eng = DeepFMEngine(cats, nums, embedding_size=16, hidden_units=(16, 16), max_batch=B, feature_dtypes=dtypes)
    eng.init_random(1234)
    batches = synth.criteo_device_batches(eng, B, 32, 777, n_cat=n_hashed)
    stream = torch.cuda.Stream()
    loss = torch.zeros(1, dtype=torch.float32, device="cuda")

    def step(i):
        eng.train_step_device(batches[i % len(batches)], loss_out=loss, stream=stream.cuda_stream)

    with torch.cuda.stream(stream):
        for i in range(warmup):
            step(i)
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    with torch.cuda.stream(stream):
        evs[0].record(stream)
        for i in range(steps):
            step(warmup + i)
            evs[i + 1].record(stream)
    torch.cuda.synchronize()
    ms = np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(steps)])
    launches = eng.last_step_launches

    # separate run under the profiler: device time of transform_kernel per step
    from torch.profiler import ProfilerActivity, profile
    n_prof = 10
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with torch.cuda.stream(stream):
            for i in range(n_prof):
                step(warmup + steps + i)
        torch.cuda.synchronize()
    t_us, n_k = 0.0, 0
    for e in prof.events():
        if e.device_type.name == "CUDA" and "transform_kernel" in e.name:
            t_us += e.device_time if hasattr(e, "device_time") else e.cuda_time
            n_k += 1
    out = {"crosses": n_cross, "hashed": n_hashed, "fields": len(eng.specs), "batch": B, "steps": steps,
           "step_ms_median": float(np.median(ms)), "step_ms_p10": float(np.percentile(ms, 10)),
           "step_ms_p90": float(np.percentile(ms, 90)), "samples_per_s": B / (float(np.median(ms)) / 1e3),
           "transform_ms_per_step": t_us / 1e3 / n_prof, "transform_launches_profiled": n_k,
           "launches_per_step": launches, "last_loss": float(loss.item())}
    eng.close()
    del batches
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--crosses", type=int, nargs="+", default=[0, 3, 6])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = gpu_info()
    rows = []
    variants = []
    for n in args.crosses:
        variants.append((n, 26))
        if n:      # control: the same number of fields, all hashed (separates the cost of a field from that of a cross)
            variants.append((0, 26 + n))
    for n, nh in variants:
        r = dict(run(n, args.steps, args.warmup, n_hashed=nh), **info)
        print(json.dumps(r), flush=True)
        rows.append(r)
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
