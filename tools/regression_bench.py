"""Cost of the squared head (DFM_HEAD_SQUARED, the regressors) on the Criteo-shaped headline step (bench.py's
deepfm_criteo_1e7_k16_h16x16_b65536: B = 65 536, 26 hashed columns of 10^7 buckets, 13 numerics, k = 16, hidden [16, 16],
Adam; the record-staged fused_rows_kernel).

Two handles on the same device-resident batches (their 0/1 labels are valid float labels for the squared head too),
one with the logistic head and one with the squared head, from the same initial weights, are timed alternately in
rounds of --steps steps each, so that clock and neighbour noise falls on both alike.  Per round
and variant: the median step time from CUDA events around every device-resident train step.  The inputs are 32 fresh
seeded batches generated on the device (~0.5 GB in all: larger than the 126 MB L2).  The GPU name and power limit are
read in the same run.

    python tools/regression_bench.py [--steps 50] [--warmup 10] [--rounds 6] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from cross_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from recommender_tensorflow_b200 import synth
    from recommender_tensorflow_b200.engine import DeepFMEngine

    B = 65536
    cats, nums = synth.criteo_columns(10 ** 7, n_cat=26)
    dtypes = {"C%d" % (f + 1): "string" for f in range(26)}
    engs = {}
    for name in ("logistic", "squared"):
        engs[name] = DeepFMEngine(cats, nums, embedding_size=16, hidden_units=(16, 16), max_batch=B, feature_dtypes=dtypes,
                                  head=name)
        engs[name].init_random(1234)
    base = synth.criteo_device_batches(engs["logistic"], B, 32, 777)
    batches = {"logistic": base, "squared": base}
    stream = torch.cuda.Stream()
    loss = torch.zeros(1, dtype=torch.float32, device="cuda")
    step_no = {k: 0 for k in engs}

    def steps(name, n, timed):
        eng, bl = engs[name], batches[name]
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)] if timed else None
        with torch.cuda.stream(stream):
            if timed:
                evs[0].record(stream)
            for i in range(n):
                eng.train_step_device(bl[step_no[name] % len(bl)], loss_out=loss, stream=stream.cuda_stream)
                step_no[name] += 1
                if timed:
                    evs[i + 1].record(stream)
        torch.cuda.synchronize()
        return np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(n)]) if timed else None

    for name in engs:
        steps(name, args.warmup, False)
    per = {k: [] for k in engs}
    for r in range(args.rounds):
        order = ("logistic", "squared") if r % 2 == 0 else ("squared", "logistic")
        for name in order:
            per[name].append(float(np.median(steps(name, args.steps, True))))
    info = gpu_info()
    rows = []
    for name in engs:
        m = per[name]
        rows.append(dict(variant=name, batch=B, steps_per_round=args.steps, rounds=args.rounds,
                         step_ms_median_per_round=m, step_ms_median=float(np.median(m)),
                         samples_per_s=B / (float(np.median(m)) / 1e3), launches_per_step=engs[name].last_step_launches,
                         graph_steps=engs[name].graph_steps, **info))
    diff = [s - lg for s, lg in zip(per["squared"], per["logistic"])]
    rows.append(dict(variant="squared - logistic", step_ms_diff_per_round=diff, step_ms_diff_median=float(np.median(diff)),
                     relative=float(np.median(diff)) / float(np.median(per["logistic"])), **info))
    for r in rows:
        print(json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
