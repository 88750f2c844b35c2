"""EVAL throughput with the metrics streamed on the device (dfm_evaluate + dfm_metrics_read, DESIGN.md §8.6) against the
per-batch predict_logits + host get_binary_metrics loop that Estimator.evaluate() runs, at the Criteo shape of the
headline step (26 hashed columns of 10^7 buckets, 13 numerics, k = 16, hidden [16, 16], B = 65 536).

The inputs are 32 seeded device batches (synth.criteo_device_batches, ~0.5 GB: larger than the 126 MB L2), cycled.  Both
loops evaluate the same --batches batches: the streamed loop enqueues every batch and reads the state once at the end;
the host loop synchronises on every batch, copies logits and labels back and computes the metrics at the end (its
[200, N] boolean matrices bound the eval-set size it can hold).  Wall times are host clocks around work that ends in a
synchronise, alternated over --rounds rounds.  Then the device time of the accumulation kernels alone (CUDA events over
--launches launches on one [B] batch) next to that of the forward pass alone (dfm_forward).  The GPU name and power limit
are read in the same run.

    python tools/eval_bench.py [--batches 16] [--rounds 3] [--launches 200] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from cross_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from recommender_tensorflow_b200 import synth
    from recommender_tensorflow_b200.trainers.model_utils import finish_binary_metrics, get_binary_metrics
    from recommender_tensorflow_b200.engine import DeepFMEngine

    B = 65536
    cats, nums = synth.criteo_columns(10 ** 7, n_cat=26)
    dtypes = {"C%d" % (f + 1): "string" for f in range(26)}
    eng = DeepFMEngine(cats, nums, embedding_size=16, hidden_units=(16, 16), max_batch=B, feature_dtypes=dtypes)
    eng.init_random(1234)
    pbs = synth.criteo_device_batches(eng, B, 32, 777)
    for pb in pbs[:8]:                                   # a few train steps: logits spread over the thresholds
        eng.train_step_device(pb)
    eng.sync()
    lab_off = [(o, n) for kind, _, o, n in pbs[0].layout if kind == "lab"][0]

    def labels_of(pb):
        o, n = lab_off
        return pb.arena[o:o + n].view(torch.float32)

    def streamed():
        eng.metrics_reset()
        for i in range(args.batches):
            eng.evaluate_batch(pbs[i % len(pbs)])
        return finish_binary_metrics(eng.metrics_state())

    def host():
        zs, ys = [], []
        for i in range(args.batches):
            pb = pbs[i % len(pbs)]
            zs.append(eng.predict_logits(pb))
            ys.append(labels_of(pb).cpu().numpy())
        return get_binary_metrics(np.concatenate(ys), np.concatenate(zs))

    streamed(), host()                                   # warm-up: allocations, module loads
    t = {"streamed": [], "host": []}
    res = {}
    for r in range(args.rounds):
        for name, fn in ((("streamed", streamed), ("host", host)) if r % 2 == 0 else (("host", host), ("streamed", streamed))):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res[name] = fn()
            t[name].append(time.perf_counter() - t0)

    # device time of the accumulation kernels and of the forward pass, one [B] batch
    st = torch.cuda.Stream()
    z = torch.empty(B, dtype=torch.float32, device="cuda")
    pb = pbs[0]
    lab = labels_of(pb)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            for _ in range(5):
                fn()
            e0.record(st)
            for _ in range(n):
                fn()
            e1.record(st)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    fwd_ms = timed(lambda: eng._check(eng.lib.dfm_forward(eng.h, C.byref(pb.raw), C.c_void_p(z.data_ptr()), C.c_void_p(st.cuda_stream))),
                   max(args.launches // 4, 10))
    acc_ms = timed(lambda: eng.metrics_accumulate(z, lab, None, st.cuda_stream), args.launches)
    eval_ms = timed(lambda: eng.evaluate_batch(pb, stream=st.cuda_stream), max(args.launches // 4, 10))
    eng.sync()
    info = gpu_info()
    N = args.batches * B
    rows = []
    for name in ("streamed", "host"):
        rows.append(dict(loop=name, samples=N, wall_s_per_round=t[name], samples_per_s=N / float(np.median(t[name])),
                         auc=res[name]["auc"], accuracy=res[name]["accuracy"], **info))
    rows.append(dict(kernels="per [B] batch", batch=B, forward_ms=fwd_ms, metrics_accumulate_ms=acc_ms, evaluate_ms=eval_ms,
                     launches=args.launches, auc_diff=res["streamed"]["auc"] - res["host"]["auc"],
                     speedup=float(np.median(t["host"])) / float(np.median(t["streamed"])), **info))
    for r in rows:
        print(json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
