#!/usr/bin/env python
"""bench.py — DeepFM train samples/sec (fwd + bwd + sparse Adam) on B200, per BASELINE.json.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl b200|reference]

A "step" is one pass of the hot path (transform -> gather/FM -> tower -> loss -> backward -> sorted sparse reduction ->
optimizers) over one batch of synthetic input.  `value` times the device-resident path (inputs already in HBM); `e2e`
times the same steps through the host-buffer C-ABI entry point (H2D of the raw columns + D2H of the loss inside the timed
region).

ONE workload for the whole 1 -> 8 series: the Criteo-shaped DeepFM (26 x 1e7 hashed rows, 13 numerics, k = 16, hidden
[16,16], 65 536 samples per GPU per step) — unsharded on one GPU, row-sharded (weak scaling) on N > 1.  At N = 1 the
line also carries `secondary` blocks for BASELINE configs[2] / [1] / [0], and every line a `zipf` block (Zipf(1.05) ids).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "DeepFM train samples/sec (fwd+bwd+sparse Adam)"

WORKLOADS = {
    # BASELINE.json configs[3] (and its single-GPU form: 26 x 1e7 rows, k=16: 16.6 GB of tables + 33 GB of Adam slots)
    "deepfm_criteo_1e7_k16_h16x16_b65536": dict(data="criteo", k=16, hidden=(16, 16), batch=65536, model="deepfm",
                                                buckets=10_000_000),
    "deepfm_criteo_1e6_k16_h16x16_b65536": dict(data="criteo", k=16, hidden=(16, 16), batch=65536, model="deepfm",
                                                buckets=1_000_000),
    # BASELINE.json configs[4]: k = 64, global batch 262 144, tables sharded over 8 GPUs, data-parallel [256,128] tower.
    # 26 x 1e8 rows x (64 + 2 x 64 Adam) fp32 = 2.0 TB does not fit 8 x 180 GB (SURVEY.md 7-2): 5e6 buckets per field
    # PER GPU are used (4e7 per field = 1.04e9 rows = 865 GB of 832-byte records at 8 GPUs), batch 32 768 per GPU.
    "deepfm_criteo_k64_h256x128_b262144": dict(data="criteo", k=64, hidden=(256, 128), batch=32768, model="deepfm",
                                               buckets_per_gpu=5_000_000),
    # BASELINE.json configs[2]: the DeepFM config with a tensor-core tower
    "deepfm_ml100k_k16_h256x128_b65536": dict(data="ml100k", k=16, hidden=(256, 128), batch=65536, model="deepfm"),
    # configs[0] / configs[1]
    "deepfm_ml100k_k4_h16x16_b32": dict(data="ml100k", k=4, hidden=(16, 16), batch=32, model="deepfm"),
    "wide_deep_ml100k_k4_h16x16_b4096": dict(data="ml100k", k=4, hidden=(16, 16), batch=4096, model="wide_deep"),
}
DEFAULT_WORKLOAD = "deepfm_criteo_1e7_k16_h16x16_b65536"
SECONDARY = ["deepfm_ml100k_k16_h256x128_b65536", "wide_deep_ml100k_k4_h16x16_b4096", "deepfm_ml100k_k4_h16x16_b32"]
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel (ncu --set full, profiles/)
TRAFFIC = {
    "deepfm_criteo_1e7_k16_h16x16_b65536": (851.8e6, "fused_rows_kernel<16,16,2> (gather + tower + in-kernel optimizer of the once-only rows: 504.5 MB read + "
                                            "347.3 MB written per launch; profiles/r02bc_fused_rows_full_summary.txt, captured before the last two "
                                            "instruction-stream changes of the kernel, which move no bytes); algorithmic record traffic of "
                                            "that kernel: 1.70 M rows x 256 B in + 1.68 M rows x 208 B out = 785 MB -> traffic / algorithmic = 1.09"),
    "deepfm_ml100k_k16_h256x128_b65536": (151.8e6, "mean of the 4 launches/step of tc::gemm_persist_kernel<16>; profiles/r01k_gemm_persist_full_summary.csv"),
}


def bytes_per_sample(dc, dn, k, slots_emb, slots_lin):
    """SURVEY.md §8(d) algorithmic bytes per sample (fp32, int32 ids, no dedup credit)."""
    inputs = 4 * dc + 4 * dn + 4
    gather = 4 * dc * (k + 1)
    update = 2 * 4 * dc * (k * (1 + slots_emb) + (1 + slots_lin))
    return inputs + gather + update


def workload_buckets(w, world):
    return w["buckets"] if "buckets" in w else w["buckets_per_gpu"] * max(world, 1)


def make_columns(w, world=1):
    from recommender_tensorflow_b200 import synth
    from recommender_tensorflow_b200.trainers import ml_100k
    if w["data"] == "ml100k":
        return ml_100k.get_feature_columns()["linear"], [], ml_100k.FEATURE_DTYPES
    cats, nums = synth.criteo_columns(workload_buckets(w, world))
    return cats, nums, {}


def make_batches(w, n_batches, seed, zipf=None):
    from recommender_tensorflow_b200 import synth
    rng = np.random.default_rng(seed)
    out = []
    if w["data"] == "ml100k":
        ml = synth.ML100K()
        for _ in range(n_batches):
            out.append(ml.fast_batch(w["batch"], rng))
    else:
        for _ in range(n_batches):
            out.append(synth.criteo_batch(w["batch"], rng, zipf_alpha=zipf))
    return out


def optimizers(w):
    from recommender_tensorflow_b200.engine import default_optimizer
    if w["model"] == "wide_deep":   # trainers/linear_deep.py:32-39 canned defaults (SURVEY §8a row 8)
        return dict(use_mf=False, loss_reduction="sum", opt_deep=default_optimizer("Adagrad", 0.001),
                    opt_linear=default_optimizer("Ftrl", 0.005))
    return dict(use_mf=True, loss_reduction="mean", opt_deep=default_optimizer("Adam", 0.001),
                opt_linear=default_optimizer("Adam", 0.001))


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.stop_flag = gpu_index, [], False

    def _run_nvml(self):
        """NVML directly (nvidia_ml_py): a query takes ~0.1 ms, so even a 20 ms timed region gets several samples."""
        import pynvml
        pynvml.nvmlInit()
        hdl = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(hdl, pynvml.NVML_CLOCK_SM)
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        while not self.stop_flag:
            sm = pynvml.nvmlDeviceGetClockInfo(hdl, pynvml.NVML_CLOCK_SM)
            r = int(get_reasons(hdl))
            self.samples.append([str(sm), str(mx), ""] + ["Active" if r & bits[k] else "Not Active"
                                                          for k in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
            time.sleep(0.002)

    def run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass                      # no NVML binding: fall back to polling nvidia-smi (slow: ~10 samples/s)
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------- reference (CPU) arm
class _EngLike:
    pass


def _eng_like(w, world=1):
    """what tests.util.oracle_cfg needs from an engine, without creating one (no CUDA)"""
    cats, nums, dtypes = make_columns(w, world)
    e = _EngLike()
    cats = sorted(cats, key=lambda c: c.name + "_embedding")
    e.specs = []
    for c in cats:
        s = c.spec()
        if s["kind"] == "bucketized":
            s["dtype"] = dtypes.get(s["source"], "float32")
        e.specs.append(s)
    e.num_columns = sorted(nums, key=lambda c: c.name)
    e.k, e.hidden = w["k"], list(w["hidden"])
    o = optimizers(w)
    e.use_linear, e.use_mf, e.use_dnn = True, o["use_mf"], True
    e.loss_reduction, e.opt_deep, e.opt_linear = o["loss_reduction"], o["opt_deep"], o["opt_linear"]
    return e


def cpu_baseline(w, seconds_target=12.0, threads=None, max_steps=200):
    """Restated reference (torch-CPU oracle, NOT TensorFlow) timed on the host cores on a bounded sample."""
    import torch
    from oracle.deepfm import OracleDeepFM, init_weights
    from tests.util import oracle_cfg
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    cfg = oracle_cfg(_eng_like(w))
    nb = sum(int(s["num_buckets"]) for s in cfg["cat"])
    shrunk = ""
    if nb > 5_000_000:   # the literal non-lazy CPU step walks the whole table every step: bound the sample
        for s in cfg["cat"]:
            if s["kind"] == "hash":
                s["num_buckets"] = min(int(s["num_buckets"]), 100_000)
        shrunk = "; hash buckets capped at 1e5/field for the CPU sample (the literal non-lazy Adam walks whole tables)"
    ora = OracleDeepFM(cfg, init_weights(cfg, 0))
    bs = min(w["batch"], 4096)
    batches = make_batches(dict(w, batch=bs), 4, 99)
    feats = []
    for f, y in batches:   # oracle takes object arrays of bytes for strings
        ff = {}
        for k, v in f.items():
            if isinstance(v, tuple):
                data, offs = v
                raw = data.tobytes()
                ff[k] = np.array([raw[offs[i]:offs[i + 1]] for i in range(len(offs) - 1)], dtype=object)
            else:
                ff[k] = v
        feats.append((ff, y))
    ora.train_step_raw(*feats[0])
    t0, n = time.perf_counter(), 0
    while True:
        ora.train_step_raw(*feats[n % len(feats)])
        n += 1
        dt = time.perf_counter() - t0
        if dt > seconds_target or n >= max_steps:
            break
    return {"value": bs * n / dt, "unit": "samples/s", "cores": threads, "kind": "port", "ms_per_cpu_step": dt / n * 1e3, "cpu_batch": bs,
            "cpu_steps": n,
            "sample": "%d steps of batch %d of the same workload, torch-CPU float32 restatement of the TF-1.12 step "
                      "(incl. literal non-lazy Adam); not TensorFlow%s" % (n, bs, shrunk)}


def run_reference(args, w, name):
    """--impl reference: the reference's CPU implementation of the path (oracle port; TF 1.12 is not installable)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step_budget = 60.0 / max(1, args.steps + args.warmup)
    base = cpu_baseline(w, seconds_target=max(5.0, min(30.0, per_step_budget * args.steps)))
    line = {"metric": METRIC, "value": base["value"], "unit": "samples/s", "n_gpus": args.gpus, "steps": base["cpu_steps"],
            "warmup": 1, "ms_per_step": base["ms_per_cpu_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": name, "batch_per_gpu": w["batch"], "embedding_size": w["k"], "hidden_units": list(w["hidden"]),
                       "note": "CPU arm: restated reference (oracle port, torch-CPU); TensorFlow 1.12 is not installable in this image; "
                               "steps / ms_per_step are the CPU steps actually run, each on a bounded sample of cpu_batch samples "
                               "(value = cpu_batch x steps / time)"},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline_subprocess(name):
    """the CPU leg in its own process: the GPU arm never loads anything under oracle/"""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", name, "--steps", "1", "--warmup", "0"],
                           capture_output=True, text=True, timeout=240, env=dict(os.environ, RANK="0", WORLD_SIZE="1", CUDA_VISIBLE_DEVICES=""))
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"unavailable": (r.stderr or r.stdout)[-300:]}
    except Exception as ex:
        return {"unavailable": repr(ex)}


def csv_decode_bench(eng, B, iters=20):
    """records/s of dfm_csv_decode on one batch of ML-100K-shaped CSV text (42 fields, quoted titles) resident in HBM,
    and from pinned host text (H2D inside the timed region).  Wall clock around the call: it returns after the
    decode finished (two stream syncs inside)."""
    import tempfile

    import torch
    from recommender_tensorflow_b200.csv_reader import GpuCsvReader
    from recommender_tensorflow_b200.trainers import ml_100k
    n_unique = min(B, 4096)
    path = os.path.join(tempfile.mkdtemp(), "bench.csv")
    ml_100k.write_synthetic_csv(path, n_unique)
    data = np.fromfile(path, dtype=np.uint8)
    body = data[int(np.flatnonzero(data == 10)[0]) + 1:]
    body = np.tile(body, (B + n_unique - 1) // n_unique)
    nl = np.flatnonzero(body == 10)
    body = body[:int(nl[B - 1]) + 1].copy()
    rd = GpuCsvReader(eng, ml_100k.COLUMNS, ml_100k.DEFAULTS, ml_100k.LABEL_COL, max_records=B, max_bytes=body.size + 64)
    dev = torch.zeros((body.size + 15) // 16 * 16, dtype=torch.uint8, device="cuda")
    dev[:body.size] = torch.from_numpy(body).cuda()
    pinned = torch.from_numpy(body).pin_memory()
    out = {"records": B, "text_bytes": int(body.size), "unit": "records/s"}
    for key, src in (("value", dev[:body.size]), ("from_pinned_host", pinned)):
        for _ in range(3):
            assert rd.decode(src).batch_size == B
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            rd.decode(src)
        torch.cuda.synchronize()
        out[key] = B * iters / (time.perf_counter() - t0)
    out["text_GBps"] = out["value"] * body.size / B / 1e9
    rd.close()
    return out


# ------------------------------------------------------------------------------------------- outputs of the timed path
DUMP_MAX_ROWS, DUMP_BLOCK = 32768, 1024


def dump_outputs(eng, loss, out_dir):
    """What the timed path hands its caller after its last step: the loss of that step (loss.npy) and the trained
    state, every variable and optimizer slot as <name>.npy ("emb/m" -> emb.m.npy), float32.  A tensor of more than
    DUMP_MAX_ROWS rows is stored as DUMP_MAX_ROWS / DUMP_BLOCK blocks of DUMP_BLOCK consecutive rows at offsets drawn
    from a fixed seed, in ascending order: the same rows for every tensor of the same height and on every run (6.5 MB
    for the default workload, about 32 MB at k = 64: under 64 MB).  Reading the state applies the optimizer steps that
    are still deferred (dfm_flush),
    outside the timed region.  Sharded runs store rank 0's shard."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().cpu().numpy().astype(np.float32))
    for var in eng.variable_names():
        for name in [var] + [var + "/" + s for s in eng.slot_names(var)]:
            rows, _ = eng.tensor_shape(name)
            if rows <= DUMP_MAX_ROWS:
                a = eng.get_tensor(name)
            else:
                starts = np.sort(np.random.default_rng(0).choice(rows // DUMP_BLOCK, DUMP_MAX_ROWS // DUMP_BLOCK, replace=False))
                a = np.concatenate([eng.get_tensor(name, int(s) * DUMP_BLOCK, DUMP_BLOCK) for s in starts])
            np.save(os.path.join(out_dir, name.replace("/", ".") + ".npy"), a)


# ------------------------------------------------------------------------------------------- one measured workload
def measure(name, args, world, rank, local, peaks, primary=True, zipf=None):
    """Times one workload on this rank's GPU (all ranks call it for the primary workload).  Returns the JSON dict on
    rank 0 (None elsewhere)."""
    import torch
    import torch.distributed as dist
    from recommender_tensorflow_b200 import synth
    from recommender_tensorflow_b200.engine import DeepFMEngine

    w = WORKLOADS[name]
    steps, warmup = (args.steps, args.warmup) if primary else (min(args.steps, 20), min(args.warmup, 5))
    if zipf:
        steps, warmup = min(steps, 10), 3
    cats, nums, dtypes = make_columns(w, world)
    B = w["batch"]
    sharded = world > 1 and w["data"] == "criteo"
    kw = dict(embedding_size=w["k"], hidden_units=w["hidden"], max_batch=B, device=local, feature_dtypes=dtypes, **optimizers(w))
    exchange = os.environ.get("DFM_SHARD_EXCHANGE", "xchg")     # "xchg": kernel stores + flags in peer memory; "nccl": all_to_all
    parity = None
    if sharded and primary and not zipf and os.environ.get("DFM_PARITY_CHECK", "1") != "0":
        # two more engines live during the check: it runs before the timed engine exists, on tables cut to <= 16 GB per GPU
        from recommender_tensorflow_b200 import synth as _synth
        rec_bytes = (3 * w["k"] + 4 + 15) // 16 * 16 * 4
        rows_gpu = 26 * workload_buckets(w, world) // world
        pc, pn = cats, nums
        note = None
        if rows_gpu * rec_bytes > 16e9:
            small = int(16e9 // rec_bytes // 26) * world
            pc, pn = _synth.criteo_columns(small)
            note = "tables cut to %d buckets per field for the check (two extra engines must fit beside nothing else)" % small
        parity = parity_check(w, kw, pc, pn, rank, world, local)
        if note:
            parity["note"] = note
    eng = DeepFMEngine(cats, nums, rank=rank if sharded else 0, world=world if sharded else 1, **kw)
    eng.init_random(1234)            # same dense tower on every rank; the table shards differ by construction (own rows)
    if sharded:
        from recommender_tensorflow_b200.sharded import ShardedTrainer, XchgTrainer
        trainer = XchgTrainer(eng) if exchange == "xchg" else ShardedTrainer(eng)

    # ---- inputs: fresh ids in every batch.  Criteo-shaped batches are generated on the device (32 of them); the
    # Zipf(1.05) variant and the ML-100K-shaped batches come from the numpy generators (8 batches)
    if w["data"] == "criteo" and not zipf:
        n_batches = 32
        packed_dev = synth.criteo_device_batches(eng, B, n_batches, 777 + rank)
        packed_host = []
        for pb in packed_dev[:8]:
            host = torch.empty(pb.arena.numel(), dtype=torch.uint8).pin_memory()
            host.copy_(pb.arena)
            packed_host.append(eng.repack_like(pb, host))
    else:
        n_batches = 8
        host_batches = make_batches(w, n_batches, 777 + rank, zipf=zipf)
        packed_host = [eng.pack(f, y) for f, y in host_batches]
        packed_dev = [eng.pack(f, y, device=True) for f, y in host_batches]
    h2d_bytes = packed_host[0].nbytes

    stream = torch.cuda.Stream()
    loss_buf = torch.zeros(1, dtype=torch.float32, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    prefetch = sharded and exchange == "xchg" and os.environ.get("DFM_SHARD_PREFETCH", "1") != "0"

    def dev_step(i, last=False):
        if sharded:
            nxt = packed_dev[(i + 1) % n_batches] if prefetch and not last else None      # requests of the next batch beside apply
            loss_buf.copy_(trainer.train_step(packed_dev[i % n_batches], B * world, next_pb=nxt).reshape(1))
        else:
            eng.train_step_device(packed_dev[i % n_batches], loss_out=loss_buf, stream=stream.cuda_stream)

    # ---------------- device-resident timing (value)
    with torch.cuda.stream(stream):
        for i in range(warmup):
            dev_step(i, last=i == warmup - 1)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for i in range(steps):
            dev_step(warmup + i, last=i == steps - 1)
        ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = eng.last_step_launches * steps
    eng.sync()
    torch.cuda.synchronize()
    last_loss = float(loss_buf.item())
    unique_rows = eng.last_unique_rows
    if primary and not zipf and args.dump_outputs:
        if rank == 0:
            dump_outputs(eng, loss_buf, args.dump_outputs)
        barrier()

    # ---------------- end-to-end through the host-buffer entry point (e2e)
    nh = len(packed_host)
    if sharded:
        stage = [torch.empty_like(packed_dev[0].arena) for _ in range(3)]
        staged = [eng.repack_like(packed_dev[0], a) for a in stage]

        # H2D copies run on their own stream, one step ahead of their first use: the columns of step i + 2 are copied while
        # step i computes (its tail already issues the requests of step i + 1, whose columns arrived during step i - 1).
        # Ring of three arenas: arena (i + 2) % 3 was last read by step i - 1, so the copy waits for that step's event.
        copy_stream = torch.cuda.Stream()
        copied = {}
        step_done = {}

        def e2e_copy(i):
            if i not in copied:
                if i - 3 in step_done:
                    copy_stream.wait_event(step_done[i - 3])
                with torch.cuda.stream(copy_stream):
                    staged[i % 3].arena.copy_(packed_host[i % nh].arena, non_blocking=True)  # H2D of the raw columns of step i
                    ev = torch.cuda.Event()
                    ev.record(copy_stream)
                copied[i] = ev

        def e2e_step(i, last=False):
            e2e_copy(i)
            nxt = None
            if prefetch and not last:
                e2e_copy(i + 1)
                nxt = staged[(i + 1) % 3]
            stream.wait_event(copied[i])
            if nxt is not None:
                stream.wait_event(copied[i + 1])
            out = trainer.train_step(staged[i % 3], B * world, next_pb=nxt)
            ev = torch.cuda.Event()
            ev.record(stream)
            step_done[i] = ev
            if not last:
                e2e_copy(i + 2)                      # in flight beside step i
            return out
        with torch.cuda.stream(stream):
            for i in range(2):
                e2e_step(i, last=i == 1)
        barrier()
        copied.clear()
        step_done.clear()
        loss_pin = torch.empty(2, dtype=torch.float32).pin_memory()
        loss_evs = [torch.cuda.Event(), torch.cuda.Event()]
        e2e_loss = float("nan")
        t0 = time.perf_counter()
        with torch.cuda.stream(stream):
            for i in range(steps):
                loss_pin[i % 2:i % 2 + 1].copy_(e2e_step(i, last=i == steps - 1).reshape(1), non_blocking=True)   # D2H of the loss, every step ...
                loss_evs[i % 2].record(stream)
                if i > 0:                                                                # ... read one step late, like
                    loss_evs[(i - 1) % 2].synchronize()                                  # dfm_train_step_host_async
                    e2e_loss = float(loss_pin[(i - 1) % 2])
            loss_evs[(steps - 1) % 2].synchronize()
            e2e_loss = float(loss_pin[(steps - 1) % 2])
        barrier()
        e2e_s = time.perf_counter() - t0
    else:
        for i in range(3):
            eng.train_step_async(packed_host[i % nh])
        eng.drain()
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            eng.train_step_async(packed_host[i % nh])     # H2D + step; returns the previous step's loss (D2H)
        e2e_loss = eng.drain()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    sampler.stop_flag = True
    sampler.join(timeout=2)

    t = torch.tensor([ms, e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_s = float(t[0]), float(t[1])

    phases = None
    if sharded:
        phases = {}
        with torch.cuda.stream(stream):
            for i in range(5):
                trainer.train_step(packed_dev[i % n_batches], B * world, timings=phases)
        phases = {k: v / 5 for k, v in phases.items()}
    else:
        eng.set_profiling(True)
        eng.train_step_device(packed_dev[0], loss_out=loss_buf)
        eng.sync()
        phases = eng.phase_ms()
        eng.set_profiling(False)

    line = None
    if rank == 0:
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        se = {"Adam": 2, "Adagrad": 1, "Ftrl": 2, "SGD": 0}
        o = optimizers(w)
        bps = bytes_per_sample(len(cats), len(nums), w["k"], se[o["opt_deep"]["name"]], se[o["opt_linear"]["name"]])
        value = B * steps * world / (ms * 1e-3)
        achieved = value / world * bps / 1e9
        traffic = TRAFFIC.get(name) if not zipf else None
        line = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "b200",
            "config": {"workload": name, "batch_per_gpu": B, "embedding_size": w["k"], "hidden_units": list(w["hidden"]),
                       "n_cat": len(cats), "n_num": len(nums), "table_rows": int(eng.row_offsets[-1]),
                       "ids": ("Zipf(%.2f) keys" % zipf) if zipf else "uniform 32-bit keys, fresh in every batch",
                       "optimizer": o["opt_deep"]["name"] + ("/" + o["opt_linear"]["name"] if w["model"] == "wide_deep" else " (TF non-lazy, exact deferred)"),
                       "l2": "per-step working set (%s) exceeds L2; inputs rotate over %d batches" % (
                           "%.0f MB of table records" % (unique_rows * 256e-6) if w["data"] == "criteo" else "activations + gradients", n_batches),
                       "parallelism": "single GPU" if world == 1 else (
                           "tables row-sharded over %d GPUs (ids / rows / gradient rows / dense gradients exchanged by %s), data-parallel "
                           "tower; global batch %d" % (world, "kernel stores into IPC-mapped peer memory over NVLink, flag-synchronised: no collective "
                                                       "and no host sync inside the step" if exchange == "xchg" else "NCCL all_to_all / all_gather", B * world)
                           if sharded else "replicas x%d" % world)},
            "gpu_launches": int(launches),
            "loss_last": last_loss,
            "unique_rows_per_step": int(unique_rows), "unique_row_ratio": unique_rows / float(B * max(len(cats), 1)),
            "e2e": {"value": B * steps * world / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_s * 1e3 / steps, "loss_last": e2e_loss,
                    "how": ("pinned host arena -> H2D copy of every step's columns on a copy stream (three device arenas, two steps ahead), sharded step (launches only), D2H of the loss every step (read one step late); "
                            "wall clock, barrier + device sync on both sides" if sharded else
                            "dfm_train_step_host_async: pinned host arena -> one H2D copy per step on a copy stream, step, "
                            "D2H of the loss; double buffered, wall clock with a device sync on both sides")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic[0] if traffic else None, "traffic_note": traffic[1] if traffic else None,
                         "bytes_per_sample": bps, "peak_source": peak_kind,
                         "scope": "whole step (all kernels of one train step; SURVEY.md 8d bytes/sample x batch / step time)"},
            "phases_ms": phases,
            "clocks": sampler.summary(),
        }
        if parity is not None:
            line["parity_check"] = parity
        if sharded:
            # SURVEY.md 8d: algorithmic NVLink bytes per sample of the sharded step (ids out, rows back, gradient rows out)
            nvb = len(cats) * (4 + 2 * 4 * (w["k"] + 1)) * (world - 1) / world
            ach = value / world * nvb / 1e9
            line["roofline_nvlink"] = {"bound": "nvlink", "achieved": ach, "peak": 770.0, "unit": "GB/s per GPU per direction", "frac": ach / 770.0,
                                       "bytes_per_sample": nvb, "peak_source": "B200_PROFILING.md measured peer copy (770 GB/s per direction)"}
        if w["hidden"] and max(w["hidden"]) >= 64 and phases and not sharded:
            # the tower GEMMs (3xTF32 on tcgen05): algorithmic fp32 flops of the tower vs the tf32 tensor peak / 3.  The
            # step is tensor-bound here: 3 x flops at the measured tf32 rate is the floor, not the HBM figure above
            d_in = (len(cats) + len(nums)) * w["k"]
            dims = [d_in] + list(w["hidden"])
            fl = 3 * 2 * B * (sum(a * b for a, b in zip(dims[:-1], dims[1:])) + dims[-1])
            tt = (phases["mlp_fwd"] + phases["mlp_bwd"]) * 1e-3
            bf16 = float(peaks.get("bf16_tflops", 1590.0))
            line["roofline_tower"] = {"bound": "tensor", "achieved": fl / tt / 1e12, "peak": bf16 / 2 / 3, "unit": "TFLOP/s (fp32-equivalent)",
                                      "frac": fl / tt / 1e12 / (bf16 / 6), "flops_per_step": fl,
                                      "tensor_floor_ms": fl / (bf16 / 6 * 1e12) * 1e3,
                                      "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (tf32 rate) / 3 (three TF32 MMAs per fp32-accurate product)"}
    eng.close()
    del packed_dev, packed_host
    torch.cuda.empty_cache()
    return line


def parity_check(w, kw, cats, nums, rank, world, local):
    """N > 1: three untimed steps through the NCCL all_to_all trainer and through the fused, flag-synchronised exchange
    from identical state on identical batches; the line carries whether the global loss and the checksum of every
    shard (tables + optimizer slots + dense tower) are equal bit for bit."""
    import torch
    import torch.distributed as dist
    from recommender_tensorflow_b200 import synth
    from recommender_tensorflow_b200.engine import DeepFMEngine
    from recommender_tensorflow_b200.sharded import ShardedTrainer, XchgTrainer
    B = w["batch"]
    out = {"steps": 3}
    engs = [DeepFMEngine(cats, nums, rank=rank, world=world, **kw) for _ in range(2)]
    for e in engs:
        e.init_random(4321)
    ta, tb = ShardedTrainer(engs[0]), XchgTrainer(engs[1])
    pbs = synth.criteo_device_batches(engs[0], B, 3, 555 + rank)
    la, lb = [], []
    for pb in pbs:
        la.append(float(ta.train_step(pb, B * world).item()))
    for pb in pbs:
        lb.append(float(tb.train_step(pb, B * world).item()))
    torch.cuda.synchronize()
    ca, cb = engs[0].state_checksum(), engs[1].state_checksum()
    flags = torch.tensor([int(la == lb), int(ca == cb)], dtype=torch.int32, device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    out.update({"loss_bits_equal": bool(flags[0].item()), "shard_checksum_equal": bool(flags[1].item()),
                "loss_nccl": la, "loss_xchg": lb, "checksum_rank0": "%016x" % cb,
                "what": "ShardedTrainer (NCCL all_to_all + all_gather) vs XchgTrainer (peer-memory stores + flags), same seed, same batches; "
                        "checksum = sum of the 32-bit patterns of every table record and dense parameter / slot on the rank, ANDed over ranks"})
    for e in engs:
        e.close()
    del pbs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default=None, help="default: %s at every N (row-sharded, weak scaling, at N>1)" % DEFAULT_WORKLOAD)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs[2]/[1]/[0] blocks at N=1")
    ap.add_argument("--no-zipf", action="store_true", help="skip the Zipf(1.05) block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss of the last one and the trained state (large tables as a "
                         "fixed, seeded sample of rows) to DIR/<name>.npy, to compare two builds on identical inputs")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    name = args.workload or DEFAULT_WORKLOAD
    w = WORKLOADS[name]
    if args.impl == "reference":
        run_reference(args, w, name)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (NCCL prints its version there)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    line = measure(name, args, world, rank, local, peaks, primary=True)
    if w["data"] == "criteo" and not args.no_zipf:
        try:      # SURVEY.md 8d: the same workload with Zipf(1.05) ids (hot rows, per-destination dedup, owner imbalance)
            z = measure(name, args, world, rank, local, peaks, primary=False, zipf=1.05)
            if rank == 0:
                line["zipf"] = {k: z[k] for k in ("value", "ms_per_step", "steps", "unique_rows_per_step", "unique_row_ratio", "e2e", "roofline",
                                                  "phases_ms", "loss_last") if k in z}
                line["zipf"]["ids"] = z["config"]["ids"]
                if "roofline_nvlink" in z:
                    line["zipf"]["roofline_nvlink"] = z["roofline_nvlink"]
        except Exception as ex:
            if rank == 0:
                line["zipf"] = {"unavailable": repr(ex)}
    if rank == 0:
        if world == 1 and not args.no_secondary and args.workload is None:
            line["secondary"] = []
            for sname in SECONDARY:
                try:
                    s = measure(sname, args, 1, 0, local, peaks, primary=False)
                    keep = {k: s[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "gpu_launches", "e2e", "roofline", "phases_ms", "loss_last")}
                    keep["config"] = s["config"]
                    if "roofline_tower" in s:
                        keep["roofline_tower"] = s["roofline_tower"]
                    line["secondary"].append(keep)
                except Exception as ex:
                    line["secondary"].append({"config": {"workload": sname}, "unavailable": repr(ex)})
            try:      # side measurement: the CSV input path decoded on the GPU (SURVEY.md 8f-2)
                from recommender_tensorflow_b200.engine import DeepFMEngine
                from recommender_tensorflow_b200.trainers import ml_100k
                e2 = DeepFMEngine(ml_100k.get_feature_columns()["linear"], (), embedding_size=4, hidden_units=(16, 16), max_batch=65536,
                                  device=local, feature_dtypes=ml_100k.FEATURE_DTYPES)
                line["csv_decode"] = csv_decode_bench(e2, 65536)
                e2.close()
            except Exception as ex:
                line["csv_decode"] = {"unavailable": repr(ex)}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_subprocess(name)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
