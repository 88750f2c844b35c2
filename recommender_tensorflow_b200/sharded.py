"""Row-sharded DeepFM step over the GPUs of one box (SURVEY.md §8e).

Tables are row-sharded (global row g lives on rank g % world at local index g / world), the dense
tower is replicated and the batch is data-parallel.  Per step every rank runs the four C-ABI phases
(`dfm_shard_requests / serve / forward_backward / apply`); between them this module performs the
collectives with `torch.distributed` (NCCL over NVLink on the GPUs, gloo in the CPU tests of the
routing logic):

    all_to_all(counts) -> all_to_all(row ids) -> [serve] -> all_to_all(rows) -> [forward/backward]
    -> all_to_all(gradient rows) + all_reduce(dense grads, loss) -> [apply]

`XchgTrainer` is the default: the same step with the exchanges fused into the kernels over NVLink peer memory and
synchronised by flags (no collective at all, csrc/xchg.cuh); `ShardedTrainer` above is the NCCL baseline it is
checked against.  `VirtualCluster` runs either set of phases for `world` engines inside ONE process on one GPU,
routing the buffers with plain tensor copies or wiring the exchange regions by raw pointers; it is how the sharded
path is checked against the single-GPU result without a multi-GPU box (B200_PROFILING.md: emulate ranks in one process, never as
co-running kernels that wait on each other).
"""
import numpy as np


def _metric_arrays(state):
    """a metric state as one int64 and one float64 vector (what the ranks all-gather)"""
    ints = np.concatenate([[state["n"]], np.ravel(state["bin_count"]), state["cls"]]).astype(np.int64)
    return ints, np.concatenate([np.ravel(state["bin_weight"]), state["w_cls"], state["sums"]]).astype(np.float64)


def _metric_state(ints, floats, head, weighted):
    nb = (ints.size - 5) // 2
    return {"head": head, "weighted": weighted, "n": np.int64(ints[0]), "bin_count": ints[1:1 + 2 * nb].reshape(2, nb),
            "cls": ints[1 + 2 * nb:], "bin_weight": floats[:2 * nb].reshape(2, nb), "w_cls": floats[2 * nb:2 * nb + 4],
            "sums": floats[2 * nb + 4:]}


def _evaluate_collective(trainer, batches, steps):
    """EVAL on one rank of a process group: each local device batch (labels and weights inside) runs the trainer's
    predict_logits, whose logits are accumulated on the device (dfm_metrics_accumulate); the ranks' metric states are
    then all-gathered and combined in rank order, so every rank returns the same dict.  Every rank must pass the same
    number of batches (the forward passes exchange rows)."""
    from .trainers.model_utils import combine_metric_states, finish_metrics
    torch, dist, eng = trainer.torch, trainer.dist, trainer.eng
    st = torch.cuda.current_stream().cuda_stream
    eng.metrics_reset(st)
    for n, pb in enumerate(batches):
        if steps is not None and n >= steps:
            break
        eng.metrics_accumulate(trainer.predict_logits(pb), pb.raw.labels, pb.raw.weights, st)
    dev = "cuda:%d" % eng.device
    ints, floats = (torch.from_numpy(a).to(dev) for a in _metric_arrays(eng.metrics_state(st)))
    all_i = torch.empty((trainer.W, ints.numel()), dtype=torch.int64, device=dev)
    all_f = torch.empty((trainer.W, floats.numel()), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(all_i, ints, group=trainer.group)
    dist.all_gather_into_tensor(all_f, floats, group=trainer.group)
    all_i, all_f = all_i.cpu().numpy(), all_f.cpu().numpy()
    return finish_metrics(combine_metric_states(_metric_state(all_i[r], all_f[r], eng.head, eng.weighted) for r in range(trainer.W)))


def split_sizes(counts, width=1):
    return [int(c) * width for c in counts]


def route_all_to_all(send_bufs, send_counts, width=1):
    """Pure routing used by VirtualCluster and by the CPU tests: send_bufs[r] is rank r's send buffer laid
    out by destination (send_counts[r][dst] items of `width` elements each).  Returns (recv_bufs, recv_counts)
    where recv_bufs[dst] is the concatenation over source ranks, in rank order."""
    import torch
    W = len(send_bufs)
    recv_counts = [[int(send_counts[src][dst]) for src in range(W)] for dst in range(W)]
    offs = [np.concatenate([[0], np.cumsum(send_counts[r])]).astype(np.int64) for r in range(W)]
    recv = []
    for dst in range(W):
        parts = [send_bufs[src][int(offs[src][dst]) * width:int(offs[src][dst + 1]) * width] for src in range(W)]
        recv.append(torch.cat(parts) if parts else send_bufs[0][:0])
    return recv, recv_counts


def _on_real_stream(step):
    """The C ABI treats a NULL stream as "the handle's own stream", so a step issued while torch's current stream is
    the legacy default stream (handle 0) would run the kernels and the collectives on two unordered streams.  Run
    such a step on a private stream, ordered after / before the default stream."""
    def wrapped(self, *a, **kw):
        torch = self.torch
        cur = torch.cuda.current_stream()
        if cur.cuda_stream != 0:
            return step(self, *a, **kw)
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream()
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            out = step(self, *a, **kw)
        cur.wait_stream(self._side)
        return out
    wrapped.__doc__ = step.__doc__
    return wrapped


class ShardedTrainer:
    """One process per GPU (torchrun); `engine` was created with rank / world of the process group."""

    def __init__(self, engine, group=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.eng, self.group = engine, group
        self.W, self.rank = engine.world, engine.rank
        dev = "cuda:%d" % engine.device
        n = engine.max_batch * max(engine.n_slots, 1)
        rw = engine.row_width
        self.req_rows = torch.empty(n, dtype=torch.int32, device=dev)
        self.recv_rows = torch.empty(2 * n + 4096, dtype=torch.int32, device=dev)
        self.reply = torch.empty((2 * n + 4096) * rw, dtype=torch.float32, device=dev)
        self.rowbuf = torch.empty(n * rw, dtype=torch.float32, device=dev)
        self.gsum = torch.empty(n * rw, dtype=torch.float32, device=dev)
        self.grecv = torch.empty((2 * n + 4096) * rw, dtype=torch.float32, device=dev)
        self.dense = torch.zeros(max(engine.dense_size, 1) + 1, dtype=torch.float32, device=dev)   # [+1]: loss rides along
        self.dense_all = torch.zeros((self.W, max(engine.dense_size, 1) + 1), dtype=torch.float32, device=dev)
        self.cnt_send = torch.empty(self.W, dtype=torch.int32, device=dev)
        self.cnt_recv = torch.empty(self.W, dtype=torch.int32, device=dev)
        self.rw = rw

    @_on_real_stream
    def train_step(self, pb, global_batch, timings=None):
        """One sharded train step on a device-resident PackedBatch; everything is enqueued on torch's current
        stream (the only host syncs are the two count exchanges).  Returns the global loss as a 0-dim cuda
        tensor.  `timings` (dict) collects per-phase device milliseconds when given (debug)."""
        torch, dist, eng, rw = self.torch, self.dist, self.eng, self.rw
        st = torch.cuda.current_stream().cuda_stream
        marks = []

        def mark(name):
            if timings is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((name, e))
        mark("start")
        send_counts = eng.shard_requests(pb, self.req_rows, st)
        mark("requests")
        self.cnt_send.copy_(torch.tensor(send_counts, dtype=torch.int32), non_blocking=True)
        dist.all_to_all_single(self.cnt_recv, self.cnt_send, group=self.group)
        recv_counts = self.cnt_recv.tolist()
        mark("counts")
        U, n_recv = sum(send_counts), sum(recv_counts)
        dist.all_to_all_single(self.recv_rows[:n_recv], self.req_rows[:U], recv_counts, send_counts, group=self.group)
        mark("a2a_ids")
        eng.shard_serve(self.recv_rows, n_recv, self.reply, st)
        mark("serve")
        dist.all_to_all_single(self.rowbuf[:U * rw], self.reply[:n_recv * rw], split_sizes(send_counts, rw),
                               split_sizes(recv_counts, rw), group=self.group)
        mark("a2a_rows")
        nd = eng.dense_size
        eng.shard_forward_backward(pb, self.rowbuf, global_batch, self.dense[nd:nd + 1], None, self.gsum, self.dense, st)
        mark("fwd_bwd")
        dist.all_to_all_single(self.grecv[:n_recv * rw], self.gsum[:U * rw], split_sizes(recv_counts, rw),
                               split_sizes(send_counts, rw), group=self.group)
        mark("a2a_grads")
        # the tower's all-reduce as all_gather + a sum in RANK ORDER: every replica adds the same numbers in the same
        # order (bit-identical replicas, and bit-identical to the fused exchange, whatever NCCL's reduction tree is)
        dist.all_gather_into_tensor(self.dense_all, self.dense, group=self.group)
        self.dense.copy_(self.dense_all[0])
        for r in range(1, self.W):
            self.dense.add_(self.dense_all[r])
        mark("allreduce")
        eng.shard_apply(self.grecv, self.dense, st)
        mark("apply")
        if timings is not None:
            torch.cuda.synchronize()
            for (n0, e0), (n1, e1) in zip(marks[:-1], marks[1:]):
                timings[n1] = timings.get(n1, 0.0) + e0.elapsed_time(e1)
        return self.dense[nd]


    @_on_real_stream
    def predict_logits(self, pb):
        """EVAL / PREDICT: logits of this rank's batch (cuda tensor [B]); no state changes."""
        torch, dist, eng, rw = self.torch, self.dist, self.eng, self.rw
        st = torch.cuda.current_stream().cuda_stream
        send_counts = eng.shard_requests(pb, self.req_rows, st)
        self.cnt_send.copy_(torch.tensor(send_counts, dtype=torch.int32), non_blocking=True)
        dist.all_to_all_single(self.cnt_recv, self.cnt_send, group=self.group)
        recv_counts = self.cnt_recv.tolist()
        U, n_recv = sum(send_counts), sum(recv_counts)
        dist.all_to_all_single(self.recv_rows[:n_recv], self.req_rows[:U], recv_counts, send_counts, group=self.group)
        eng.shard_serve(self.recv_rows, n_recv, self.reply, st)
        dist.all_to_all_single(self.rowbuf[:U * rw], self.reply[:n_recv * rw], split_sizes(send_counts, rw),
                               split_sizes(recv_counts, rw), group=self.group)
        logits = torch.empty(pb.batch_size, dtype=torch.float32, device=self.rowbuf.device)
        eng.shard_forward(pb, self.rowbuf, logits, st)
        return logits

    @_on_real_stream
    def evaluate(self, batches, steps=None):
        """EVAL metrics of the head over this rank's device batches, combined over all ranks (the same dict on every
        rank).  steps: stop after that many batches."""
        return _evaluate_collective(self, batches, steps)


class XchgTrainer:
    """One process per GPU.  The exchanges are fused into the kernels: every rank's exchange region (fixed-capacity id /
    gradient-row segments per (source, owner), a row buffer, dense-gradient slots, flags) is mapped into its peers
    through CUDA IPC; the producing kernels store straight into the destination GPU over NVLink and stamp a flag there,
    the consuming stream waits on that flag with a one-warp kernel (csrc/xchg.cuh).  A train step is ONE C-ABI call that
    only launches kernels: no collective, no host synchronisation, no count exchange.  NCCL is used once, at
    construction, to exchange the 64-byte IPC handles.

    Ordering ("e" = exchange round, incremented by every train / predict call on every rank alike):
        push ids(e) | wait ids | serve(e) | wait rows | forward_backward(e): gradient rows, dense push |
        wait gradient rows | sparse apply | wait dense | dense apply
    Buffer reuse.  ids / headers are double buffered by the parity of e: an owner may still be sorting the ids of round e
    (side stream) when a fast peer already pushes round e+1, but round e+2 cannot start on any rank before this owner
    has finished apply(e+1), i.e. all of round e.  Rows, gradient rows and dense slots are single buffered: their next
    writer is a peer's serve(e+1) / forward_backward(e+1), which wait for MY ids(e+1) / MY rows(e+1); I produce those
    only after my forward_backward(e) / apply(e) - the readers of the old contents - in stream order."""

    def __init__(self, engine, group=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.eng, self.group = engine, group
        self.W, self.rank = engine.world, engine.rank
        dev = "cuda:%d" % engine.device
        mine = torch.frombuffer(bytearray(engine.xchg_export()), dtype=torch.uint8).to(dev)
        allh = torch.empty(self.W * 64, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, mine, group=group)
        engine.xchg_import(bytes(allh.cpu().numpy().tobytes()))
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)
        dist.barrier(group=group)          # every rank has mapped every region before the first store

    @_on_real_stream
    def train_step(self, pb, global_batch, timings=None, next_pb=None):
        """Enqueue one sharded train step on torch's current stream; returns the global loss (0-dim cuda tensor, valid
        once the stream reaches it).  timings (dict): per-phase device milliseconds (adds events, debug)."""
        torch, eng = self.torch, self.eng
        st = torch.cuda.current_stream().cuda_stream
        if timings is None:
            eng.xchg_train_step(pb, global_batch, self.loss, None, st, next_pb=next_pb)
            return self.loss[0]
        marks = []

        def mark(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append((name, e))
        mark("start")
        eng.xchg_begin(pb, st); mark("requests+push")
        eng.xchg_serve(True, st); mark("serve")
        eng.xchg_forward_backward(pb, global_batch, None, st); mark("fwd_bwd")
        eng.xchg_apply(self.loss, st); mark("apply")
        torch.cuda.synchronize()
        for (n0, e0), (n1, e1) in zip(marks[:-1], marks[1:]):
            timings[n1] = timings.get(n1, 0.0) + e0.elapsed_time(e1)
        return self.loss[0]

    @_on_real_stream
    def predict_logits(self, pb):
        """EVAL / PREDICT: logits of this rank's batch (cuda tensor [B]); no state changes."""
        torch, eng = self.torch, self.eng
        st = torch.cuda.current_stream().cuda_stream
        logits = torch.empty(pb.batch_size, dtype=torch.float32, device=self.loss.device)
        eng.xchg_begin(pb, st)
        eng.xchg_serve(False, st)
        eng.xchg_forward(pb, logits, st)
        return logits

    @_on_real_stream
    def evaluate(self, batches, steps=None):
        """EVAL metrics of the head over this rank's device batches, combined over all ranks with one all_gather at the
        end (the same dict on every rank).  steps: stop after that many batches."""
        return _evaluate_collective(self, batches, steps)


class VirtualCluster:
    """`world` engines in one process on one GPU; same phases, routing by tensor copies (or, with p2p=True,
    by the fused peer-memory stores — the handles are wired with raw pointers since they share a process)."""

    def __init__(self, engines, p2p=False):
        import torch
        self.torch = torch
        self.engs = engines
        self.W = len(engines)
        self.p2p = p2p            # True: the flag-synchronised fused exchange (dfm_xchg_*), wired by raw pointers
        if p2p:
            ptrs = [e.xchg_buffer() for e in engines]
            for e in engines:
                e.xchg_set_peers(ptrs)

    def _train_step_p2p(self, pbs, return_logits):
        """The phases rank by rank (every flag is set before the kernel that waits for it is launched: kernels that
        wait on one another must never share a GPU)."""
        torch = self.torch
        dev = "cuda:%d" % self.engs[0].device
        global_batch = sum(pb.batch_size for pb in pbs)
        for e, pb in zip(self.engs, pbs):
            e.xchg_begin(pb)
        for e in self.engs:
            e.sync()
        for e in self.engs:
            e.xchg_serve(True)
        for e in self.engs:
            e.sync()
        logits = []
        for e, pb in zip(self.engs, pbs):
            lg = torch.empty(pb.batch_size, dtype=torch.float32, device=dev)
            e.xchg_forward_backward(pb, global_batch, lg)
            logits.append(lg)
        for e in self.engs:
            e.sync()
        losses = []
        for e in self.engs:
            ls = torch.zeros(1, dtype=torch.float32, device=dev)
            e.xchg_apply(ls)
            losses.append(ls)
        for e in self.engs:
            e.sync()
        vals = [float(x.item()) for x in losses]
        assert all(v == vals[0] for v in vals), "ranks disagree on the global loss: %r" % (vals,)
        if return_logits:
            return vals[0], torch.cat(logits).cpu().numpy()
        return vals[0]

    def train_step(self, pbs, return_logits=False):
        if self.p2p:
            return self._train_step_p2p(pbs, return_logits)
        torch, W = self.torch, self.W
        dev = "cuda:%d" % self.engs[0].device
        rw = self.engs[0].row_width
        global_batch = sum(pb.batch_size for pb in pbs)
        req, counts = [], []
        for e, pb in zip(self.engs, pbs):
            buf = torch.empty(pb.batch_size * max(e.n_slots, 1), dtype=torch.int32, device=dev)
            counts.append(e.shard_requests(pb, buf))
            req.append(buf[:sum(counts[-1])])
        recv_rows, recv_counts = route_all_to_all(req, counts)
        replies = []
        for e, rr in zip(self.engs, recv_rows):
            rep = torch.empty(max(rr.numel(), 1) * rw, dtype=torch.float32, device=dev)
            e.shard_serve(rr.contiguous(), rr.numel(), rep)
            e.sync()
            replies.append(rep[:rr.numel() * rw])
        rowbufs, _ = route_all_to_all(replies, recv_counts, rw)
        gsums, denses, logits = [], [], []
        nd = self.engs[0].dense_size
        for e, pb, rb, c in zip(self.engs, pbs, rowbufs, counts):
            U = sum(c)
            gs = torch.empty(max(U, 1) * rw, dtype=torch.float32, device=dev)
            dn = torch.zeros(nd + 1, dtype=torch.float32, device=dev)
            lg = torch.empty(pb.batch_size, dtype=torch.float32, device=dev)
            rbc = rb.contiguous() if rb.numel() else torch.zeros(rw, dtype=torch.float32, device=dev)
            e.shard_forward_backward(pb, rbc, global_batch, dn[nd:nd + 1], lg, gs, dn)
            e.sync()
            gsums.append(gs[:U * rw]); denses.append(dn); logits.append(lg)
        grecv, _ = route_all_to_all(gsums, counts, rw)
        total = denses[0].clone()                     # all_reduce, summed in rank order
        for dn in denses[1:]:
            total += dn
        for e, gr in zip(self.engs, grecv):
            grc = gr.contiguous() if gr.numel() else torch.zeros(rw, dtype=torch.float32, device=dev)
            e.shard_apply(grc, total)
            e.sync()
        loss = float(total[nd].item())
        if return_logits:
            return loss, torch.cat(logits).cpu().numpy()
        return loss

    def predict_logits(self, pbs):
        """EVAL / PREDICT: logits of all ranks' batches, concatenated in rank order (numpy)."""
        return self.torch.cat(self._rank_logits(pbs)).cpu().numpy()

    def evaluate(self, batches, steps=None):
        """EVAL metrics of the head: batches yields one list of device PackedBatches (labels and weights inside) per
        step, one per rank.  Each rank accumulates its logits on the device (dfm_metrics_accumulate); the states are
        combined in rank order on the host.  steps: stop after that many steps."""
        from .trainers.model_utils import combine_metric_states, finish_metrics
        for e in self.engs:
            e.metrics_reset()
        for n, pbs in enumerate(batches):
            if steps is not None and n >= steps:
                break
            for e, pb, lg in zip(self.engs, pbs, self._rank_logits(pbs)):
                e.metrics_accumulate(lg, pb.raw.labels, pb.raw.weights)
        return finish_metrics(combine_metric_states(e.metrics_state() for e in self.engs))

    def _rank_logits(self, pbs):
        """logits of each rank's batch: cuda tensors, computed and synchronised"""
        torch = self.torch
        dev = "cuda:%d" % self.engs[0].device
        rw = self.engs[0].row_width
        outs = []
        if self.p2p:
            for e, pb in zip(self.engs, pbs):
                e.xchg_begin(pb)
            for e in self.engs:
                e.sync()
            for e in self.engs:
                e.xchg_serve(False)
            for e in self.engs:
                e.sync()
            for e, pb in zip(self.engs, pbs):
                lg = torch.empty(pb.batch_size, dtype=torch.float32, device=dev)
                e.xchg_forward(pb, lg)
                e.sync()
                outs.append(lg)
        else:
            req, counts = [], []
            for e, pb in zip(self.engs, pbs):
                buf = torch.empty(pb.batch_size * max(e.n_slots, 1), dtype=torch.int32, device=dev)
                counts.append(e.shard_requests(pb, buf))
                req.append(buf[:sum(counts[-1])])
            recv_rows, recv_counts = route_all_to_all(req, counts)
            replies = []
            for e, rr in zip(self.engs, recv_rows):
                rep = torch.empty(max(rr.numel(), 1) * rw, dtype=torch.float32, device=dev)
                e.shard_serve(rr.contiguous(), rr.numel(), rep)
                e.sync()
                replies.append(rep[:rr.numel() * rw])
            rowbufs, _ = route_all_to_all(replies, recv_counts, rw)
            for e, pb, rb in zip(self.engs, pbs, rowbufs):
                lg = torch.empty(pb.batch_size, dtype=torch.float32, device=dev)
                rbc = rb.contiguous() if rb.numel() else torch.zeros(rw, dtype=torch.float32, device=dev)
                e.shard_forward(pb, rbc, lg)
                e.sync()
                outs.append(lg)
        return outs

    def state(self, names_with_slots):
        """Global arrays reassembled from the shards (dense variables from rank 0)."""
        out = {}
        for name in names_with_slots:
            base = name.split("/")[0]
            if base in ("emb", "lin"):
                parts = [e.get_tensor(name) for e in self.engs]
                R = sum(p.shape[0] for p in parts)
                full = np.empty((R,) + parts[0].shape[1:], dtype=np.float32)
                for r, p in enumerate(parts):
                    full[r::self.W] = p
                out[name] = full
            else:
                out[name] = self.engs[0].get_tensor(name)
        return out
