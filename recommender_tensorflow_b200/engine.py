"""Host-side driver of the C ABI: one `DeepFMEngine` = one `dfm_handle` (model instance on a GPU).

This is the layer `model_fn` (trainers/deep_fm.py) sits on.  It owns no arithmetic: it sorts the
feature columns into TF's model order, packs raw feature columns into one pinned arena and calls
libdeepfm_b200.so.  torch is used only as the pinned/device memory allocator.
"""
import ctypes as C

import os

import numpy as np

from . import _lib
from ._lib import DfmError

_ALIGN = 256


def default_optimizer(name="Adam", learning_rate=0.001):
    """Hyper-parameters of tf.train.<name>Optimizer(learning_rate) (trainers/model_utils.py:57-66)."""
    if name not in _lib.OPT_KIND:
        raise KeyError(name)   # same failure mode as optimizer_classes[optimizer_name]
    if name == "RMSProp":   # tf.train.RMSPropOptimizer defaults: decay 0.9, momentum 0, epsilon 1e-10, rms slot = ones
        return dict(name=name, lr=float(learning_rate), beta1=0.0, beta2=0.9, eps=1e-10, init_acc=1.0)
    return dict(name=name, lr=float(learning_rate), beta1=0.9, beta2=0.999, eps=1e-8, init_acc=0.1)


def _opt_struct(o):
    return _lib.Optimizer(_lib.OPT_KIND[o["name"]], o["lr"], o.get("beta1", 0.9), o.get("beta2", 0.999),
                          o.get("eps", 1e-8), o.get("init_acc", 0.1))


def _torch():
    import torch
    return torch


def cross_spec(column, feature_dtypes=None, multivalent=None):
    """Resolve a feature_column.CrossedColumn into the spec the library takes: the constituents become source specs in
    HASHING order.  TF-1.12 `_CrossedColumn._transform_feature` flattens nested crosses (`_collect_leaf_level_keys`) and
    `sparse_ops._sparse_cross_internal` hands SparseTensor inputs to the op before dense ones, keeping key order within
    each group: categorical keys and multivalent raw keys are sparse, single-valued raw keys (decode_csv output) dense."""
    from .feature_column import DEFAULT_HASH_KEY
    fd, mv = dict(feature_dtypes or {}), dict(multivalent or {})
    sparse, dense = [], []
    for key in column.leaf_keys():
        if isinstance(key, str):
            if key not in fd:
                raise ValueError("crossed_column %s: dtype of raw feature %r is unknown (pass it in feature_dtypes)"
                                 % (column.name, key))
            d = fd[key]
            if d not in ("int32", "string"):
                raise ValueError("crossed_column %s: raw feature %r is %s; sparse_cross takes only int64 and string inputs"
                                 % (column.name, key, d))
            s = dict(name=key, source=key, kind="raw", dtype=d, num_buckets=0, width=int(mv.get(key, 1)))
            (sparse if s["width"] > 1 else dense).append(s)
        else:
            s = key.spec()
            s["width"] = int(mv.get(s["source"], 1))
            if s["kind"] == "bucketized":
                s["dtype"] = fd.get(s["source"], key.source_column.dtype)
                if s["dtype"] == "string":
                    raise ValueError("bucketized column %s needs a numeric feature" % s["name"])
            sparse.append(s)
    keys = sparse + dense
    if len(keys) > _lib.MAX_CROSS_KEYS:
        raise ValueError("crossed_column %s: %d keys, at most %d are supported" % (column.name, len(keys), _lib.MAX_CROSS_KEYS))
    width = int(np.prod([k["width"] for k in keys]))
    return dict(name=column.name, source=None, kind="crossed", dtype=None, num_buckets=int(column.hash_bucket_size),
                hash_key=int(column.hash_key or DEFAULT_HASH_KEY), keys=keys, width=width)


def pack_vocabulary(vocab, dtype):
    """A vocabulary as dfm_column takes it: strings -> (uint8 bytes, int64 offsets[V + 1]), ints -> int64[V]."""
    if dtype != "string":
        return np.ascontiguousarray(np.array(vocab, dtype=np.int64))
    enc = [v if isinstance(v, bytes) else v.encode() for v in vocab]
    offsets = np.zeros(len(enc) + 1, dtype=np.int64)
    np.cumsum(np.fromiter(map(len, enc), dtype=np.int64, count=len(enc)), out=offsets[1:])
    data = np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8)
    return data, offsets


class PackedBatch:
    """Raw feature columns of one batch laid out back to back in one arena (host pinned or device)."""

    def __init__(self, arena, base_ptr, raw, keep, nbytes, batch_size, on_device, layout=None):
        self.arena, self.base_ptr, self.raw, self._keep = arena, base_ptr, raw, keep
        self.nbytes, self.batch_size, self.on_device = nbytes, batch_size, on_device
        self.layout = layout or []        # [(kind, index, byte offset, bytes)] of the columns inside the arena


class DeepFMEngine:
    def __init__(self, categorical_columns, numeric_columns=(), embedding_size=4, hidden_units=(16, 16),
                 use_linear=True, use_mf=True, use_dnn=True, loss_reduction="mean", opt_deep=None,
                 opt_linear=None, max_batch=65536, device=0, feature_dtypes=None, sort_columns=True, rank=0, world=1, dropout=0.0, dropout_seed=0,
                 multivalent=None, activation="relu"):
        self.lib = _lib.load()
        # params["activation"] (trainers/deep_fm.py:22): a name, None (identity) or a callable named like a tf.nn activation
        act = activation if (activation is None or isinstance(activation, str)) else getattr(activation, "__name__", str(activation))
        if act not in _lib.ACTIVATIONS:
            raise ValueError("activation %r is not one of %s" % (activation, sorted(k for k in _lib.ACTIVATIONS if k)))
        self.activation = "identity" if act in (None, "linear") else act
        cats = list(categorical_columns)
        nums = list(numeric_columns)
        if sort_columns:   # tf.feature_column.input_layer / linear_model iterate columns sorted by name
            cats = sorted(cats, key=lambda c: c.name + "_embedding")
            nums = sorted(nums, key=lambda c: c.name)
        self.cat_columns, self.num_columns = cats, nums
        self.k = int(embedding_size)
        self.hidden = [int(x) for x in hidden_units]
        self.use_linear, self.use_mf, self.use_dnn = bool(use_linear), bool(use_mf), bool(use_dnn)
        self.loss_reduction = loss_reduction
        self.opt_deep = opt_deep or default_optimizer()
        self.opt_linear = opt_linear or default_optimizer()
        self.max_batch, self.device = int(max_batch), int(device)
        self.rank, self.world = int(rank), int(world)
        self.dropout, self.dropout_seed = float(dropout or 0.0), int(dropout_seed)
        fd = dict(feature_dtypes or {})
        mv = dict(multivalent or {})      # raw feature key -> value slots per sample (multi-hot / multivalent column)
        self.specs = []
        # source columns of crossed columns (deduplicated); their raw data follows the model columns' in a batch
        self.src_specs = []
        for c in cats:
            if c.kind == "crossed":
                s = cross_spec(c, fd, mv)
                s["key_idx"] = []
                for k in s["keys"]:
                    if k not in self.src_specs:
                        self.src_specs.append(k)
                    s["key_idx"].append(self.src_specs.index(k))
                self.specs.append(s)
                continue
            s = c.spec()
            s["width"] = int(mv.get(s["source"], 1))
            if s["kind"] == "bucketized":
                s["dtype"] = fd.get(s["source"], c.source_column.dtype)
            self.specs.append(s)
        # every raw column a batch carries, in cat_data order: model columns (a crossed one has none), then sources
        self.raw_specs = self.specs + self.src_specs
        self.num_buckets = [int(s["num_buckets"]) for s in self.specs]
        self.n_slots = sum(s["width"] for s in self.specs)
        self.row_offsets = np.concatenate([[0], np.cumsum(self.num_buckets)]).astype(np.int64)
        self._keep = []
        cols = (_lib.Column * max(len(cats), 1))()
        srcs = (_lib.Column * max(len(self.src_specs), 1))()
        for col, s in list(zip(cols, self.specs)) + list(zip(srcs, self.src_specs)):
            col.name = s["name"].encode()
            col.kind = _lib.COL_KIND[s["kind"]]
            col.dtype = _lib.DTYPE[s["dtype"] or "int32"]
            col.num_buckets = s["num_buckets"]
            col.width = s["width"]
            if s["kind"] == "crossed":
                arr = (C.c_int32 * len(s["key_idx"]))(*s["key_idx"])
                self._keep.append(arr)
                col.n_keys, col.keys, col.hash_key = len(s["key_idx"]), C.cast(arr, C.POINTER(C.c_int32)), s["hash_key"]
            if s["kind"] == "bucketized":
                arr = (C.c_float * len(s["boundaries"]))(*s["boundaries"])
                self._keep.append(arr)
                col.boundaries = C.cast(arr, C.POINTER(C.c_float))
                col.n_boundaries = len(s["boundaries"])
            if s["kind"] == "vocab":
                packed = pack_vocabulary(s["vocab"], s["dtype"])
                self._keep.append(packed)
                if s["dtype"] == "string":
                    col.vocab_data = packed[0].ctypes.data
                    col.vocab_offsets = packed[1].ctypes.data_as(C.POINTER(C.c_int64))
                else:
                    col.vocab_int = packed.ctypes.data_as(C.POINTER(C.c_int64))
                col.vocab_size = len(s["vocab"])
                col.num_oov = s["num_oov"]
            if s["kind"] in ("vocab", "identity") and s.get("default_value") not in (None, -1):
                col.default_value, col.has_default = int(s["default_value"]), 1
        hid = (C.c_int32 * max(len(self.hidden), 1))(*self.hidden)
        cfg = _lib.Config(len(cats), C.cast(cols, C.POINTER(_lib.Column)), len(nums), self.k, len(self.hidden),
                          C.cast(hid, C.POINTER(C.c_int32)), int(self.use_linear), int(self.use_mf), int(self.use_dnn),
                          _lib.LOSS_RED[loss_reduction], _opt_struct(self.opt_deep), _opt_struct(self.opt_linear),
                          self.max_batch, self.device, self.rank, self.world, None, self.dropout, self.dropout_seed,
                          _lib.ACTIVATIONS[self.activation], len(self.src_specs), C.cast(srcs, C.POINTER(_lib.Column)))
        self._keep += [cols, srcs, hid]
        handle = C.c_void_p()
        rc = self.lib.dfm_create(C.byref(cfg), C.byref(handle))
        if rc != _lib.DFM_OK:
            msg = (self.lib.dfm_last_error(None) or b"").decode()
            if rc == -1:
                raise ValueError(msg)      # same exception type as trainers/deep_fm.py:31-34
            raise DfmError(rc, msg)
        self.h = handle

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc):
        if rc != _lib.DFM_OK:
            raise DfmError(rc, (self.lib.dfm_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.dfm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def global_step(self):
        return int(self.lib.dfm_global_step(self.h))

    def state_checksum(self):
        """order-independent 64-bit checksum of the whole trained state on this handle (flushes first)"""
        v = C.c_uint64(0)
        self._check(self.lib.dfm_state_checksum(self.h, C.byref(v)))
        return int(v.value)

    @property
    def last_unique_rows(self):
        return int(self.lib.dfm_last_unique_rows(self.h))

    @property
    def last_step_launches(self):
        return int(self.lib.dfm_last_step_launches(self.h))

    @property
    def graph_steps(self):
        """train steps replayed as a single CUDA graph (small batches)"""
        return int(self.lib.dfm_graph_steps(self.h))

    def sync(self):
        self._check(self.lib.dfm_sync(self.h))

    def flush(self):
        self._check(self.lib.dfm_flush(self.h, None))

    def set_profiling(self, on=True):
        self._check(self.lib.dfm_set_profiling(self.h, int(on)))

    def phase_ms(self):
        names = ["transform", "sort", "segments", "catchup", "gather", "mlp_fwd", "loss", "mlp_bwd", "reduce",
                 "update", "dense"]
        return {n: float(self.lib.dfm_phase_ms(self.h, n.encode())) for n in names}

    # ------------------------------------------------------------------ variables
    def tensor_shape(self, name):
        r, e = C.c_int64(), C.c_int64()
        self._check(self.lib.dfm_tensor_rows(self.h, name.encode(), C.byref(r), C.byref(e)))
        return int(r.value), int(e.value)

    def variable_names(self):
        names = []
        if self.use_mf or self.use_dnn:
            names.append("emb")
            if self.num_columns:
                names.append("num_emb")
        if self.use_dnn:
            for i in range(len(self.hidden)):
                names += ["W%d" % i, "b%d" % i]
            names += ["Wo", "bo"]
        if self.use_linear:
            names.append("lin")
            if self.num_columns:
                names.append("num_lin")
            names.append("bias")
        return names

    def slot_names(self, var):
        grp = self.opt_linear if var in ("lin", "num_lin", "bias") else self.opt_deep
        return {"Adam": ["m", "v"], "Adagrad": ["acc"], "Ftrl": ["acc", "lin"], "SGD": [], "RMSProp": ["rms", "mom"]}[grp["name"]]

    def set_tensor(self, name, value, row_begin=0):
        value = np.ascontiguousarray(value, dtype=np.float32)
        rows, elems = self.tensor_shape(name)
        n_rows = value.size // max(elems, 1)
        self._check(self.lib.dfm_set_tensor(self.h, name.encode(), row_begin, n_rows, value.ctypes.data_as(C.c_void_p)))

    def get_tensor(self, name, row_begin=0, n_rows=None):
        rows, elems = self.tensor_shape(name)
        n_rows = rows - row_begin if n_rows is None else n_rows
        out = np.empty((n_rows, elems), dtype=np.float32)
        self._check(self.lib.dfm_get_tensor(self.h, name.encode(), row_begin, n_rows, out.ctypes.data_as(C.c_void_p)))
        return out

    def set_weights(self, weights):
        for name, val in weights.items():
            self.set_tensor(name, val)

    def state(self):
        """All variables and optimizer slots, keyed like oracle.deepfm.OracleDeepFM.state()."""
        out = {}
        for v in self.variable_names():
            out[v] = self.get_tensor(v)
            for s in self.slot_names(v):
                out[v + "/" + s] = self.get_tensor(v + "/" + s)
        return out

    # ------------------------------------------------------------------ checkpoints (tf.train.Saver surface)
    def tf_variable_map(self, scheme="deep_fm"):
        """TF-1.12 checkpoint variable name -> (generic tensor name, row_begin, n_rows, shape).
        scheme 'deep_fm': names created by trainers/deep_fm.py::model_fn; 'canned': DNNLinearCombinedClassifier."""
        m = {}
        emb_fmt = ("input_layer/input_layer/%s_embedding/embedding_weights" if scheme == "deep_fm"
                   else "dnn/input_from_feature_columns/input_layer/%s_embedding/embedding_weights")
        for f, s in enumerate(self.specs):
            r0, n = int(self.row_offsets[f]), int(self.num_buckets[f])
            if self.use_mf or self.use_dnn:
                m[emb_fmt % s["name"]] = ("emb", r0, n, (n, self.k))
            if self.use_linear:
                m["linear/linear_model/%s/weights" % s["name"]] = ("lin", r0, n, (n, 1))
        dn = len(self.num_columns)
        if dn and (self.use_mf or self.use_dnn):
            m["input_layer/numeric_embeddings"] = ("num_emb", 0, dn, (1, dn, self.k))
        if self.use_linear:
            for j, c in enumerate(self.num_columns):
                m["linear/linear_model/%s/weights" % c.key] = ("num_lin", j, 1, (1, 1))
            m["linear/linear_model/bias_weights"] = ("bias", 0, 1, (1,))
        if self.use_dnn:
            pre = "dnn/dnn/" if scheme == "deep_fm" else "dnn/"
            mid = "/dense" if scheme == "deep_fm" else ""
            fan_in = (len(self.specs) + dn) * self.k
            for i, hsz in enumerate(self.hidden):
                m["%shiddenlayer_%d%s/kernel" % (pre, i, mid)] = ("W%d" % i, 0, fan_in, (fan_in, hsz))
                m["%shiddenlayer_%d%s/bias" % (pre, i, mid)] = ("b%d" % i, 0, hsz, (hsz,))
                fan_in = hsz
            m["%slogits%s/kernel" % (pre, mid)] = ("Wo", 0, fan_in, (fan_in, 1))
            m["%slogits%s/bias" % (pre, mid)] = ("bo", 0, 1, (1,))
        return m

    _SLOT_TF = {"m": "Adam", "v": "Adam_1", "acc": {"Adagrad": "Adagrad", "Ftrl": "accum"}, "lin": "linear",
                "rms": "RMSProp", "mom": "RMSProp_1"}

    def save_checkpoint(self, path, scheme="deep_fm"):
        """Variables + optimizer slots + global_step under TF-1.12 names, as one .npz (flushes deferred Adam)."""
        out = {"global_step": np.int64(self.global_step)}
        for tf_name, (g, r0, n, shape) in self.tf_variable_map(scheme).items():
            out[tf_name] = self.get_tensor(g, r0, n).reshape(shape)
            grp = self.opt_linear if g in ("lin", "num_lin", "bias") else self.opt_deep
            for sl in self.slot_names(g):
                t = self._SLOT_TF[sl]
                t = t[grp["name"]] if isinstance(t, dict) else t
                out[tf_name + "/" + t] = self.get_tensor(g + "/" + sl, r0, n).reshape(shape)
        # TF keeps the running products beta1_power / beta2_power as variables; here they are a function of global_step
        # (dfm_set_global_step rebuilds them with the same float32 running product), stored for inspection / exchange
        for grp_name, grp in (("deep", self.opt_deep), ("linear", self.opt_linear)):
            if grp["name"] == "Adam":
                b1p, b2p = np.float32(1.0), np.float32(1.0)
                for _ in range(int(self.global_step)):
                    b1p, b2p = np.float32(b1p * np.float32(grp["beta1"])), np.float32(b2p * np.float32(grp["beta2"]))
                out["beta1_power/" + grp_name], out["beta2_power/" + grp_name] = b1p, b2p
        # written next to the target and renamed into place: a crash mid-write never leaves a truncated model.ckpt-N.npz
        tmp = path + ".tmp.npz"
        np.savez(tmp, **out)
        os.replace(tmp, path)
        return path

    def load_checkpoint(self, path, scheme="deep_fm"):
        data = np.load(path)
        for tf_name, (g, r0, n, shape) in self.tf_variable_map(scheme).items():
            self.set_tensor(g, data[tf_name].reshape(n, -1), r0)
            grp = self.opt_linear if g in ("lin", "num_lin", "bias") else self.opt_deep
            for sl in self.slot_names(g):
                t = self._SLOT_TF[sl]
                t = t[grp["name"]] if isinstance(t, dict) else t
                self.set_tensor(g + "/" + sl, data[tf_name + "/" + t].reshape(n, -1), r0)
        self._check(self.lib.dfm_set_global_step(self.h, int(data["global_step"])))

    # -- row-sharded handles (world > 1): one shard file per rank, merged on the host when an unsharded checkpoint is wanted
    def _shard_tensor_names(self):
        names = []
        for v in self.variable_names():
            names.append(v)
            names += [v + "/" + sl for sl in self.slot_names(v)]
        return names

    def save_checkpoint_shard(self, path):
        """This rank's rows of every table (+ slots), the replicated dense tower and global_step as one .npz (flushes the
        deferred Adam).  Table tensors hold the LOCAL rows: global row g lives on rank g % world at index g // world."""
        out = {"global_step": np.int64(self.global_step), "rank": np.int64(self.rank), "world": np.int64(self.world)}
        for n in self._shard_tensor_names():
            out[n] = self.get_tensor(n)
        tmp = path + ".tmp.npz"
        np.savez(tmp, **out)
        os.replace(tmp, path)
        return path

    def load_checkpoint_shard(self, path):
        data = np.load(path)
        if int(data["rank"]) != self.rank or int(data["world"]) != self.world:
            raise ValueError("shard %s belongs to rank %d of %d" % (path, int(data["rank"]), int(data["world"])))
        for n in self._shard_tensor_names():
            self.set_tensor(n, data[n])
        self._check(self.lib.dfm_set_global_step(self.h, int(data["global_step"])))

    def merge_checkpoint_shards(self, shard_paths, out_path, scheme="deep_fm"):
        """Host-side gather of the rows: the shard files of every rank -> ONE checkpoint under the TF-1.12 variable names,
        loadable by an unsharded engine of the same model (load_checkpoint).  `self` only supplies the variable map."""
        shards = sorted((np.load(p) for p in shard_paths), key=lambda d: int(d["rank"]))
        world = int(shards[0]["world"])
        if [int(d["rank"]) for d in shards] != list(range(world)):
            raise ValueError("need exactly one shard per rank 0..%d" % (world - 1))
        R = int(self.row_offsets[-1])

        def full(name):
            base = name.split("/")[0]
            if base not in ("emb", "lin"):
                return shards[0][name]                      # replicated
            width = shards[0][name].shape[1]
            g = np.empty((R, width), dtype=np.float32)
            for r, d in enumerate(shards):
                g[r::world] = d[name][:len(range(r, R, world))]
            return g
        out = {"global_step": np.int64(int(shards[0]["global_step"]))}
        for tf_name, (gname, r0, n, shape) in self.tf_variable_map(scheme).items():
            out[tf_name] = full(gname)[r0:r0 + n].reshape(shape)
            grp = self.opt_linear if gname in ("lin", "num_lin", "bias") else self.opt_deep
            for sl in self.slot_names(gname):
                t = self._SLOT_TF[sl]
                t = t[grp["name"]] if isinstance(t, dict) else t
                out[tf_name + "/" + t] = full(gname + "/" + sl)[r0:r0 + n].reshape(shape)
        tmp = out_path + ".tmp.npz"
        np.savez(tmp, **out)
        os.replace(tmp, out_path)
        return out_path

    def init_random(self, seed=0):
        self._check(self.lib.dfm_init_random(self.h, seed))

    # ------------------------------------------------------------------ batches
    def _segments(self, features, labels):
        """-> list of (kind, index, ndarray) in arena order; kind in cat|off|num|lab."""
        segs = []
        B = None
        for f, s in enumerate(self.raw_specs):
            if s["kind"] == "crossed":
                continue
            raw = features[s["source"]]
            if s["dtype"] == "string":
                if isinstance(raw, tuple):
                    data, offs = raw
                    data = np.ascontiguousarray(data, dtype=np.uint8)
                    offs = np.ascontiguousarray(offs, dtype=np.int32)
                else:
                    vals = [v if isinstance(v, bytes) else str(v).encode() for v in np.asarray(raw, dtype=object).reshape(-1)]
                    lens = np.fromiter((len(v) for v in vals), dtype=np.int64, count=len(vals))
                    offs = np.zeros(len(vals) + 1, dtype=np.int32)
                    np.cumsum(lens, out=offs[1:])
                    data = np.frombuffer(b"".join(vals) or b"\0", dtype=np.uint8)
                n = (offs.shape[0] - 1) // s["width"]
                segs += [("off", f, offs), ("cat", f, data)]
            else:
                arr = np.asarray(raw).reshape(-1)          # multivalent: [B, width] row-major
                want = np.int32 if s["dtype"] == "int32" else np.float32
                if arr.dtype != want:
                    arr = arr.astype(want)
                n = arr.shape[0] // s["width"]
                segs.append(("cat", f, np.ascontiguousarray(arr)))
            if B is None:
                B = n
            elif B != n:
                raise ValueError("feature %s has %d rows, expected %d" % (s["source"], n, B))
        for j, c in enumerate(self.num_columns):
            arr = np.ascontiguousarray(np.asarray(features[c.key]).reshape(-1), dtype=np.float32)
            if B is None:
                B = arr.shape[0]
            segs.append(("num", j, arr))
        if labels is not None:
            segs.append(("lab", 0, np.ascontiguousarray(np.asarray(labels).reshape(-1), dtype=np.float32)))
        return segs, B

    def pack(self, features, labels=None, device=False, pinned=True):
        """Lay the raw columns out in ONE arena so that the H2D transfer is a single copy."""
        segs, B = self._segments(features, labels)
        offs, total = [], 0
        for _, _, a in segs:
            offs.append(total)
            total += (a.nbytes + _ALIGN - 1) // _ALIGN * _ALIGN
        total = max(total, _ALIGN)
        keep = []
        if device or pinned:
            torch = _torch()
        if pinned and not device and torch.cuda.is_available():
            host = torch.empty(total, dtype=torch.uint8).pin_memory()
        elif device:
            host = torch.empty(total, dtype=torch.uint8)
        else:
            host = None
        if host is not None:
            hv = host.numpy()
        else:
            hv = np.empty(total, dtype=np.uint8)
        for (kind, idx, a), o in zip(segs, offs):
            hv[o:o + a.nbytes] = a.view(np.uint8).reshape(-1)
        if device:
            arena = host.to("cuda:%d" % self.device)
            base = arena.data_ptr()
        elif host is not None:
            arena, base = host, host.data_ptr()
        else:
            arena, base = hv, hv.ctypes.data
        nc, nn = max(len(self.raw_specs), 1), max(len(self.num_columns), 1)
        cat = (C.c_void_p * nc)()
        off = (C.c_void_p * nc)()
        num = (C.c_void_p * nn)()
        lab = None
        for (kind, idx, a), o in zip(segs, offs):
            if kind == "cat":
                cat[idx] = base + o
            elif kind == "off":
                off[idx] = base + o
            elif kind == "num":
                num[idx] = base + o
            else:
                lab = base + o
        raw = _lib.RawBatch(B, C.cast(cat, C.POINTER(C.c_void_p)), C.cast(off, C.POINTER(C.c_void_p)),
                            C.cast(num, C.POINTER(C.c_void_p)), lab)
        keep += [cat, off, num]
        layout = [(kind, idx, o, a.nbytes) for (kind, idx, a), o in zip(segs, offs)]
        return PackedBatch(arena, base, raw, keep, total, B, device, layout)

    def repack_like(self, pb, arena):
        """A PackedBatch over another arena (torch uint8 tensor, host pinned or device) with pb's column layout."""
        base = arena.data_ptr()
        nc, nn = max(len(self.raw_specs), 1), max(len(self.num_columns), 1)
        cat = (C.c_void_p * nc)()
        off = (C.c_void_p * nc)()
        num = (C.c_void_p * nn)()
        lab = None
        for kind, idx, o, _ in pb.layout:
            if kind == "cat":
                cat[idx] = base + o
            elif kind == "off":
                off[idx] = base + o
            elif kind == "num":
                num[idx] = base + o
            else:
                lab = base + o
        raw = _lib.RawBatch(pb.batch_size, C.cast(cat, C.POINTER(C.c_void_p)), C.cast(off, C.POINTER(C.c_void_p)),
                            C.cast(num, C.POINTER(C.c_void_p)), lab)
        return PackedBatch(arena, base, raw, [cat, off, num], pb.nbytes, pb.batch_size, arena.is_cuda, pb.layout)

    def _as_batch(self, features, labels, device=False):
        if isinstance(features, PackedBatch):
            return features
        return self.pack(features, labels, device=device)

    # ------------------------------------------------------------------ the hot path
    def transform(self, features):
        """ids [B, n_cat] int32 in model order (-1 = empty bag): K1 alone."""
        torch = _torch()
        pb = self._as_batch(features, None, device=True)
        out = torch.empty((pb.batch_size, self.n_slots), dtype=torch.int32, device="cuda:%d" % self.device)
        self._check(self.lib.dfm_transform(self.h, C.byref(pb.raw), C.c_void_p(out.data_ptr()), None))
        self.sync()
        return out.cpu().numpy()

    def train_step(self, features, labels=None, return_logits=False):
        """One train step from HOST buffers (H2D + step + D2H of the loss)."""
        pb = self._as_batch(features, labels)
        if pb.on_device:
            return self.train_step_device(pb, return_logits)
        loss = C.c_float()
        logits = np.empty(pb.batch_size, dtype=np.float32) if return_logits else None
        self._check(self.lib.dfm_train_step_host(self.h, C.byref(pb.raw), C.byref(loss),
                                                 logits.ctypes.data_as(C.c_void_p) if return_logits else None))
        return (float(loss.value), logits) if return_logits else float(loss.value)

    def train_step_async(self, pb):
        """Pipelined host step: returns the loss of the previously enqueued step (NaN on the first)."""
        prev = C.c_float()
        self._check(self.lib.dfm_train_step_host_async(self.h, C.byref(pb.raw), C.byref(prev)))
        return float(prev.value)

    def drain(self):
        last = C.c_float()
        self._check(self.lib.dfm_train_step_host_drain(self.h, C.byref(last)))
        return float(last.value)

    def train_step_device(self, pb, return_logits=False, loss_out=None, stream=None):
        """One train step on a device-resident PackedBatch; enqueues only (no sync) unless logits are wanted."""
        torch = _torch()
        dev = "cuda:%d" % self.device
        if loss_out is None:
            loss_out = torch.empty(1, dtype=torch.float32, device=dev)
        logits = torch.empty(pb.batch_size, dtype=torch.float32, device=dev) if return_logits else None
        self._check(self.lib.dfm_train_step(self.h, C.byref(pb.raw), C.c_void_p(loss_out.data_ptr()),
                                            C.c_void_p(logits.data_ptr()) if return_logits else None,
                                            C.c_void_p(stream) if stream else None))
        if return_logits:
            self.sync()
            return float(loss_out.item()), logits.cpu().numpy()
        return loss_out

    def prefetch(self, pb, after_stream=None):
        """Input-pipeline lookahead: compute the ids / sort / segments of the NEXT device batch on the library's side
        stream while the current step runs; the next train_step_device(pb) adopts them."""
        self._check(self.lib.dfm_prefetch_batch(self.h, C.byref(pb.raw), C.c_void_p(after_stream) if after_stream else None))

    def predict_logits(self, features):
        pb = self._as_batch(features, None)
        out = np.empty(pb.batch_size, dtype=np.float32)
        if pb.on_device:
            torch = _torch()
            t = torch.empty(pb.batch_size, dtype=torch.float32, device="cuda:%d" % self.device)
            self._check(self.lib.dfm_forward(self.h, C.byref(pb.raw), C.c_void_p(t.data_ptr()), None))
            self.sync()
            return t.cpu().numpy()
        self._check(self.lib.dfm_forward_host(self.h, C.byref(pb.raw), out.ctypes.data_as(C.c_void_p)))
        return out

    # ------------------------------------------------------------------ layer_summary side outputs
    def summary_names(self):
        """TF name scopes of the tensors trainers/deep_fm.py passes to layer_summary, in the library's order."""
        names = []
        if self.use_linear:
            names.append("linear/linear")
        if self.use_mf:
            names.append("mf/logits")
        if self.use_dnn:
            names += ["dnn/dnn/hiddenlayer_%d" % i for i in range(len(self.hidden))] + ["dnn/dnn/logits"]
        return names + ["deep_fm/logits"]

    @staticmethod
    def summary_bucket_limits():
        n = C.c_int32(0)
        lib = _lib.load()
        lib.dfm_summary_bucket_limits(None, C.byref(n))
        lim = np.empty(n.value, dtype=np.float64)
        lib.dfm_summary_bucket_limits(lim.ctypes.data_as(C.POINTER(C.c_double)), C.byref(n))
        return lim

    def layer_summary(self, features, train=True):
        """trainers/model_utils.py:4-6 for every tensor the reference summarises (trainers/deep_fm.py:43,89,105,110,115),
        computed on the device for this batch with the weights as of the latest step (call it BEFORE the train step whose
        summaries it stands for).  -> {scope: {"fraction_of_zero_values": f, "activation": HistogramProto fields}}"""
        pb = features if isinstance(features, PackedBatch) else self.pack(features, None, device=True)
        names = self.summary_names()
        limits = self.summary_bucket_limits()
        stats = np.zeros((len(names), 6), dtype=np.float64)
        buckets = np.zeros((len(names), limits.size), dtype=np.int64)
        n = C.c_int32(0)
        self._check(self.lib.dfm_layer_summary(self.h, C.byref(pb.raw), int(bool(train)), stats.ctypes.data_as(C.c_void_p),
                                               buckets.ctypes.data_as(C.c_void_p), len(names), C.byref(n)))
        assert n.value == len(names)
        out = {}
        for i, name in enumerate(names):
            nz = np.nonzero(buckets[i])[0]
            out[name] = {"fraction_of_zero_values": float(stats[i, 5]),
                         "activation": {"min": float(stats[i, 0]), "max": float(stats[i, 1]), "num": float(stats[i, 2]),
                                        "sum": float(stats[i, 3]), "sum_squares": float(stats[i, 4]),
                                        "bucket_limit": limits[nz].tolist(), "bucket": buckets[i, nz].astype(np.float64).tolist()}}
        return out

    def summary_tensor(self, which, n):
        """host copy of a tensor of the last layer_summary call (0 linear, 1 mf, 2 hidden, 3 dnn logit, 4 logits)"""
        out = np.empty(int(n), dtype=np.float32)
        self._check(self.lib.dfm_layer_summary_tensor(self.h, int(which), int(n), out.ctypes.data_as(C.c_void_p)))
        return out

    # ------------------------------------------------------------------ row sharding (world > 1)
    @property
    def row_width(self):
        return int(self.lib.dfm_shard_row_width(self.h))

    @property
    def dense_size(self):
        return int(self.lib.dfm_dense_size(self.h))

    def shard_requests(self, pb, req_rows_out, stream=None):
        """-> counts per owner (list of ints); req_rows_out (int32 cuda tensor) receives the unique local-row ids."""
        counts = (C.c_int32 * self.world)()
        self._check(self.lib.dfm_shard_requests(self.h, C.byref(pb.raw), C.c_void_p(req_rows_out.data_ptr()), counts,
                                                C.c_void_p(stream) if stream else None))
        return list(counts)

    def shard_serve(self, recv_rows, n_recv, reply, stream=None):
        self._check(self.lib.dfm_shard_serve(self.h, C.c_void_p(recv_rows.data_ptr()), int(n_recv), C.c_void_p(reply.data_ptr()),
                                             C.c_void_p(stream) if stream else None))

    def shard_forward_backward(self, pb, rowbuf, global_batch, loss, logits, gsum, dense_grad, stream=None):
        self._check(self.lib.dfm_shard_forward_backward(
            self.h, C.byref(pb.raw), C.c_void_p(rowbuf.data_ptr()), int(global_batch), C.c_void_p(loss.data_ptr()),
            C.c_void_p(logits.data_ptr()) if logits is not None else None, C.c_void_p(gsum.data_ptr()),
            C.c_void_p(dense_grad.data_ptr()), C.c_void_p(stream) if stream else None))

    def shard_apply(self, grecv, dense_grad, stream=None):
        self._check(self.lib.dfm_shard_apply(self.h, C.c_void_p(grecv.data_ptr()), C.c_void_p(dense_grad.data_ptr()),
                                             C.c_void_p(stream) if stream else None))

    def shard_requests_counts(self, pb, stream=None):
        counts = (C.c_int32 * self.world)()
        self._check(self.lib.dfm_shard_requests(self.h, C.byref(pb.raw), None, counts, C.c_void_p(stream) if stream else None))
        return list(counts)

    def shard_forward(self, pb, rowbuf, logits, stream=None):
        """forward pass alone on the served rows (collective path)"""
        self._check(self.lib.dfm_shard_forward(self.h, C.byref(pb.raw), C.c_void_p(rowbuf.data_ptr()),
                                               C.c_void_p(logits.data_ptr()), C.c_void_p(stream) if stream else None))

    # ---- flag-synchronised exchange over peer memory (include/deepfm_b200.h: dfm_xchg_*) ----
    def xchg_export(self):
        buf = (C.c_ubyte * 64)()
        self._check(self.lib.dfm_xchg_export(self.h, buf))
        return bytes(buf)

    def xchg_import(self, all_handles):
        assert len(all_handles) == self.world * 64
        buf = (C.c_ubyte * len(all_handles)).from_buffer_copy(all_handles)
        self._check(self.lib.dfm_xchg_import(self.h, buf))

    def xchg_buffer(self):
        out = C.c_void_p()
        self._check(self.lib.dfm_xchg_buffer(self.h, C.byref(out)))
        return int(out.value)

    def xchg_set_peers(self, ptrs):
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        self._check(self.lib.dfm_xchg_set_peers(self.h, arr))

    def xchg_begin(self, pb, stream=None):
        self._check(self.lib.dfm_xchg_begin(self.h, C.byref(pb.raw), C.c_void_p(stream) if stream else None))

    def xchg_serve(self, train=True, stream=None):
        self._check(self.lib.dfm_xchg_serve(self.h, int(bool(train)), C.c_void_p(stream) if stream else None))

    def xchg_forward_backward(self, pb, global_batch, logits=None, stream=None):
        self._check(self.lib.dfm_xchg_forward_backward(self.h, C.byref(pb.raw), int(global_batch),
                                                       C.c_void_p(logits.data_ptr()) if logits is not None else None,
                                                       C.c_void_p(stream) if stream else None))

    def xchg_apply(self, loss_out, stream=None):
        self._check(self.lib.dfm_xchg_apply(self.h, C.c_void_p(loss_out.data_ptr()), C.c_void_p(stream) if stream else None))

    def xchg_train_step(self, pb, global_batch, loss_out, logits=None, stream=None, next_pb=None):
        """one whole sharded step: launches only (no collective, no host synchronisation).  next_pb: the batch of the NEXT
        step; its requests are computed beside this step's apply phase (the next call must then be given that batch)."""
        self._check(self.lib.dfm_xchg_train_step_next(self.h, C.byref(pb.raw), C.byref(next_pb.raw) if next_pb is not None else None,
                                                      int(global_batch), C.c_void_p(loss_out.data_ptr()),
                                                      C.c_void_p(logits.data_ptr()) if logits is not None else None,
                                                      C.c_void_p(stream) if stream else None))

    def xchg_forward(self, pb, logits, stream=None):
        self._check(self.lib.dfm_xchg_forward(self.h, C.byref(pb.raw), C.c_void_p(logits.data_ptr()), C.c_void_p(stream) if stream else None))

    def set_weights_sharded(self, weights):
        """Load GLOBAL arrays: table rows are sliced to the rows this rank owns (g % world == rank)."""
        for name, val in weights.items():
            base = name.split("/")[0]
            if base in ("emb", "lin"):
                val = np.asarray(val)[self.rank::self.world]
            self.set_tensor(name, val)
