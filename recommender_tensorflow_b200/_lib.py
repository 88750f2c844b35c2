"""ctypes binding of libdeepfm_b200.so (C ABI declared in include/deepfm_b200.h).

The product path has no CPU fallback: if the CUDA library is missing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdeepfm_b200.so")

DFM_OK = 0
ERRORS = {-1: "INVALID_ARG", -2: "CUDA", -3: "OUT_OF_RANGE", -4: "UNSUPPORTED", -5: "NCCL", -6: "NOT_FOUND", -7: "PARSE", -8: "PEER"}
MAX_CAT, MAX_NUM, MAX_HIDDEN = 64, 64, 8

COL_KIND = {"hash": 0, "bucketized": 1, "vocab": 2, "identity": 3, "crossed": 4, "raw": 5}
MAX_CROSS_KEYS = 8
DTYPE = {"int32": 0, "float32": 1, "string": 2}
OPT_KIND = {"Adam": 0, "Adagrad": 1, "Ftrl": 2, "SGD": 3, "RMSProp": 4}
LOSS_RED = {"mean": 0, "sum": 1}


class Column(C.Structure):
    _fields_ = [("name", C.c_char_p), ("kind", C.c_int32), ("dtype", C.c_int32), ("num_buckets", C.c_int64),
                ("boundaries", C.POINTER(C.c_float)), ("n_boundaries", C.c_int32),
                ("vocab", C.POINTER(C.c_char_p)), ("vocab_size", C.c_int32), ("num_oov", C.c_int32), ("width", C.c_int32),
                ("n_keys", C.c_int32), ("keys", C.POINTER(C.c_int32)), ("hash_key", C.c_uint64),
                ("vocab_data", C.c_void_p), ("vocab_offsets", C.POINTER(C.c_int64)), ("vocab_int", C.POINTER(C.c_int64)),
                ("default_value", C.c_int64), ("has_default", C.c_int32)]


class Optimizer(C.Structure):
    _fields_ = [("kind", C.c_int32), ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
                ("eps", C.c_float), ("init_acc", C.c_float)]


class Config(C.Structure):
    _fields_ = [("n_cat", C.c_int32), ("cat", C.POINTER(Column)), ("n_num", C.c_int32),
                ("embedding_size", C.c_int32), ("n_hidden", C.c_int32), ("hidden_units", C.POINTER(C.c_int32)),
                ("use_linear", C.c_int32), ("use_mf", C.c_int32), ("use_dnn", C.c_int32),
                ("loss_reduction", C.c_int32), ("opt_deep", Optimizer), ("opt_linear", Optimizer),
                ("max_batch", C.c_int32), ("device", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32),
                ("nccl_comm", C.c_void_p), ("dropout", C.c_float), ("head", C.c_int32), ("dropout_seed", C.c_uint64),
                ("activation", C.c_int32), ("n_src", C.c_int32), ("src", C.POINTER(Column)), ("weighted", C.c_int32)]
ACTIVATIONS = {"relu": 0, "tanh": 1, "sigmoid": 2, "identity": 3, "linear": 3, None: 3}
HEADS = {"logistic": 0, "squared": 1}       # DFM_HEAD_*


METRIC_BINS = 201        # DFM_METRIC_BINS


class MetricState(C.Structure):
    """dfm_metric_state: the raw EVAL metric state of a handle (include/deepfm_b200.h)"""
    _fields_ = [("n", C.c_int64), ("bin_count", (C.c_int64 * METRIC_BINS) * 2), ("tp", C.c_int64), ("fp", C.c_int64),
                ("fn", C.c_int64), ("correct", C.c_int64), ("bin_weight", (C.c_double * METRIC_BINS) * 2),
                ("w_tp", C.c_double), ("w_fp", C.c_double), ("w_fn", C.c_double), ("w_correct", C.c_double),
                ("sum_w", C.c_double), ("sum_wy", C.c_double), ("sum_wpred", C.c_double), ("sum_wloss", C.c_double)]


class RawBatch(C.Structure):
    _fields_ = [("batch_size", C.c_int32), ("cat_data", C.POINTER(C.c_void_p)),
                ("cat_offsets", C.POINTER(C.c_void_p)), ("num_data", C.POINTER(C.c_void_p)),
                ("labels", C.c_void_p), ("weights", C.c_void_p)]


_SIGS = {
    "dfm_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "dfm_destroy": (None, [C.c_void_p]),
    "dfm_last_error": (C.c_char_p, [C.c_void_p]),
    "dfm_tensor_rows": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfm_set_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64, C.c_int64, C.c_void_p]),
    "dfm_get_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64, C.c_int64, C.c_void_p]),
    "dfm_init_random": (C.c_int, [C.c_void_p, C.c_uint64]),
    "dfm_transform": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p, C.c_void_p]),
    "dfm_train_step": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfm_train_step_host": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.POINTER(C.c_float), C.c_void_p]),
    "dfm_train_step_host_async": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.POINTER(C.c_float)]),
    "dfm_train_step_host_drain": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "dfm_prefetch_batch": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p]),
    "dfm_forward": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p, C.c_void_p]),
    "dfm_forward_host": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p]),
    "dfm_metrics_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dfm_metrics_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "dfm_evaluate": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p]),
    "dfm_evaluate_host": (C.c_int, [C.c_void_p, C.POINTER(RawBatch)]),
    "dfm_metrics_read": (C.c_int, [C.c_void_p, C.POINTER(MetricState), C.c_void_p]),
    "dfm_summary_bucket_limits": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "dfm_layer_summary": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]),
    "dfm_layer_summary_tensor": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p]),
    "dfm_flush": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dfm_sync": (C.c_int, [C.c_void_p]),
    "dfm_global_step": (C.c_int64, [C.c_void_p]),
    "dfm_state_checksum": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "dfm_last_unique_rows": (C.c_int64, [C.c_void_p]),
    "dfm_set_global_step": (C.c_int, [C.c_void_p, C.c_int64]),
    "dfm_last_step_launches": (C.c_int64, [C.c_void_p]),
    "dfm_graph_steps": (C.c_int64, [C.c_void_p]),
    "dfm_set_profiling": (C.c_int, [C.c_void_p, C.c_int32]),
    "dfm_phase_ms": (C.c_float, [C.c_void_p, C.c_char_p]),
    "dfm_shard_row_width": (C.c_int, [C.c_void_p]),
    "dfm_num_slots": (C.c_int, [C.c_void_p]),
    "dfm_dense_size": (C.c_int64, [C.c_void_p]),
    "dfm_shard_requests": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "dfm_shard_serve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "dfm_shard_forward_backward": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfm_shard_apply": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfm_shard_forward": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfm_xchg_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dfm_xchg_import": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dfm_xchg_buffer": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "dfm_xchg_set_peers": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "dfm_xchg_begin": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p]),
    "dfm_xchg_serve": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dfm_xchg_forward_backward": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_int64, C.c_void_p, C.c_void_p]),
    "dfm_xchg_apply": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfm_xchg_train_step": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfm_xchg_train_step_next": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.POINTER(RawBatch), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfm_xchg_forward": (C.c_int, [C.c_void_p, C.POINTER(RawBatch), C.c_void_p, C.c_void_p]),
    "dfm_csv_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "dfm_csv_destroy": (None, [C.c_void_p]),
    "dfm_csv_last_error": (C.c_char_p, [C.c_void_p]),
    "dfm_csv_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.c_void_p]),
    "dfm_csv_decode_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.c_void_p]),
    "dfm_csv_load": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "dfm_csv_decode_lines": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "dfm_csv_num_records": (C.c_int32, [C.c_void_p]),
    "dfm_csv_int_column": (C.c_void_p, [C.c_void_p, C.c_int32]),
    "dfm_csv_str_bytes": (C.c_void_p, [C.c_void_p, C.c_int32]),
    "dfm_csv_str_offsets": (C.c_void_p, [C.c_void_p, C.c_int32]),
    "dfm_csv_float_column": (C.c_void_p, [C.c_void_p, C.c_int32]),
    "dfm_csv_labels": (C.c_void_p, [C.c_void_p]),
    "dfm_test_sort_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]),
    "dfm_test_sort_pairs_algo": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32]),
    "dfm_test_fingerprint64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "dfm_test_replay": (C.c_int, [C.POINTER(Optimizer), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32]),
    "dfm_test_tc_gemm": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "dfm_version": (C.c_char_p, []),
}
EXPORTS = sorted(_SIGS)

_lib = None


def load():
    """Load the CUDA library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libdeepfm_b200.so is missing (%s): build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or recommender_tensorflow_b200/csrc/build.sh. There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class DfmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("deepfm_b200 error %s (%d): %s" % (ERRORS.get(code, "?"), code, msg))
        self.code = code
