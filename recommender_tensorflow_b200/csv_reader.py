"""GPU CSV input path (SURVEY.md §8f rank 2): whole records in, device-resident raw batch out.

`GpuCsvReader` binds `dfm_csv_*` (include/deepfm_b200.h): the equivalent of the reference's
`tf.data.TextLineDataset(csv)` + `tf.decode_csv(value, DEFAULTS)` + `rating >= cutoff`
(trainers/ml_100k.py:44-58) with the field work done by CUDA kernels.  `decode()` returns a
`PackedBatch` whose column pointers alias the reader's device buffers (valid until the next decode),
ready for `DeepFMEngine.train_step_device / transform / predict_logits`.
"""
import ctypes as C

import numpy as np

from . import _lib
from .engine import DfmError, PackedBatch

CSV_SKIP, CSV_INT32, CSV_STRING, CSV_FLOAT32 = 0, 1, 2, 3


class CsvConfig(C.Structure):
    _fields_ = [("n_fields", C.c_int32), ("kind", C.POINTER(C.c_int32)), ("int_default", C.POINTER(C.c_int32)),
                ("str_default", C.POINTER(C.c_char_p)), ("label_field", C.c_int32), ("label_min", C.c_int32),
                ("max_records", C.c_int32), ("max_bytes", C.c_int64), ("device", C.c_int32),
                ("float_default", C.POINTER(C.c_float)), ("field_delim", C.c_int32), ("as_float", C.POINTER(C.c_int32))]


def _default_dtype(d):
    """record_defaults entry -> the dtype tf.decode_csv gives the field"""
    if isinstance(d, (int, np.integer)):
        return "int32"
    return "float32" if isinstance(d, (float, np.floating)) else "string"


class GpuCsvReader:
    def __init__(self, engine, columns, defaults, label_col=None, cutoff=5, max_records=65536, max_bytes=None, field_delim=","):
        """columns / defaults: the CSV schema (names and `record_defaults`, e.g. trainers.ml_100k.COLUMNS / DEFAULTS;
        [0] is int32, [0.0] float32, anything else a string).  Only the fields `engine` consumes (plus the label) are
        materialised; the rest is parsed for structure only.  A numeric column reads a float32 field, or an int32 field
        converted with tf.to_float.  field_delim: one character, as tf.decode_csv's."""
        self.lib = _lib.load()
        self.eng = engine
        self.columns = list(columns)
        wanted = {}
        for s in engine.raw_specs:          # model columns and the source columns of crossed ones
            if s["kind"] == "crossed":
                continue
            if s["width"] != 1:
                raise ValueError("GpuCsvReader: multivalent column %r has no CSV encoding in the reference" % s["source"])
            wanted[s["source"]] = s["dtype"]
        numeric = {c.key for c in engine.num_columns}
        delim = field_delim.encode() if isinstance(field_delim, str) else bytes(field_delim)
        if len(delim) != 1:
            raise ValueError("field_delim must be one byte, got %r" % (field_delim,))
        n = len(self.columns)
        kind = (C.c_int32 * n)()
        idef = (C.c_int32 * n)()
        sdef = (C.c_char_p * n)()
        fdef = (C.c_float * n)()
        as_float = (C.c_int32 * n)()
        for j, (name, d) in enumerate(zip(self.columns, defaults)):
            dt = _default_dtype(d[0])
            if name in wanted and wanted[name] != dt:
                raise ValueError("column %r: model expects %s, CSV default %r says otherwise" % (name, wanted[name], d))
            if name in numeric and dt == "string":
                raise ValueError("column %r: numeric column expects float32 or int32, CSV default %r says otherwise" % (name, d))
            if name in wanted or name in numeric or name == label_col:
                kind[j] = {"int32": CSV_INT32, "float32": CSV_FLOAT32, "string": CSV_STRING}[dt]
            else:
                kind[j] = CSV_SKIP
            as_float[j] = int(name in numeric and dt == "int32")
            if dt == "int32":
                idef[j] = int(d[0])
            elif dt == "float32":
                fdef[j] = float(d[0])
            else:
                sdef[j] = str(d[0]).encode()
        missing = [k for k in list(wanted) + sorted(numeric) if k not in self.columns]
        if missing:
            raise ValueError("model columns missing from the CSV schema: %r" % missing)
        self.label_field = self.columns.index(label_col) if label_col is not None else -1
        self.max_records = int(max_records)
        self.max_bytes = int(max_bytes or 512 * self.max_records)
        cfg = CsvConfig(n, C.cast(kind, C.POINTER(C.c_int32)), C.cast(idef, C.POINTER(C.c_int32)), C.cast(sdef, C.POINTER(C.c_char_p)),
                        self.label_field, int(cutoff), self.max_records, self.max_bytes, engine.device,
                        C.cast(fdef, C.POINTER(C.c_float)), delim[0], C.cast(as_float, C.POINTER(C.c_int32)))
        self._keep = [kind, idef, sdef, fdef, as_float]
        h = C.c_void_p()
        rc = self.lib.dfm_csv_create(C.byref(cfg), C.byref(h))
        if rc != _lib.DFM_OK:
            raise DfmError(rc, (self.lib.dfm_csv_last_error(None) or b"").decode())
        self.h = h
        self._field = {name: j for j, name in enumerate(self.columns)}

    def close(self):
        if getattr(self, "h", None):
            self.lib.dfm_csv_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != _lib.DFM_OK:
            msg = (self.lib.dfm_csv_last_error(self.h) or b"").decode()
            if rc == -7:
                raise ValueError(msg)       # tf.decode_csv raises InvalidArgumentError; input errors are ValueErrors here
            raise DfmError(rc, msg)

    def decode(self, text, stream=None):
        """text: bytes / bytearray / numpy uint8 array / pinned torch uint8 tensor holding whole records (host), or a
        cuda uint8 tensor (16-byte aligned, padded to a multiple of 16).  -> PackedBatch on the device."""
        n_rec = C.c_int32(0)
        st = C.c_void_p(stream) if stream else None
        if not stream:
            self.eng.sync()      # the previous batch aliases the buffers this decode overwrites; a step may still be reading them
        if hasattr(text, "is_cuda") and text.is_cuda:
            self._check(self.lib.dfm_csv_decode(self.h, C.c_void_p(text.data_ptr()), int(text.numel()), C.byref(n_rec), st))
        elif hasattr(text, "data_ptr"):
            self._check(self.lib.dfm_csv_decode_host(self.h, C.c_void_p(text.data_ptr()), int(text.numel()), C.byref(n_rec), st))
        else:
            buf = text if isinstance(text, np.ndarray) else np.frombuffer(bytes(text), dtype=np.uint8)
            self._check(self.lib.dfm_csv_decode_host(self.h, C.c_void_p(buf.ctypes.data), int(buf.size), C.byref(n_rec), st))
        return self._batch(n_rec.value)

    def load_file(self, source):
        """File-resident mode: upload the whole CSV (path or bytes) once; -> number of lines (line 0 = header, if any)."""
        data = np.fromfile(source, dtype=np.uint8) if isinstance(source, str) else np.frombuffer(bytes(source), dtype=np.uint8)
        n = C.c_int64(0)
        self._check(self.lib.dfm_csv_load(self.h, C.c_void_p(data.ctypes.data), int(data.size), C.byref(n)))
        return int(n.value)

    def decode_lines(self, line_idx, stream=None):
        """Decode the given lines of the loaded file (record i of the batch = line line_idx[i]) -> PackedBatch."""
        idx = np.ascontiguousarray(line_idx, dtype=np.int32)
        if not stream:
            self.eng.sync()
        self._check(self.lib.dfm_csv_decode_lines(self.h, C.c_void_p(idx.ctypes.data), int(idx.size), C.c_void_p(stream) if stream else None))
        return self._batch(int(idx.size))

    def _batch(self, n):
        eng = self.eng
        nc = max(len(eng.raw_specs), 1)
        cat = (C.c_void_p * nc)()
        off = (C.c_void_p * nc)()
        num = (C.c_void_p * max(len(eng.num_columns), 1))()
        for i, s in enumerate(eng.raw_specs):
            if s["kind"] == "crossed":
                continue
            f = self._field[s["source"]]
            if s["dtype"] == "string":
                cat[i] = self.lib.dfm_csv_str_bytes(self.h, f)
                off[i] = self.lib.dfm_csv_str_offsets(self.h, f)
            elif s["dtype"] == "float32":      # bucketized column over a float32 field
                cat[i] = self.lib.dfm_csv_float_column(self.h, f)
            else:
                cat[i] = self.lib.dfm_csv_int_column(self.h, f)
        for j, c in enumerate(eng.num_columns):
            num[j] = self.lib.dfm_csv_float_column(self.h, self._field[c.key])
        lab = self.lib.dfm_csv_labels(self.h) if self.label_field >= 0 else None
        raw = _lib.RawBatch(n, C.cast(cat, C.POINTER(C.c_void_p)), C.cast(off, C.POINTER(C.c_void_p)),
                            C.cast(num, C.POINTER(C.c_void_p)), lab)
        return PackedBatch(None, 0, raw, [cat, off, num, self], 0, n, True)

    # ---- read-back helpers (tests, debugging) ----
    @staticmethod
    def _d2h(ptr, nbytes):
        import torch
        if not nbytes:
            return np.empty(0, dtype=np.uint8)

        class _View:      # device memory owned by the reader, exposed through the CUDA array interface
            __cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}
        torch.cuda.synchronize()
        return torch.as_tensor(_View(), device="cuda").cpu().numpy()

    def column(self, name):
        """Decoded column as numpy: int32 [n], float32 [n] or an object array of bytes (strings).  An int32 field that
        a numeric column reads as float32 comes back as int32; float_column() gives its float32 copy."""
        f = self._field[name]
        n = int(self.lib.dfm_csv_num_records(self.h))
        p = self.lib.dfm_csv_int_column(self.h, f)
        if p:
            return self._d2h(p, 4 * n).view(np.int32).copy()
        if self.lib.dfm_csv_float_column(self.h, f):
            return self.float_column(name)
        offs = self._d2h(self.lib.dfm_csv_str_offsets(self.h, f), 4 * (n + 1)).view(np.int32).copy()
        data = self._d2h(self.lib.dfm_csv_str_bytes(self.h, f), int(offs[-1])).tobytes()
        return np.array([data[offs[i]:offs[i + 1]] for i in range(n)], dtype=object)

    def float_column(self, name):
        """float32 [n] of a float32 field, or of an int32 field that a numeric column reads"""
        p = self.lib.dfm_csv_float_column(self.h, self._field[name])
        if not p:
            raise ValueError("column %r has no float32 copy: it is neither a float32 field nor an int32 field a numeric column reads" % name)
        n = int(self.lib.dfm_csv_num_records(self.h))
        return self._d2h(p, 4 * n).view(np.float32).copy()

    def labels(self):
        n = int(self.lib.dfm_csv_num_records(self.h))
        return self._d2h(self.lib.dfm_csv_labels(self.h), 4 * n).view(np.float32).copy()
