"""Mirror of the reference's trainers/deep_fm.py on top of the CUDA engine.

`model_fn(features, labels, mode, params)` keeps the reference's signature, param names, defaults
and error behaviour (trainers/deep_fm.py:11-34).  TensorFlow builds a graph once and then runs
`train_op`; here there is no graph: the first call builds the engine (cached in `params`), and
every TRAIN call executes one `session.run(train_op)` equivalent on the given batch.
"""
import glob
import os
import shutil
from argparse import ArgumentParser
from collections import namedtuple

import numpy as np

from ..engine import DeepFMEngine, PackedBatch
from .ml_100k import FEATURE_DTYPES, ModeKeys, get_feature_columns, get_input_fn
from .model_utils import (check_regression_head, get_binary_metrics, get_binary_predictions, get_optimizer,
                          get_regression_metrics, get_regression_predictions, get_weights, weight_column_key, finish_metrics)

EstimatorSpec = namedtuple("EstimatorSpec", ["mode", "loss", "train_op", "predictions", "eval_metric_ops", "global_step"])
_ENGINE_KEY = "_b200_engine"
# params["head"] -> (engine head, predictions, EVAL metrics): the reference's contrib binary_classification_head, or
# regression_head (label_dimension 1, mean squared error, identity inverse link) to predict the rating itself
_HEADS = {"binary": ("logistic", get_binary_predictions, get_binary_metrics),
          "regression": ("squared", get_regression_predictions, get_regression_metrics)}


def _head(params):
    head = params.get("head", "binary")
    if head not in _HEADS:
        raise ValueError("params['head'] must be one of %s, got %r" % (sorted(_HEADS), head))
    if head == "regression":
        check_regression_head(params.get("label_dimension", 1), params.get("inverse_link_fn"), params.get("loss_fn"))
    return _HEADS[head]


def _build_engine(params, batch_size):
    categorical_columns = params.get("categorical_columns", [])
    numeric_columns = params.get("numeric_columns", [])
    use_linear = params.get("use_linear", True)
    use_mf = params.get("use_mf", True)
    use_dnn = params.get("use_dnn", True)
    embedding_size = params.get("embedding_size", 4)
    hidden_units = params.get("hidden_units", [16, 16])
    activation_fn = params.get("activation", "relu")
    dropout = params.get("dropout", 0)
    optimizer = params.get("optimizer", "Adam")
    learning_rate = params.get("learning_rate", 0.001)
    # weight_column of the binary head (contrib binary_classification_head(weight_column=...)): absent in the
    # reference's model_fn, so None keeps the unweighted model
    weighted = weight_column_key(params.get("weight_column")) is not None
    head = _head(params)[0]
    # check params (trainers/deep_fm.py:28-34)
    if (len(categorical_columns) + len(numeric_columns)) == 0:
        raise ValueError("At least 1 feature column of categorical_columns or numeric_columns must be specified.")
    if not (use_linear or use_mf or use_dnn):
        raise ValueError("At least 1 of linear, mf or dnn component must be used.")
    # params["activation"]: a tf.nn callable in the reference (default tf.nn.relu); here its name, a callable named
    # relu / tanh / sigmoid / identity, or None (tf.layers.dense without activation)
    opt = get_optimizer(optimizer, learning_rate)
    eng = DeepFMEngine(categorical_columns, numeric_columns, embedding_size=embedding_size, hidden_units=hidden_units,
                       use_linear=bool(use_linear), use_mf=bool(use_mf), use_dnn=bool(use_dnn), loss_reduction="mean",
                       opt_deep=opt, opt_linear=dict(opt), max_batch=params.get("max_batch", max(batch_size, 1)),
                       device=params.get("device", 0), feature_dtypes=params.get("feature_dtypes", FEATURE_DTYPES),
                       dropout=float(dropout or 0.0), dropout_seed=int(params.get("dropout_seed", 0)), activation=activation_fn,
                       weighted=weighted, head=head)
    # the variable initialisers TF runs when the graph is first executed (truncated normal 1/sqrt(k) for the embedding
    # tables, glorot uniform for the dense kernels, zeros for linear weights and biases); RunConfig.tf_random_seed
    seed = params.get("tf_random_seed")
    eng.init_random(int(seed) if seed is not None else int.from_bytes(os.urandom(4), "little"))
    return eng


def _batch_size(features):
    if hasattr(features, "batch_size"):      # a PackedBatch (e.g. decoded on the GPU by get_gpu_input_fn)
        return int(features.batch_size)
    v = next(iter(features.values()))
    return (len(v[1]) - 1) if isinstance(v, tuple) else len(v)


def model_fn(features, labels, mode, params):
    """trainers/deep_fm.py:11-125.  TRAIN: one train step; EVAL: loss + head metrics; PREDICT: predictions."""
    engine = params.get(_ENGINE_KEY)
    if engine is None:
        engine = params[_ENGINE_KEY] = _build_engine(params, _batch_size(features))
    weight_column = params.get("weight_column")
    _, predictions, eval_metrics = _head(params)
    if mode == ModeKeys.TRAIN:
        # a device batch (get_gpu_input_fn) carries its weights inside; a host batch has them among its features
        weights = None if isinstance(features, PackedBatch) else get_weights(features, weight_column, _batch_size(features))
        loss, logits = engine.train_step(features, labels, return_logits=True, weights=weights)
        return EstimatorSpec(mode, loss, None, predictions(logits), None, engine.global_step)
    logits = engine.predict_logits(features)
    preds = predictions(logits)
    if mode == ModeKeys.PREDICT:
        return EstimatorSpec(mode, None, None, preds, None, engine.global_step)
    metrics = eval_metrics(labels, logits, get_weights(features, weight_column, logits.shape[0]))
    return EstimatorSpec(mode, metrics["average_loss"], None, preds, metrics, engine.global_step)


class Estimator:
    """Minimal stand-in for tf.estimator.Estimator(model_fn, model_dir, config, params): train /
    evaluate / predict loops around model_fn, checkpoints as .npz (variables + optimizer slots)."""

    KEEP_CHECKPOINT_MAX = 5      # trainers/conf_utils.py:6-10
    SAVE_CHECKPOINTS_SECS = 60   # trainers/conf_utils.py:6-10 (RunConfig(save_checkpoints_secs=60))
    SAVE_SUMMARY_STEPS = 100     # RunConfig default: layer_summary side outputs every 100 steps

    def __init__(self, model_fn, model_dir=None, config=None, params=None):
        self.model_fn, self.model_dir, self.config, self.params = model_fn, model_dir, config, dict(params or {})
        self._restored = False

    # -- checkpoints: tf.train.Saver equivalents (variables + slots under TF-1.12 names, .npz container)
    def latest_checkpoint(self):
        if not self.model_dir:
            return None
        found = glob.glob(os.path.join(self.model_dir, "model.ckpt-*.npz"))
        return max(found, key=lambda p: int(p.rsplit("-", 1)[1].split(".")[0])) if found else None

    def save_checkpoint(self):
        if not self.model_dir or self.engine is None:
            return None
        os.makedirs(self.model_dir, exist_ok=True)
        path = os.path.join(self.model_dir, "model.ckpt-%d.npz" % self.engine.global_step)
        self.engine.save_checkpoint(path)
        old = sorted(glob.glob(os.path.join(self.model_dir, "model.ckpt-*.npz")),
                     key=lambda p: int(p.rsplit("-", 1)[1].split(".")[0]))
        for p in old[:-self.KEEP_CHECKPOINT_MAX]:
            os.remove(p)
        return path

    def _maybe_restore(self):
        """Estimator semantics: a model_dir that already holds a checkpoint is resumed (the trainer wipes it
        first unless --restore is given, trainers/deep_fm.py:147-148)."""
        if not self._restored and self.engine is not None:
            self._restored = True
            ck = self.latest_checkpoint()
            if ck:
                self.engine.load_checkpoint(ck)

    @property
    def engine(self):
        return self.params.get(_ENGINE_KEY)

    def build(self, max_batch):
        """Create the model before the first batch arrives (the GPU input path needs the engine to bind its reader)."""
        if self.engine is None:
            self.params[_ENGINE_KEY] = _build_engine(self.params, max_batch)
        self._maybe_restore()
        return self.engine

    def write_summaries(self, feats):
        """trainers/model_utils.py:4-6: zero fraction + histogram of every summarised tensor -> model_dir/summaries.jsonl"""
        if not self.model_dir or not self.SAVE_SUMMARY_STEPS:
            return
        import json
        os.makedirs(self.model_dir, exist_ok=True)
        rec = {"step": self.engine.global_step + 1, "summaries": self.engine.layer_summary(feats, train=True)}
        with open(os.path.join(self.model_dir, "summaries.jsonl"), "a") as f:
            f.write(json.dumps(rec) + "\n")

    def train(self, input_fn, steps=None, max_steps=None, log_every=100):
        import time
        loss = None
        last_save = time.time()
        for feats, labels in input_fn():
            if self.engine is None:
                self.params[_ENGINE_KEY] = _build_engine(self.params, _batch_size(feats))
            self._maybe_restore()
            eng = self.engine
            if max_steps is not None and eng.global_step >= max_steps:
                break
            if self.SAVE_SUMMARY_STEPS and eng.global_step % self.SAVE_SUMMARY_STEPS == 0:
                self.write_summaries(feats)
            spec = self.model_fn(feats, labels, ModeKeys.TRAIN, self.params)
            loss = spec.loss
            if self.SAVE_CHECKPOINTS_SECS and time.time() - last_save >= self.SAVE_CHECKPOINTS_SECS:
                self.save_checkpoint()
                last_save = time.time()
            if log_every and spec.global_step % log_every == 0:
                print("INFO:b200:loss = %.6f, step = %d" % (loss, spec.global_step))
            if steps is not None:
                steps -= 1
                if steps <= 0:
                    break
        self.save_checkpoint()
        return loss

    def evaluate(self, input_fn):
        ys, zs, ws = [], [], []
        weight_column = self.params.get("weight_column")
        _, _, eval_metrics = _head(self.params)
        zkey = "predictions" if eval_metrics is get_regression_metrics else "logits"    # the head's logits, [B, 1]
        for feats, labels in input_fn():
            if self.engine is None:
                self.params[_ENGINE_KEY] = _build_engine(self.params, _batch_size(feats))
            self._maybe_restore()
            spec = self.model_fn(feats, labels, ModeKeys.EVAL, self.params)
            ys.append(np.asarray(labels, dtype=np.float32).reshape(-1))
            zs.append(spec.predictions[zkey].reshape(-1))
            if weight_column is not None:
                ws.append(get_weights(feats, weight_column, zs[-1].shape[0]))
        if not ys:
            raise ValueError("evaluate(): input_fn yielded no batches")
        m = eval_metrics(np.concatenate(ys), np.concatenate(zs), np.concatenate(ws) if ws else None)
        m["global_step"] = self.engine.global_step
        return m

    def evaluate_streaming(self, input_fn, steps=None):
        """evaluate() with the metrics streamed on the device (DESIGN.md §8.6): every batch's forward pass and metric
        accumulation run on the GPU, nothing per example is copied back or kept on the host.  Same metric names plus
        global_step; the AUCs use TF's float32 predictions and thresholds, so they can differ from evaluate()'s float64
        ones for predictions at a threshold.  steps: stop after that many batches.  With get_gpu_input_fn(...,
        device_labels=True) the labels and weights stay on the device."""
        weight_column = self.params.get("weight_column")
        _head(self.params)
        n = 0
        for feats, labels in input_fn():
            if steps is not None and n >= steps:
                break
            if self.engine is None:
                self.params[_ENGINE_KEY] = _build_engine(self.params, _batch_size(feats))
            self._maybe_restore()
            if n == 0:
                self.engine.metrics_reset()
            weights = None if isinstance(feats, PackedBatch) else get_weights(feats, weight_column, _batch_size(feats))
            self.engine.evaluate_batch(feats, labels, weights)
            n += 1
        if not n:
            raise ValueError("evaluate_streaming(): input_fn yielded no batches")
        m = finish_metrics(self.engine.metrics_state())
        m["global_step"] = self.engine.global_step
        return m

    def predict(self, input_fn):
        for item in input_fn():
            feats = item[0] if isinstance(item, tuple) and len(item) == 2 and isinstance(item[0], dict) else item
            if self.engine is None:
                self.params[_ENGINE_KEY] = _build_engine(self.params, _batch_size(feats))
            if not self._restored:
                # tf.estimator.Estimator.predict restores the latest checkpoint and fails when there is none
                if self.engine.global_step == 0 and self.latest_checkpoint() is None:
                    raise ValueError("Could not find trained model in model_dir: %s." % self.model_dir)
                self._maybe_restore()
            spec = self.model_fn(feats, None, ModeKeys.PREDICT, self.params)
            n = next(iter(spec.predictions.values())).shape[0]
            for i in range(n):
                yield {k: v[i] for k, v in spec.predictions.items()}


def train_and_evaluate(args):
    """trainers/deep_fm.py:128-178 (local run: train to max_steps, then one evaluation)."""
    if not args.restore:
        shutil.rmtree(args.job_dir, ignore_errors=True)
    feature_columns = get_feature_columns(embedding_size=args.embedding_size)
    estimator = Estimator(model_fn=model_fn, model_dir=args.job_dir, params={
        "categorical_columns": feature_columns["linear"],
        "use_linear": not args.exclude_linear, "use_mf": not args.exclude_mf, "use_dnn": not args.exclude_dnn,
        "embedding_size": args.embedding_size, "hidden_units": args.hidden_units, "dropout": args.dropout,
        "max_batch": args.batch_size, "tf_random_seed": getattr(args, "seed", None)})
    if getattr(args, "gpu_input", False):     # tf.decode_csv on the device (csv_reader.GpuCsvReader); same record stream
        from .ml_100k import get_gpu_input_fn
        eng = estimator.build(args.batch_size)
        train_fn = get_gpu_input_fn(args.train_csv, eng, batch_size=args.batch_size, seed=getattr(args, "seed", None))
        eval_fn = get_gpu_input_fn(args.test_csv, eng, ModeKeys.EVAL, batch_size=args.batch_size)
    else:
        train_fn = get_input_fn(args.train_csv, batch_size=args.batch_size, seed=getattr(args, "seed", None))
        eval_fn = get_input_fn(args.test_csv, ModeKeys.EVAL, batch_size=args.batch_size)
    estimator.train(train_fn, max_steps=args.train_steps)
    metrics = estimator.evaluate(eval_fn)
    print("INFO:b200:eval " + ", ".join("%s = %s" % kv for kv in sorted(metrics.items())))
    return metrics


if __name__ == "__main__":
    parser = ArgumentParser()
    parser.add_argument("--train-csv", default="data/ml-100k/train.csv")
    parser.add_argument("--test-csv", default="data/ml-100k/test.csv")
    parser.add_argument("--seed", type=int, default=None, help="tf_random_seed: variable initialisers and the shuffle")
    parser.add_argument("--gpu-input", action="store_true", help="decode the CSV records on the GPU instead of in Python")
    parser.add_argument("--job-dir", default="checkpoints/deep_fm")
    parser.add_argument("--restore", action="store_true")
    parser.add_argument("--exclude-linear", action="store_true")
    parser.add_argument("--exclude-mf", action="store_true")
    parser.add_argument("--exclude-dnn", action="store_true")
    parser.add_argument("--embedding-size", type=int, default=4)
    parser.add_argument("--hidden-units", type=int, nargs="+", default=[16, 16])
    parser.add_argument("--dropout", type=float, default=0.1, help="dropout rate (default: %(default)s)")
    parser.add_argument("--batch-size", type=int, default=32)
    parser.add_argument("--train-steps", type=int, default=20000)
    train_and_evaluate(parser.parse_args())
