"""Mirror of trainers/linear_deep.py: the canned tf.estimator.DNNLinearCombinedClassifier
(trainers/linear_deep.py:32-39) = wide&deep: linear_model(linear columns) + DNN(input_layer(deep
columns)), no FM term, SUM loss, Adagrad(0.001) on the dnn side and FTRL(min(0.005, 1/sqrt(n_linear)))
on the linear side (TF-1.12 canned defaults, SURVEY.md §8a row 8).  DNNLinearCombinedRegressor is the same model
with the regression head (squared error on the float label, the logits as predictions)."""
import math
import os

import numpy as np

from ..engine import DeepFMEngine, PackedBatch, default_optimizer
from .ml_100k import FEATURE_DTYPES, ModeKeys
from .model_utils import (check_regression_head, finish_metrics, get_binary_metrics, get_binary_predictions, get_regression_metrics,
                          get_regression_predictions, get_weights, weight_column_key)

_DNN_LEARNING_RATE = 0.001
_LINEAR_LEARNING_RATE = 0.005


class _CannedBase:
    """train / evaluate / predict loops shared by the canned-estimator mirrors, with the Estimator's checkpoint
    behaviour (resume from model_dir, save at the end of train(), keep_checkpoint_max = 5)."""
    engine = None
    model_dir = None
    weight_column = None       # weight_column: a feature key or numeric_column whose value weights each example
    KEEP_CHECKPOINT_MAX = 5
    _restored = False
    # the head: *Classifier binary (sigmoid cross-entropy), *Regressor regression (squared error, label_dimension 1)
    HEAD = "binary"
    _ENGINE_HEAD = {"binary": "logistic", "regression": "squared"}

    def _head_fns(self):
        """(predictions, EVAL metrics) of the head"""
        if self.HEAD == "regression":
            return get_regression_predictions, get_regression_metrics
        return get_binary_predictions, get_binary_metrics

    def _weights(self, feats, n=None):
        """per-example weights of a host batch (None when unweighted; a device batch carries its own)"""
        if self.weight_column is None or (n is None and isinstance(feats, PackedBatch)):
            return None
        from .deep_fm import _batch_size
        return get_weights(feats, self.weight_column, _batch_size(feats) if n is None else n)

    def _finish_init(self, model_dir, tf_random_seed):
        """Variable initialisers (TF runs them on the first session.run; RunConfig.tf_random_seed): embeddings truncated
        normal, kernels glorot uniform - without this the tower starts at zero and, with ReLU, stays dead."""
        self.engine.init_random(int(tf_random_seed) if tf_random_seed is not None else int.from_bytes(os.urandom(4), "little"))
        self.model_dir = model_dir

    def latest_checkpoint(self):
        import glob
        found = glob.glob(os.path.join(self.model_dir, "model.ckpt-*.npz")) if self.model_dir else []
        return max(found, key=lambda p: int(p.rsplit("-", 1)[1].split(".")[0])) if found else None

    def save_checkpoint(self):
        import glob
        if not self.model_dir:
            return None
        os.makedirs(self.model_dir, exist_ok=True)
        path = os.path.join(self.model_dir, "model.ckpt-%d.npz" % self.engine.global_step)
        self.engine.save_checkpoint(path, scheme="canned")
        old = sorted(glob.glob(os.path.join(self.model_dir, "model.ckpt-*.npz")), key=lambda p: int(p.rsplit("-", 1)[1].split(".")[0]))
        for p in old[:-self.KEEP_CHECKPOINT_MAX]:
            os.remove(p)
        return path

    def _maybe_restore(self):
        if not self._restored:
            self._restored = True
            ck = self.latest_checkpoint()
            if ck:
                self.engine.load_checkpoint(ck, scheme="canned")

    def train(self, input_fn, steps=None, max_steps=None):
        loss = None
        self._maybe_restore()
        for feats, labels in input_fn():
            if max_steps is not None and self.engine.global_step >= max_steps:
                break
            loss = self.engine.train_step(feats, labels, weights=self._weights(feats))
            if steps is not None:
                steps -= 1
                if steps <= 0:
                    break
        self.save_checkpoint()
        return loss

    def evaluate(self, input_fn):
        ys, zs, ws = [], [], []
        self._maybe_restore()
        for feats, labels in input_fn():
            ys.append(np.asarray(labels, dtype=np.float32).reshape(-1))
            zs.append(self.engine.predict_logits(feats))
            if self.weight_column is not None:
                ws.append(self._weights(feats, zs[-1].shape[0]))
        m = self._head_fns()[1](np.concatenate(ys), np.concatenate(zs), np.concatenate(ws) if ws else None)
        m["global_step"] = self.engine.global_step
        return m

    def evaluate_streaming(self, input_fn, steps=None):
        """evaluate() with the metrics streamed on the device (DESIGN.md §8.6): same metric names plus global_step; the
        AUCs use TF's float32 predictions and thresholds.  steps: stop after that many batches."""
        self._maybe_restore()
        self.engine.metrics_reset()
        n = 0
        for feats, labels in input_fn():
            if steps is not None and n >= steps:
                break
            self.engine.evaluate_batch(feats, labels, self._weights(feats))
            n += 1
        if not n:
            raise ValueError("evaluate_streaming(): input_fn yielded no batches")
        m = finish_metrics(self.engine.metrics_state())
        m["global_step"] = self.engine.global_step
        return m

    def predict(self, input_fn):
        self._maybe_restore()
        for item in input_fn():
            feats = item[0] if isinstance(item, tuple) else item
            preds = self._head_fns()[0](self.engine.predict_logits(feats))
            for i in range(next(iter(preds.values())).shape[0]):
                yield {k: v[i] for k, v in preds.items()}


class DNNLinearCombinedClassifier(_CannedBase):
    def __init__(self, model_dir=None, linear_feature_columns=None, dnn_feature_columns=None, dnn_hidden_units=None,
                 dnn_dropout=None, config=None, max_batch=4096, device=0, feature_dtypes=FEATURE_DTYPES, tf_random_seed=None,
                 weight_column=None):
        weight_column_key(weight_column)        # type check, as TF's constructor does
        self.weight_column = weight_column
        linear_feature_columns = list(linear_feature_columns or [])
        dnn_feature_columns = list(dnn_feature_columns or [])
        if not linear_feature_columns and not dnn_feature_columns:
            raise ValueError("Either linear_feature_columns or dnn_feature_columns must be defined.")
        cats = [c.categorical_column for c in dnn_feature_columns] or linear_feature_columns
        if linear_feature_columns and dnn_feature_columns and [c.name for c in cats] != [c.name for c in linear_feature_columns]:
            raise NotImplementedError("linear and dnn sides must be built on the same categorical columns "
                                      "(as in trainers/ml_100k.py:37-38)")
        dims = {c.dimension for c in dnn_feature_columns}
        if len(dims) > 1:
            raise NotImplementedError("all embedding columns must share one dimension")
        lin_lr = min(_LINEAR_LEARNING_RATE, 1.0 / math.sqrt(max(len(linear_feature_columns), 1)))
        self.engine = DeepFMEngine(cats, (), embedding_size=(dims.pop() if dims else 4),
                                   hidden_units=list(dnn_hidden_units or []), use_linear=bool(linear_feature_columns),
                                   use_mf=False, use_dnn=bool(dnn_feature_columns), loss_reduction="sum",
                                   opt_deep=default_optimizer("Adagrad", _DNN_LEARNING_RATE),
                                   opt_linear=default_optimizer("Ftrl", lin_lr), max_batch=max_batch, device=device,
                                   dropout=float(dnn_dropout or 0.0),
                                   feature_dtypes=feature_dtypes, weighted=weight_column is not None,
                                   head=self._ENGINE_HEAD[self.HEAD])
        self._finish_init(model_dir, tf_random_seed)


class DNNLinearCombinedRegressor(DNNLinearCombinedClassifier):
    """canned tf.estimator.DNNLinearCombinedRegressor (TF 1.12): DNNLinearCombinedClassifier's model, optimizers,
    checkpoint names and SUM reduction with the regression head"""
    HEAD = "regression"

    def __init__(self, model_dir=None, linear_feature_columns=None, dnn_feature_columns=None, dnn_hidden_units=None,
                 dnn_dropout=None, label_dimension=1, weight_column=None, config=None, max_batch=4096, device=0,
                 feature_dtypes=FEATURE_DTYPES, tf_random_seed=None):
        check_regression_head(label_dimension)
        super().__init__(model_dir=model_dir, linear_feature_columns=linear_feature_columns, dnn_feature_columns=dnn_feature_columns,
                         dnn_hidden_units=dnn_hidden_units, dnn_dropout=dnn_dropout, config=config, max_batch=max_batch,
                         device=device, feature_dtypes=feature_dtypes, tf_random_seed=tf_random_seed, weight_column=weight_column)


def canned_train_and_evaluate(args, build):
    """trainers/linear.py:10-44 / deep.py / linear_deep.py `train_and_evaluate` (local run: train to train_steps, evaluate)."""
    import shutil
    from .ml_100k import get_feature_columns, get_input_fn
    if not args.restore:
        shutil.rmtree(args.job_dir, ignore_errors=True)
    estimator = build(get_feature_columns(embedding_size=args.embedding_size), args)
    estimator.train(get_input_fn(args.train_csv, batch_size=args.batch_size, seed=getattr(args, "seed", None)), max_steps=args.train_steps)
    metrics = estimator.evaluate(get_input_fn(args.test_csv, ModeKeys.EVAL, batch_size=args.batch_size))
    print("INFO:b200:eval " + ", ".join("%s = %s" % kv for kv in sorted(metrics.items())))
    return metrics


def canned_parser(job_dir, hidden=False):
    """the flags of the reference's canned trainers (trainers/linear.py:47-63, deep.py, linear_deep.py)"""
    from argparse import ArgumentParser
    parser = ArgumentParser()
    parser.add_argument("--train-csv", default="data/ml-100k/train.csv")
    parser.add_argument("--test-csv", default="data/ml-100k/test.csv")
    parser.add_argument("--restore", action="store_true")
    parser.add_argument("--job-dir", default=job_dir)
    parser.add_argument("--embedding-size", type=int, default=4)
    if hidden:
        parser.add_argument("--hidden-units", type=int, nargs="+", default=[16, 16])
        parser.add_argument("--dropout", type=float, default=0.1)
    parser.add_argument("--batch-size", type=int, default=32)
    parser.add_argument("--train-steps", type=int, default=20000)
    parser.add_argument("--seed", type=int, default=None)
    return parser


def train_and_evaluate(args):
    return canned_train_and_evaluate(args, lambda fc, a: DNNLinearCombinedClassifier(
        model_dir=a.job_dir, linear_feature_columns=fc["linear"], dnn_feature_columns=fc["deep"], dnn_hidden_units=a.hidden_units,
        dnn_dropout=a.dropout, max_batch=a.batch_size, tf_random_seed=a.seed))


if __name__ == "__main__":
    train_and_evaluate(canned_parser("checkpoints/linear_deep", hidden=True).parse_args())
