"""Mirror of trainers/model_utils.py: optimizer lookup and the binary and regression heads' outputs."""
import numpy as np

from ..engine import default_optimizer
from ..feature_column import NumericColumn


def layer_summary(value):
    """trainers/model_utils.py:4-6: tf.nn.zero_fraction scalar + activation histogram of a tensor, host side."""
    v = np.asarray(value, dtype=np.float32).reshape(-1)
    hist, edges = np.histogram(v, bins=30) if v.size else (np.zeros(30, int), np.zeros(31))
    return {"fraction_of_zero_values": float((v == 0).mean()) if v.size else 0.0, "activation": (hist, edges)}


def get_optimizer(optimizer_name="Adam", learning_rate=0.001):
    """trainers/model_utils.py:57-66 — Adagrad | Adam | Ftrl | RMSProp | SGD with `learning_rate` only
    (an unknown name raises KeyError, like optimizer_classes[optimizer_name] in the reference)."""
    return default_optimizer(optimizer_name, learning_rate)


def get_binary_predictions(logits):
    """trainers/model_utils.py:9-21 / binary head predictions."""
    logits = np.asarray(logits, dtype=np.float32).reshape(-1, 1)
    logistic = 1.0 / (1.0 + np.exp(-logits))
    return {"logits": logits, "logistic": logistic, "probabilities": np.concatenate([1 - logistic, logistic], 1),
            "class_ids": (logistic > 0.5).astype(np.int64), "class_id": (logistic > 0.5).astype(np.int32)}


def get_regression_predictions(logits):
    """regression_head predictions (TF 1.12 head.py _RegressionHeadWithMeanSquaredErrorLoss, identity inverse link):
    the logits [B, 1] under the key "predictions"; there are no probabilities or classes."""
    return {"predictions": np.asarray(logits, dtype=np.float32).reshape(-1, 1)}


def check_regression_head(label_dimension=1, inverse_link_fn=None, loss_fn=None, n_classes=None):
    """The regression head is built for label_dimension = 1 with the identity inverse link and the mean squared error;
    anything else is rejected rather than silently trained as that model."""
    if label_dimension != 1:
        raise ValueError("label_dimension must be 1 (got %r): only single-output regression is implemented" % (label_dimension,))
    if inverse_link_fn is not None:
        raise ValueError("inverse_link_fn is not supported: the regression head predicts the logits (identity link)")
    if loss_fn is not None:
        raise ValueError("a custom loss_fn is not supported: the regression head's loss is the squared error")
    if n_classes not in (None, 2):
        raise ValueError("n_classes=%r: multi-class heads are not supported" % (n_classes,))


def weight_column_key(weight_column):
    """weight_column of the estimators / binary head: None, a feature key or a numeric_column -> the feature key or None"""
    if weight_column is None:
        return None
    if isinstance(weight_column, str):
        return weight_column
    if isinstance(weight_column, NumericColumn):
        return weight_column.key
    raise TypeError("Weight column must be either a string or _NumericColumn. Given type: {}.".format(type(weight_column)))


def get_weights(features, weight_column, n):
    """head.py _get_weights_and_check_match_logits (TF 1.12): the weight feature as float32 [n] (tf.to_float).  A missing
    feature raises KeyError, weights whose shape does not match the n logits ([n] or [n, 1]) raise ValueError.  Zero,
    negative and fractional weights are accepted, as in TF.  A device batch (PackedBatch) carries its weights inside
    the batch; its host copy, when one was read back for the metrics, is its `weights` attribute."""
    key = weight_column_key(weight_column)
    if key is None:
        return None
    if isinstance(features, dict):
        if key not in features:
            raise KeyError(key)
        w = features[key]
    else:
        w = getattr(features, "weights", None)
        if w is None:
            raise KeyError(key)
    w = np.asarray(w).astype(np.float32)
    if w.shape not in ((n,), (n, 1)):
        raise ValueError("weights shape must be [D0, 1] or [D0] matching logits [%d, 1]; got %s" % (n, list(w.shape)))
    return w.reshape(-1)


def _auc(labels, probs, curve="ROC", num_thresholds=200, weights=None):
    """tf.metrics.auc: trapezoidal over num_thresholds evenly spaced thresholds (+/- epsilon ends).  weights: the
    confusion counts are sums of the per-example weights."""
    eps = 1e-7
    th = np.concatenate([[0.0 - eps], (np.arange(1, num_thresholds - 1)) / (num_thresholds - 1.0), [1.0 + eps]])
    pos = labels > 0.5
    pred = probs[None, :] > th[:, None]
    if weights is None:
        tp = (pred & pos[None, :]).sum(1).astype(np.float64)
        fp = (pred & ~pos[None, :]).sum(1).astype(np.float64)
        fn = pos.sum() - tp
        tn = (~pos).sum() - fp
    else:
        tp = (pred & pos[None, :]).astype(np.float64) @ weights
        fp = (pred & ~pos[None, :]).astype(np.float64) @ weights
        fn = weights[pos].sum() - tp
        tn = weights[~pos].sum() - fp
    return _auc_trapezoid(tp, fp, fn, tn, curve)


def _auc_trapezoid(tp, fp, fn, tn, curve="ROC"):
    """tf.metrics.auc's summation_method='trapezoidal' over the confusion counts at the thresholds (ascending)"""
    eps = 1e-7
    if curve == "ROC":
        x = fp / (fp + tn + eps)
        y = (tp + eps) / (tp + fn + eps)
    else:
        x = (tp + eps) / (tp + fn + eps)
        y = (tp + eps) / (tp + fp + eps)
    return float(np.sum((x[:-1] - x[1:]) * (y[:-1] + y[1:]) / 2.0))


def _safe_div(num, den):
    """metrics_impl precision / recall: num / den where den > 0, else 0"""
    return float(num / den) if den > 0 else 0.0


def get_binary_metrics(labels, logits, weights=None):
    """Metrics the binary head reports in EVAL mode (accuracy, accuracy_baseline, auc, auc_precision_recall,
    average_loss, label/mean, precision, prediction/mean, recall; cf. trainers/model_utils.py:39-54 and TF 1.12 head.py
    _eval_metric_ops).  precision and recall are those of the predicted class p > 0.5 (0 when nothing is predicted
    positive, resp. nothing is positive, as metrics_impl's _safe_div); accuracy_baseline is max(label/mean,
    1 - label/mean) (head.py _accuracy_baseline).  weights (weight_column): every metric is weighted - means are
    sum(w x) / sum(w), the AUC and precision / recall counts are sums of weights, and loss is sum(w l)."""
    y = np.asarray(labels, dtype=np.float64).reshape(-1)
    z = np.asarray(logits, dtype=np.float64).reshape(-1)
    p = 1.0 / (1.0 + np.exp(-z))
    loss = np.maximum(z, 0) - z * y + np.log1p(np.exp(-np.abs(z)))
    pred, pos = p > 0.5, y > 0.5
    if weights is not None:
        w = np.asarray(weights, dtype=np.float32).astype(np.float64).reshape(-1)
        if w.shape != y.shape:
            raise ValueError("weights shape %s does not match labels %s" % (list(w.shape), list(y.shape)))
        sw = w.sum()
        tp, fp, fn = w[pred & pos].sum(), w[pred & ~pos].sum(), w[~pred & pos].sum()
        m = {"accuracy": float((w * (pred == pos)).sum() / sw), "auc": _auc(y, p, weights=w),
             "auc_precision_recall": _auc(y, p, "PR", weights=w), "average_loss": float((w * loss).sum() / sw),
             "loss": float((w * loss).sum()), "label/mean": float((w * y).sum() / sw), "prediction/mean": float((w * p).sum() / sw)}
    else:
        tp, fp, fn = (pred & pos).sum(), (pred & ~pos).sum(), (~pred & pos).sum()
        m = {"accuracy": float((pred == pos).mean()), "auc": _auc(y, p), "auc_precision_recall": _auc(y, p, "PR"),
             "average_loss": float(loss.mean()), "loss": float(loss.sum()), "label/mean": float(y.mean()),
             "prediction/mean": float(p.mean())}
    m["precision"], m["recall"] = _safe_div(tp, tp + fp), _safe_div(tp, tp + fn)
    m["accuracy_baseline"] = max(m["label/mean"], 1.0 - m["label/mean"])
    return m


def get_regression_metrics(labels, logits, weights=None):
    """Metrics the regression head reports in EVAL mode (TF 1.12 head.py _RegressionHeadWithMeanSquaredErrorLoss.
    _eval_metric_ops: average_loss, label/mean, prediction/mean) plus `loss`, the summed loss, as for the binary head.
    The per-example loss is (y - z)^2; weights (weight_column) make every metric weighted: means are
    sum(w x) / sum(w) and loss is sum(w l)."""
    y = np.asarray(labels, dtype=np.float64).reshape(-1)
    z = np.asarray(logits, dtype=np.float64).reshape(-1)
    if y.shape != z.shape:
        raise ValueError("labels shape %s does not match logits %s (label_dimension is 1)" % (list(y.shape), list(z.shape)))
    loss = (y - z) ** 2
    w = np.ones_like(y)
    if weights is not None:
        w = np.asarray(weights, dtype=np.float32).astype(np.float64).reshape(-1)
        if w.shape != y.shape:
            raise ValueError("weights shape %s does not match labels %s" % (list(w.shape), list(y.shape)))
    sw = w.sum()
    return {"average_loss": float((w * loss).sum() / sw), "loss": float((w * loss).sum()),
            "label/mean": float((w * y).sum() / sw), "prediction/mean": float((w * z).sum() / sw)}


# ---------------------------------------------------------------------------- metrics streamed on the device
# A metric state (DeepFMEngine.metrics_state, dfm_metric_state in include/deepfm_b200.h) is a dict:
#   head "logistic" | "squared", weighted (bool);
#   int64:   n, bin_count [2, 201] (negatives, positives per bin = number of TF's 200 float32 thresholds below the float32
#            p), cls [4] = tp, fp, fn, correct of the class z > 0 against label > 0.5;
#   float64: bin_weight [2, 201] and w_cls [4], the same as sums of the weights, and sums [4] = sum w, sum w y,
#            sum w pred (p, or z for the squared head), sum w loss.
STATE_INT_FIELDS = ("n", "bin_count", "cls")
STATE_FLOAT_FIELDS = ("bin_weight", "w_cls", "sums")


def combine_metric_states(states):
    """The states of several ranks (or stream segments) as one: integer fields summed, float64 fields summed in the
    order given (rank order), so every rank that combines the same list gets the same bits."""
    states = list(states)
    if not states:
        raise ValueError("combine_metric_states: no states")
    out = {"head": states[0]["head"], "weighted": states[0]["weighted"]}
    for s in states[1:]:
        if (s["head"], s["weighted"]) != (out["head"], out["weighted"]):
            raise ValueError("metric states of different heads / weighting cannot be combined")
    for k in STATE_INT_FIELDS:
        out[k] = np.sum([np.asarray(s[k], dtype=np.int64) for s in states], axis=0, dtype=np.int64)
    for k in STATE_FLOAT_FIELDS:
        acc = np.array(states[0][k], dtype=np.float64)
        for s in states[1:]:
            acc = acc + np.asarray(s[k], dtype=np.float64)
        out[k] = acc
    return out


def finish_binary_metrics(state):
    """get_binary_metrics' keys from a logistic-head metric state: the same _auc trapezoid over the per-threshold
    confusion counts (suffix sums of the bins) and the same epsilon and _safe_div conventions.  Unweighted states are
    finished from the exact int64 counts, weighted ones from the float64 weight sums."""
    if state["head"] != "logistic":
        raise ValueError("finish_binary_metrics: the state is of the %s head" % state["head"])
    weighted = bool(state["weighted"])
    bins = np.asarray(state["bin_weight"] if weighted else state["bin_count"]).astype(np.float64)
    tp_c, fp_c, fn_c, ok_c = (np.asarray(state["w_cls"] if weighted else state["cls"]).astype(np.float64))
    sw, swy, swp, swl = np.asarray(state["sums"], dtype=np.float64)
    if not weighted:
        sw = float(state["n"])
    # tp / fp at threshold j: the positives / negatives in bins j + 1 .. 200 (p above threshold j)
    tp = np.cumsum(bins[1, ::-1])[::-1][1:]
    fp = np.cumsum(bins[0, ::-1])[::-1][1:]
    fn = bins[1].sum() - tp
    tn = bins[0].sum() - fp
    lm = float(swy / sw)
    return {"accuracy": float(ok_c / sw), "accuracy_baseline": max(lm, 1.0 - lm),
            "auc": _auc_trapezoid(tp, fp, fn, tn), "auc_precision_recall": _auc_trapezoid(tp, fp, fn, tn, "PR"),
            "average_loss": float(swl / sw), "loss": float(swl), "label/mean": lm,
            "precision": _safe_div(tp_c, tp_c + fp_c), "prediction/mean": float(swp / sw), "recall": _safe_div(tp_c, tp_c + fn_c)}


def finish_regression_metrics(state):
    """get_regression_metrics' keys from a squared-head metric state"""
    if state["head"] != "squared":
        raise ValueError("finish_regression_metrics: the state is of the %s head" % state["head"])
    sw, swy, swz, swl = np.asarray(state["sums"], dtype=np.float64)
    if not state["weighted"]:
        sw = float(state["n"])
    return {"average_loss": float(swl / sw), "loss": float(swl), "label/mean": float(swy / sw), "prediction/mean": float(swz / sw)}


def finish_metrics(state):
    """the metrics of the state's head"""
    return finish_binary_metrics(state) if state["head"] == "logistic" else finish_regression_metrics(state)
