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
    if curve == "ROC":
        x = fp / (fp + tn + eps)
        y = (tp + eps) / (tp + fn + eps)
    else:
        x = (tp + eps) / (tp + fn + eps)
        y = (tp + eps) / (tp + fp + eps)
    return float(np.sum((x[:-1] - x[1:]) * (y[:-1] + y[1:]) / 2.0))


def get_binary_metrics(labels, logits, weights=None):
    """Metrics the binary head reports in EVAL mode (accuracy, auc, auc_precision_recall,
    average_loss, label/mean, prediction/mean; cf. trainers/model_utils.py:39-54).  weights (weight_column, head.py
    _eval_metric_ops): every metric is weighted - means are sum(w x) / sum(w), the AUC confusion counts are sums of
    weights, and loss is sum(w l)."""
    y = np.asarray(labels, dtype=np.float64).reshape(-1)
    z = np.asarray(logits, dtype=np.float64).reshape(-1)
    p = 1.0 / (1.0 + np.exp(-z))
    loss = np.maximum(z, 0) - z * y + np.log1p(np.exp(-np.abs(z)))
    if weights is not None:
        w = np.asarray(weights, dtype=np.float32).astype(np.float64).reshape(-1)
        if w.shape != y.shape:
            raise ValueError("weights shape %s does not match labels %s" % (list(w.shape), list(y.shape)))
        sw = w.sum()
        return {"accuracy": float((w * ((p > 0.5) == (y > 0.5))).sum() / sw), "auc": _auc(y, p, weights=w),
                "auc_precision_recall": _auc(y, p, "PR", weights=w), "average_loss": float((w * loss).sum() / sw),
                "loss": float((w * loss).sum()), "label/mean": float((w * y).sum() / sw), "prediction/mean": float((w * p).sum() / sw)}
    return {"accuracy": float(((p > 0.5) == (y > 0.5)).mean()), "auc": _auc(y, p), "auc_precision_recall": _auc(y, p, "PR"),
            "average_loss": float(loss.mean()), "loss": float(loss.sum()), "label/mean": float(y.mean()),
            "prediction/mean": float(p.mean())}


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
