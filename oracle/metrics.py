"""Reference of the heads' EVAL metrics as the device streams them (csrc/metrics.cuh, include/deepfm_b200.h
dfm_metric_state), in numpy.

Logistic head, TF 1.12:
- metrics_impl._confusion_matrix_at_thresholds casts the predictions to float32 and compares them with
  `constant(thresholds, dtype=float32)`, thresholds = [0 - 1e-7] + [(i + 1) / (num_thresholds - 1) for i in
  range(num_thresholds - 2)] + [1 + 1e-7] with num_thresholds = 200 (metrics_impl.auc), by `predictions > thresholds`.
  A sample therefore lands in bin = number of thresholds below its float32 p; tp / fp at threshold j are the positives /
  negatives of the bins above j.  Here p = float32(1) / (float32(1) + exp(-z)) in float32, the device's expression.
- labels are cast to bool (`math_ops.cast(labels, dtypes.bool)`); on 0/1 labels that is label > 0.5, the rule of the
  host get_binary_metrics, kept for any float label.
- head.py _eval_metric_ops: accuracy, precision and recall compare the class_ids = argmax([0, z]) = (z > 0), a tie
  going to class 0; precision = tp / (tp + fp) and recall = tp / (tp + fn), 0 when the denominator is not > 0
  (metrics_impl.precision / recall); accuracy_baseline = max(label/mean, 1 - label/mean) (head.py _accuracy_baseline).
- label/mean, prediction/mean, average_loss and loss are weighted sums; they are formed in float64, p and the sigmoid
  cross-entropy max(z, 0) - z y + log1p(exp(-|z|)) evaluated in float64 from the float32 logit, as the host function does.
Squared head (head.py _RegressionHeadWithMeanSquaredErrorLoss): sums of w, w y, w z and w (y - z)^2 in float64.

An unweighted batch counts with w = 1.  States add field by field: across batches in stream order, across ranks in rank
order.
"""
import numpy as np

BINS = 201


def thresholds():
    """TF 1.12's 200 AUC thresholds as float32, converted from the Python doubles as constant() does"""
    th = [0.0 - 1e-7] + [(i + 1) * 1.0 / (200 - 1) for i in range(200 - 2)] + [1.0 + 1e-7]
    return np.array(th, dtype=np.float32)


def prob32(logits):
    z = np.asarray(logits, dtype=np.float32)
    with np.errstate(over="ignore"):
        return np.float32(1) / (np.float32(1) + np.exp(-z))


def empty_state(head="logistic", weighted=False):
    return {"head": head, "weighted": bool(weighted), "n": np.int64(0), "bin_count": np.zeros((2, BINS), np.int64),
            "cls": np.zeros(4, np.int64), "bin_weight": np.zeros((2, BINS)), "w_cls": np.zeros(4), "sums": np.zeros(4)}


def batch_state(logits, labels, weights=None, head="logistic"):
    """the state of one batch"""
    z32 = np.asarray(logits, dtype=np.float32).reshape(-1)
    y32 = np.asarray(labels, dtype=np.float32).reshape(-1)
    w = np.ones(z32.shape, np.float64) if weights is None else np.asarray(weights, dtype=np.float32).astype(np.float64).reshape(-1)
    z, y = z32.astype(np.float64), y32.astype(np.float64)
    s = empty_state(head, weights is not None)
    s["n"] = np.int64(z.size)
    if head == "squared":
        s["sums"] = np.array([w.sum(), (w * y).sum(), (w * z).sum(), (w * (y - z) ** 2).sum()])
        return s
    bins = np.searchsorted(thresholds(), prob32(z32), side="left")      # number of thresholds t < p
    pos, cls = y32 > 0.5, z32 > 0
    for c, sel in ((0, ~pos), (1, pos)):
        s["bin_count"][c] = np.bincount(bins[sel], minlength=BINS)
        s["bin_weight"][c] = np.bincount(bins[sel], weights=w[sel], minlength=BINS)
    masks = (cls & pos, cls & ~pos, ~cls & pos, cls == pos)
    s["cls"] = np.array([m.sum() for m in masks], np.int64)
    s["w_cls"] = np.array([w[m].sum() for m in masks])
    p = 1.0 / (1.0 + np.exp(-z))
    loss = np.maximum(z, 0) - z * y + np.log1p(np.exp(-np.abs(z)))
    s["sums"] = np.array([w.sum(), (w * y).sum(), (w * p).sum(), (w * loss).sum()])
    return s


def add(a, b):
    """state a followed by state b"""
    out = dict(a)
    for k in ("n", "bin_count", "cls"):
        out[k] = a[k] + b[k]
    for k in ("bin_weight", "w_cls", "sums"):
        out[k] = a[k] + b[k]
    return out


def stream_state(batches, head="logistic", weighted=False):
    """batches: iterable of (logits, labels, weights or None) in stream order"""
    s = empty_state(head, weighted)
    for z, y, w in batches:
        s = add(s, batch_state(z, y, w, head))
    return s


def near_threshold(logits, ulps=8):
    """samples whose float32 p lies within `ulps` float32 steps of a threshold: the device's expf may put them in the
    neighbouring bin"""
    p = prob32(np.asarray(logits, dtype=np.float32).reshape(-1))
    th = thresholds()
    j = np.clip(np.searchsorted(th, p), 1, th.size - 1)
    gap = np.minimum(np.abs(p - th[j - 1]), np.abs(th[j] - p))
    return gap <= ulps * np.spacing(p)
