"""Mirror of trainers/linear.py: the canned tf.estimator.LinearClassifier (trainers/linear.py:30-34) on the
"linear" feature columns = linear_model only, SUM loss, FTRL with the canned default learning rate
min(0.2, 1/sqrt(n_columns)) (TF-1.12 canned/linear.py).  LinearRegressor is the same model with the regression head."""
import math

from ..engine import DeepFMEngine, default_optimizer
from .linear_deep import _CannedBase, canned_parser, canned_train_and_evaluate
from .ml_100k import FEATURE_DTYPES
from .model_utils import check_regression_head, weight_column_key

_LEARNING_RATE = 0.2


class LinearClassifier(_CannedBase):
    def __init__(self, feature_columns, model_dir=None, config=None, max_batch=4096, device=0, feature_dtypes=FEATURE_DTYPES,
                 tf_random_seed=None, weight_column=None):
        weight_column_key(weight_column)        # type check, as TF's constructor does
        self.weight_column = weight_column
        cols = list(feature_columns)
        if not cols:
            raise ValueError("feature_columns must be defined.")
        lr = min(_LEARNING_RATE, 1.0 / math.sqrt(len(cols)))
        self.engine = DeepFMEngine(cols, (), use_linear=True, use_mf=False, use_dnn=False, loss_reduction="sum",
                                   opt_deep=default_optimizer("Ftrl", lr), opt_linear=default_optimizer("Ftrl", lr),
                                   max_batch=max_batch, device=device, feature_dtypes=feature_dtypes, weighted=weight_column is not None,
                                   head=self._ENGINE_HEAD[self.HEAD])
        self._finish_init(model_dir, tf_random_seed)      # (linear weights start at zero like TF's; the seed is unused here)


class LinearRegressor(LinearClassifier):
    """canned tf.estimator.LinearRegressor (TF 1.12): LinearClassifier's model, optimizer, checkpoint names and SUM
    reduction with the regression head"""
    HEAD = "regression"

    def __init__(self, feature_columns, model_dir=None, label_dimension=1, weight_column=None, config=None, max_batch=4096,
                 device=0, feature_dtypes=FEATURE_DTYPES, tf_random_seed=None):
        check_regression_head(label_dimension)
        super().__init__(feature_columns, model_dir=model_dir, config=config, max_batch=max_batch, device=device,
                         feature_dtypes=feature_dtypes, tf_random_seed=tf_random_seed, weight_column=weight_column)


def train_and_evaluate(args):
    return canned_train_and_evaluate(args, lambda fc, a: LinearClassifier(fc["linear"], model_dir=a.job_dir, max_batch=a.batch_size,
                                                                          tf_random_seed=a.seed))


if __name__ == "__main__":
    train_and_evaluate(canned_parser("checkpoints/linear").parse_args())
