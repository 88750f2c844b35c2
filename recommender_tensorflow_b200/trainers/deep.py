"""Mirror of trainers/deep.py: the canned tf.estimator.DNNClassifier (trainers/deep.py:32-38) on the "deep"
(embedding) feature columns = DNN tower only, SUM loss, Adagrad with the canned default learning rate 0.05
(TF-1.12 canned/dnn.py).  DNNRegressor is the same model with the regression head."""
from ..engine import DeepFMEngine, default_optimizer
from .linear_deep import _CannedBase, canned_parser, canned_train_and_evaluate
from .ml_100k import FEATURE_DTYPES
from .model_utils import check_regression_head, weight_column_key

_LEARNING_RATE = 0.05


class DNNClassifier(_CannedBase):
    def __init__(self, hidden_units, feature_columns, model_dir=None, dropout=None, config=None, max_batch=4096, device=0,
                 feature_dtypes=FEATURE_DTYPES, tf_random_seed=None, weight_column=None):
        weight_column_key(weight_column)        # type check, as TF's constructor does
        self.weight_column = weight_column
        cols = list(feature_columns)
        if not cols:
            raise ValueError("feature_columns must be defined.")
        dims = {c.dimension for c in cols}
        if len(dims) != 1:
            raise NotImplementedError("all embedding columns must share one dimension")
        self.engine = DeepFMEngine([c.categorical_column for c in cols], (), embedding_size=dims.pop(),
                                   hidden_units=list(hidden_units), use_linear=False, use_mf=False, use_dnn=True,
                                   loss_reduction="sum", opt_deep=default_optimizer("Adagrad", _LEARNING_RATE),
                                   opt_linear=default_optimizer("Adagrad", _LEARNING_RATE), max_batch=max_batch, device=device,
                                   feature_dtypes=feature_dtypes, dropout=float(dropout or 0.0), weighted=weight_column is not None,
                                   head=self._ENGINE_HEAD[self.HEAD])
        self._finish_init(model_dir, tf_random_seed)


class DNNRegressor(DNNClassifier):
    """canned tf.estimator.DNNRegressor (TF 1.12): DNNClassifier's model, optimizer, checkpoint names and SUM reduction
    with the regression head"""
    HEAD = "regression"

    def __init__(self, hidden_units, feature_columns, model_dir=None, label_dimension=1, weight_column=None, dropout=None,
                 config=None, max_batch=4096, device=0, feature_dtypes=FEATURE_DTYPES, tf_random_seed=None):
        check_regression_head(label_dimension)
        super().__init__(hidden_units, feature_columns, model_dir=model_dir, dropout=dropout, config=config, max_batch=max_batch,
                         device=device, feature_dtypes=feature_dtypes, tf_random_seed=tf_random_seed, weight_column=weight_column)


def train_and_evaluate(args):
    return canned_train_and_evaluate(args, lambda fc, a: DNNClassifier(a.hidden_units, fc["deep"], model_dir=a.job_dir, dropout=a.dropout,
                                                                       max_batch=a.batch_size, tf_random_seed=a.seed))


if __name__ == "__main__":
    train_and_evaluate(canned_parser("checkpoints/deep", hidden=True).parse_args())
