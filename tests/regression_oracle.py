"""Reference for the squared head (DFM_HEAD_SQUARED, the regressors): the oracle step with TF 1.12's regression head.

regression_head / canned *Regressor (head.py _RegressionHeadWithMeanSquaredErrorLoss, label_dimension 1, no
inverse_link_fn): the per-sample loss is losses.mean_squared_error unreduced, l_b = (y_b - z_b)^2 with y = tf.to_float
(label), so dz_b = 2 (z_b - y_b).  SUM gives sum(w l), SUM_OVER_BATCH_SIZE ('mean') sum(w l) / B; the weight (when
given) multiplies l_b and dz_b after the reduction scale, as for the binary head.  head="logistic" without weights is
OracleDeepFM's own step; the backward below restates OracleDeepFM.grads with dz as its input."""
import numpy as np
import torch

from oracle.deepfm import OracleDeepFM
from tests.util import OraclePair, oracle_cfg


class HeadOracleDeepFM(OracleDeepFM):
    _w = None        # weights of the step in progress (train_step / train_step_raw pass them down to grads)

    def __init__(self, cfg, weights, dtype=torch.float32):
        super().__init__(cfg, weights, dtype)
        self.head = cfg.get("head", "logistic")
        if self.head not in ("logistic", "squared"):
            raise ValueError(self.head)

    def loss_vec(self, z, y):
        if self.head == "squared":
            d = z - y
            return d * d
        return OracleDeepFM.loss_vec(z, y)

    def grads(self, ids, x, y, w=None):
        w = self._w if w is None else w
        if w is None and self.head == "logistic":
            return super().grads(ids, x, y)
        z, c = self.forward(ids, x, keep=True, train=True)
        y = torch.as_tensor(np.asarray(y, dtype=np.float32).reshape(-1), dtype=self.dt)
        B = z.shape[0]
        lv = self.loss_vec(z, y)
        dz = 2 * (z - y) if self.head == "squared" else torch.sigmoid(z) - y
        if self.red == "mean":
            dz = dz / B
        if w is not None:
            wt = torch.as_tensor(np.asarray(w, dtype=np.float32).reshape(-1), dtype=self.dt)
            lv = lv * wt
            dz = dz * wt
        loss = lv.mean() if self.red == "mean" else lv.sum()
        return loss, z, self.backward(c, dz)

    def backward(self, c, dz):
        """OracleDeepFM.grads from dz = dL/dz on: the gradient of every variable"""
        W = {n: v.w for n, v in self.vars.items()}
        g = {}
        rows, valid, x = c["rows"], c["valid"], c["x"]
        B = dz.shape[0]
        flat_rows = rows[valid]
        if self.use_linear:
            g["lin"] = ("sparse", flat_rows, dz[:, None].expand(B, self.n_slots)[valid])
            g["bias"] = dz.sum().reshape(1)
            if self.dn:
                g["num_lin"] = x.t() @ dz
        if self.use_mf or self.use_dnn:
            E = c["E"]
            dE = torch.zeros_like(E)
            if self.use_mf:
                dE = dE + dz[:, None, None] * (c["s"][:, None, :] - E)
            if self.use_dnn:
                acts = c["acts"]
                L = len(self.hidden)
                dh = dz[:, None] * W["Wo"][:, 0][None, :]
                g["Wo"] = acts[L].t() @ dz[:, None]
                g["bo"] = dz.sum().reshape(1)
                fprime = {"relu": lambda yv: (yv > 0).to(self.dt), "tanh": lambda yv: 1 - yv * yv,
                          "sigmoid": lambda yv: yv * (1 - yv), "identity": lambda yv: torch.ones_like(yv)}[self.activation]
                for i in reversed(range(L)):
                    dh = dh * fprime(c["pre"][i])
                    if c["masks"][i] is not None:
                        dh = dh * c["masks"][i]
                    g["W%d" % i] = acts[i].t() @ dh
                    g["b%d" % i] = dh.sum(0)
                    dh = dh @ W["W%d" % i].t()
                dE = dE + dh.reshape(E.shape)
            dEs = (dE[:, :self.dc] * c["inv"][:, :, None])[:, self.slot_field]
            g["emb"] = ("sparse", flat_rows, dEs[valid])
            if self.dn:
                g["num_emb"] = (x[:, :, None] * dE[:, self.dc:]).sum(0)
        return g

    def train_step(self, ids, x, y, w=None):
        prev, self._w = self._w, (self._w if w is None else w)
        try:
            return super().train_step(ids, x, y)
        finally:
            self._w = prev

    def train_step_raw(self, features, labels, weights=None):
        prev, self._w = self._w, weights
        try:
            return super().train_step_raw(features, labels)
        finally:
            self._w = prev


class HeadOraclePair(OraclePair):
    """float32 / float64 oracles with a head and optional per-example weights"""

    def train_step_raw(self, feats, y, w=None):
        self.last64 = self.o64.train_step_raw(feats, y, w)
        return self.o32.train_step_raw(feats, y, w)


def head_pair(engine, weights):
    """oracles of `engine` (its head included) from the initial weights make_pair injected into it"""
    cfg = oracle_cfg(engine, head=engine.head)
    return HeadOraclePair(HeadOracleDeepFM(cfg, weights), HeadOracleDeepFM(cfg, weights, dtype=torch.float64))
