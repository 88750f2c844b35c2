"""Reference for per-example weights (weight_column): the oracle step with the binary head's weighted loss.

TF 1.12 (head.py _get_weights_and_check_match_logits, losses_impl.compute_weighted_loss): the per-sample loss and its
gradient dz are multiplied by the sample's weight; SUM gives sum(w l), SUM_OVER_BATCH_SIZE ('mean') sum(w l) / B - the
number of samples, not sum(w).  Without weights every method is OracleDeepFM's own."""
import numpy as np
import torch

from oracle.deepfm import OracleDeepFM
from tests.util import OraclePair, oracle_cfg


class WeightedOracleDeepFM(OracleDeepFM):
    _w = None        # weights of the step in progress (train_step / train_step_raw pass them down to grads)

    def grads(self, ids, x, y, w=None):
        w = self._w if w is None else w
        if w is None:
            return super().grads(ids, x, y)
        # OracleDeepFM.grads with the weight applied where lv and dz are formed; the backward below is its restatement
        z, c = self.forward(ids, x, keep=True, train=True)
        y = torch.as_tensor(np.asarray(y), dtype=self.dt)
        w = torch.as_tensor(np.asarray(w, dtype=np.float32).reshape(-1), dtype=self.dt)
        B = z.shape[0]
        lv = self.loss_vec(z, y) * w
        loss = lv.mean() if self.red == "mean" else lv.sum()
        dz = torch.sigmoid(z) - y
        if self.red == "mean":
            dz = dz / B
        dz = dz * w
        W = {n: v.w for n, v in self.vars.items()}
        g = {}
        rows, valid, x = c["rows"], c["valid"], c["x"]
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
        return loss, z, g

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


def weighted_pair(engine, weights):
    """float32 / float64 weighted oracles of `engine` from the initial weights make_pair injected into it"""
    cfg = oracle_cfg(engine)
    return OraclePair(WeightedOracleDeepFM(cfg, weights), WeightedOracleDeepFM(cfg, weights, dtype=torch.float64))


def weighted_step(pair, feats, y, w):
    """one weighted step of both oracles of an OraclePair (pair.last64 calibrates the tolerances, as in tests/util.py)"""
    pair.last64 = pair.o64.train_step_raw(feats, y, w)
    return pair.o32.train_step_raw(feats, y, w)
