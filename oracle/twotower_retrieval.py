"""ORACLE (test infrastructure, never the product path): tfrs.tasks.Retrieval's sampling-bias correction on top of
oracle/twotower.py, and the streaming frequency estimator of Yi et al. (RecSys 2019, "Sampling-bias-corrected neural
modeling for large corpus item recommendations", Algorithm 2) as a literal sequential loop.

Retrieval(temperature=tau).call(q, c, candidate_ids=ids, candidate_sampling_probability=p, sample_weight=w), in the
order of TFRS's Retrieval.call, for query row i and in-batch candidate column j:
  1. s_ij = q_i . c_j / tau                       (temperature None: tau = 1)
  2. s_ij -= log(clip(p_j, 1e-6, 1))              (every column, the label column included)
  3. accidental hits: finfo(float32).min / 100 added, as oracle/twotower.py
  4. loss = sum_i w_i (logsumexp_j s_ij - s_ii)   (w None: 1; reduction SUM)
With none of the options the loss is TwoTowerOracle.loss itself, so the results are those of the existing oracle bit for
bit.  The weights enter through cross_entropy's class weights: the label of row i is class i, so class weight i is the
sample weight of row i."""
import numpy as np
import torch

from .twotower import MIN_FLOAT, TwoTowerOracle

DEFAULT_ALPHA = 0.01


class RetrievalOracle(TwoTowerOracle):
    def __init__(self, *args, temperature=None, **kw):
        super().__init__(*args, **kw)
        self.temperature = temperature

    def loss(self, u_idx, i_idx, cand_ids=None, labels=None, cand_prob=None, sample_weight=None):
        if self.temperature is None and cand_prob is None and sample_weight is None:
            return super().loss(u_idx, i_idx, cand_ids, labels)
        if self.rdZero:
            raise ValueError("the retrieval options need the in-batch softmax")
        q, c = self.towers(u_idx, i_idx)
        scores = self.mm(q, c.T)
        B = scores.shape[0]
        if self.temperature is not None:
            scores = scores / self.temperature
        if cand_prob is not None:
            p = torch.as_tensor(np.asarray(cand_prob), dtype=self.dtype)
            scores = scores - torch.log(torch.clamp(p, 1e-6, 1.0))[None, :]
        if cand_ids is not None:
            ids = torch.as_tensor(np.asarray(cand_ids))
            dup = (ids[:, None] == ids[None, :]).to(self.dtype) - torch.eye(B, dtype=self.dtype)
            scores = scores + dup * MIN_FLOAT
        w = None if sample_weight is None else torch.as_tensor(np.asarray(sample_weight), dtype=self.dtype)
        return torch.nn.functional.cross_entropy(scores, torch.arange(B), weight=w, reduction="sum")

    def loss_and_grads(self, u_idx, i_idx, cand_ids=None, labels=None, cand_prob=None, sample_weight=None):
        for v in self.t.values():
            v.grad = None
        l = self.loss(u_idx, i_idx, cand_ids, labels, cand_prob, sample_weight)
        l.backward()
        return l.detach()

    def step(self, u_idx, i_idx, cand_ids=None, labels=None, cand_prob=None, sample_weight=None):
        l = self.loss_and_grads(u_idx, i_idx, cand_ids, labels, cand_prob, sample_weight)
        with torch.no_grad():
            for k, w in self.t.items():
                g = w.grad if w.grad is not None else torch.zeros_like(w)
                self.acc[k] += g * g
                w -= self.lr * g / (self.acc[k].sqrt() + 1e-7)
        return float(l)


class StreamingFrequency:
    """Algorithm 2 of Yi et al. with one exact slot per item-table row: last[y] (int64), gap[y] (fp32), step counter t.
    update(ids) is one training step: t += 1, then for every id in batch order whose last[y] is not yet t,
    gap[y] = (1 - alpha) gap[y] + alpha (t - last[y]) with each product and the sum rounded to fp32, last[y] = t."""

    def __init__(self, rows, alpha=DEFAULT_ALPHA):
        self.last = np.zeros(rows, np.int64)
        self.gap = np.zeros(rows, np.float32)
        self.t = 0
        self.alpha = np.float32(alpha)

    def update(self, ids):
        self.t += 1
        a = self.alpha
        om = np.float32(np.float32(1.0) - a)
        for y in np.asarray(ids).tolist():
            if self.last[y] == self.t:                   # a duplicate of this batch: updated once
                continue
            self.gap[y] = np.float32(np.float32(om * self.gap[y]) + np.float32(a * np.float32(self.t - self.last[y])))
            self.last[y] = self.t

    def probability(self, ids):
        g = self.gap[np.asarray(ids)]
        p = np.ones(len(g), np.float32)
        big = g >= 1.0
        p[big] = np.float32(1.0) / g[big]
        return np.clip(p, np.float32(1e-6), np.float32(1.0))
