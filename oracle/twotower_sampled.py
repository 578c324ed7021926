"""ORACLE (test infrastructure, never the product path): mixed negative sampling for two-tower training (Yang et al.,
WWW 2020, "Mixed negative sampling for learning two-tower neural networks in recommendations"): the sampled-negative
stream and TFRS Retrieval called with more candidates than queries.

Stream.  Draw k (0 <= k < M) of training step t (the first step is t = 1) for replica r, from item-table rows [lo, hi):
  w = philox4x32_10(ctr = (k, uint32(t), uint32(t >> 32), TAG_TWOTOWER_NEG), key = (seed, r))
  id = lo + ((w.x * (hi - lo)) >> 32)                         (oracle/philox.py's _mulshift)
Uniform with replacement.  r is 0 in a single process; on real ranks each replica draws with its rank.

Loss.  Retrieval.call(q, c_all, candidate_ids=ids_all) with c_all = item tower of concat(i, sampled) (n = B + M rows):
labels tf.eye(B, n), so the label of row b is column b; column j != b whose id equals i[b] gets finfo(float32).min / 100
(a sampled copy of the row's own positive is masked too); logits times 1 / temperature; loss = sum_b w_b (lse_b - s_bb).
Candidate probabilities are not defined with sampled negatives (the logQ correction of a mixed pool needs each sampled
column's probability under both routes)."""
import numpy as np
import torch

from .philox import MASK, _mulshift, philox4x32_10
from .twotower import MIN_FLOAT
from .twotower_retrieval import RetrievalOracle

TAG_TWOTOWER_NEG = 0x7E


def sampled_negatives(M, seed, step, replica, lo, hi):
    """The M rows (int32) that training step `step` of replica `replica` draws from [lo, hi)."""
    k = np.arange(M, dtype=np.uint64)
    t = np.uint64(step)
    ctr = np.stack([k & MASK, np.full(M, t & MASK, np.uint64), np.full(M, t >> np.uint64(32), np.uint64),
                    np.full(M, TAG_TWOTOWER_NEG, np.uint64)], axis=1).astype(np.uint32)
    w = philox4x32_10(ctr, (seed, replica))[:, 0]
    return (lo + _mulshift(w, hi - lo)).astype(np.int32)


class SampledOracle(RetrievalOracle):
    """RetrievalOracle whose loss / step take extra candidate rows `sampled` (item-table rows)."""

    def loss(self, u_idx, i_idx, cand_ids=None, labels=None, cand_prob=None, sample_weight=None, sampled=None):
        if sampled is None or len(sampled) == 0:
            return super().loss(u_idx, i_idx, cand_ids, labels, cand_prob, sample_weight)
        if self.rdZero or cand_prob is not None:
            raise ValueError("sampled negatives need the in-batch softmax and take no candidate probabilities")
        i_idx, sampled = np.asarray(i_idx), np.asarray(sampled)
        q, c = self.towers(u_idx, np.concatenate([i_idx, sampled]))
        scores = self.mm(q, c.T)
        B, n = scores.shape
        if self.temperature is not None:
            scores = scores / self.temperature
        if cand_ids is not None:
            ids = torch.as_tensor(np.asarray(cand_ids).astype(np.int64))
            ids_all = torch.cat([ids, torch.as_tensor(sampled.astype(np.int64))])
            dup = (ids[:, None] == ids_all[None, :]).to(self.dtype) - torch.eye(B, n, dtype=self.dtype)
            scores = scores + dup * MIN_FLOAT
        w = None
        if sample_weight is not None:                        # class weights: the label of row b is class b < B
            w = torch.zeros(n, dtype=self.dtype)
            w[:B] = torch.as_tensor(np.asarray(sample_weight), dtype=self.dtype)
        return torch.nn.functional.cross_entropy(scores, torch.arange(B), weight=w, reduction="sum")

    def loss_and_grads(self, u_idx, i_idx, cand_ids=None, labels=None, cand_prob=None, sample_weight=None, sampled=None):
        for v in self.t.values():
            v.grad = None
        l = self.loss(u_idx, i_idx, cand_ids, labels, cand_prob, sample_weight, sampled)
        l.backward()
        return l.detach()

    def step(self, u_idx, i_idx, cand_ids=None, labels=None, cand_prob=None, sample_weight=None, sampled=None):
        l = self.loss_and_grads(u_idx, i_idx, cand_ids, labels, cand_prob, sample_weight, sampled)
        with torch.no_grad():
            for k, w in self.t.items():
                g = w.grad if w.grad is not None else torch.zeros_like(w)
                self.acc[k] += g * g
                w -= self.lr * g / (self.acc[k].sqrt() + 1e-7)
        return float(l)
