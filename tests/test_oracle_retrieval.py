"""CPU: the retrieval options of the two-tower oracle (oracle/twotower_retrieval.py) -- temperature, candidate sampling
probabilities and sample weights in the order of tfrs Retrieval.call -- against an independent autograd restatement,
with neutral options against the option-free oracle, and the streaming frequency estimator on a hand-worked case."""
import numpy as np
import pytest
import torch

from oracle import twotower as OT
from oracle import twotower_retrieval as OR

U, I, E, S, B = 60, 25, 16, 12, 40


def _batch(seed):
    rng = np.random.default_rng(seed)
    u = rng.integers(2, U + 2, B)
    i = rng.integers(2, I + 2, B)                                      # 25 items over 40 rows: accidental hits
    return u, i


def _restated(o, u, i, tau, p, w):
    """The TFRS call order written out in float64: logits / tau, minus log(clip(p)), hits masked, weighted SUM of
    logsumexp - label logit."""
    t = {k: v.detach().double().clone().requires_grad_(True) for k, v in o.t.items()}
    q = t["Eu"][torch.as_tensor(u)] @ t["Wu"] + t["bu"]
    c = t["Ei"][torch.as_tensor(i)] @ t["Wi"] + t["bi"]
    s = (q @ c.T) / tau
    s = s - torch.log(torch.clamp(torch.as_tensor(p, dtype=torch.float64), 1e-6, 1.0))[None, :]
    ids = torch.as_tensor(i)
    hit = (ids[:, None] == ids[None, :]) & ~torch.eye(B, dtype=torch.bool)
    s = torch.where(hit, s + float(np.finfo(np.float32).min) / 100.0, s)
    loss = (torch.as_tensor(w, dtype=torch.float64) * (torch.logsumexp(s, 1) - torch.diagonal(s))).sum()
    loss.backward()
    return float(loss.detach()), {k: v.grad for k, v in t.items()}


@pytest.mark.parametrize("tau", [0.05, 1.0, 3.0])
def test_options_match_the_tfrs_call_order(tau):
    u, i = _batch(1)
    rng = np.random.default_rng(2)
    p = (1.0 / (1.0 + np.arange(B)) ** 2).astype(np.float32)          # skewed, the tail below the 1e-6 clip
    p[B // 2:] = 1e-8
    rng.shuffle(p)
    w = rng.uniform(0.0, 2.0, B).astype(np.float32)
    w[[0, 7, 19]] = 0.0
    o = OR.RetrievalOracle(U, I, E, S, seed=4, temperature=tau)
    loss = float(o.loss_and_grads(u, i, cand_ids=i, cand_prob=p, sample_weight=w))
    ref, grads = _restated(o, u, i, tau, p, w)
    np.testing.assert_allclose(loss, ref, rtol=2e-5)
    scale = max(g.abs().max().item() for g in grads.values())     # bu's entries cancel to ~0 in the sum over rows
    for k, g in grads.items():
        got = o.t[k].grad.double()
        assert (got - g).abs().max().item() <= 1e-5 * scale, (k, (got - g).abs().max().item(), scale)


def test_weight_zero_removes_the_row():
    u, i = _batch(3)
    o = OR.RetrievalOracle(U, I, E, S, seed=4, temperature=0.5)
    w = np.ones(B, np.float32)
    full = float(o.loss(u, i, cand_ids=i, sample_weight=w).detach())
    w[5] = 0.0
    part = float(o.loss(u, i, cand_ids=i, sample_weight=w).detach())
    keep = np.arange(B) != 5
    # row 5 only leaves as a query: its candidate stays a column of every other row
    ref, _ = _restated(o, u, i, 0.5, np.ones(B, np.float32), keep.astype(np.float32))
    np.testing.assert_allclose(part, ref, rtol=2e-5)
    assert part < full


def test_neutral_options_equal_the_option_free_oracle_bit_for_bit():
    u, i = _batch(5)
    base = OT.TwoTowerOracle(U, I, E, S, seed=9)
    opt = OR.RetrievalOracle(U, I, E, S, seed=9, temperature=1.0)
    lb = base.loss_and_grads(u, i, cand_ids=i)
    lo = opt.loss_and_grads(u, i, cand_ids=i, cand_prob=np.ones(B, np.float32), sample_weight=np.ones(B, np.float32))
    assert torch.equal(lb, lo)
    for k in base.t:
        assert torch.equal(base.t[k].grad, opt.t[k].grad), k
    # no options at all: the option-free loss itself, through Adagrad steps too
    plain = OR.RetrievalOracle(U, I, E, S, seed=9)
    base2 = OT.TwoTowerOracle(U, I, E, S, seed=9)
    for s in range(3):
        u, i = _batch(10 + s)
        assert plain.step(u, i, cand_ids=i) == base2.step(u, i, cand_ids=i)
    for k in base2.t:
        assert torch.equal(base2.t[k], plain.t[k]), k


def test_streaming_frequency_hand_worked_case():
    f = OR.StreamingFrequency(5, alpha=0.5)
    f.update([2, 3, 2])            # t = 1: gap[2] = .5 * 0 + .5 * 1 = .5 once (the duplicate is skipped); gap[3] = .5
    assert f.t == 1 and list(f.last) == [0, 0, 1, 1, 0] and list(f.gap) == [0, 0, 0.5, 0.5, 0]
    f.update([2, 4])               # t = 2: gap[2] = .25 + .5 * (2 - 1) = .75; gap[4] = .5 * 2 = 1
    assert list(f.last) == [0, 0, 2, 1, 2] and list(f.gap) == [0, 0, 0.75, 0.5, 1.0]
    f.update([3, 3, 4])            # t = 3: gap[3] = .25 + .5 * (3 - 1) = 1.25; gap[4] = .5 + .5 * 1 = 1
    assert list(f.last) == [0, 0, 2, 3, 3] and list(f.gap) == [0, 0, 0.75, 1.25, 1.0]
    assert f.gap.dtype == np.float32 and f.last.dtype == np.int64
    # p = 1 / gap, 1 where gap < 1 (never seen, or seen more than once per step on average)
    np.testing.assert_array_equal(f.probability([2, 3, 4, 0]), np.array([1.0, 0.8, 1.0, 1.0], np.float32))


def test_streaming_frequency_rounds_in_fp32():
    f = OR.StreamingFrequency(3, alpha=0.01)
    g = np.float32(0)
    for t in range(1, 8):
        f.update([1] if t % 3 else [1, 2])
        g = np.float32(np.float32(np.float32(0.99) * g) + np.float32(np.float32(0.01) * np.float32(1)))
        assert f.gap[1] == g
    assert f.gap[1].dtype == np.float32
