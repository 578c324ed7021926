"""Mixed negative sampling for two-tower training (brk_tt_sampled: brk_twotower_step_sampled,
brk_twotower_train_step_sampled, brk_twotower_step_sharded_sampled; TwoTowerModel / ShardedTwoTowerNet(sampledNegatives=M))
against oracle/twotower_sampled.py: the drawn rows bit for bit, the loss and the trained state with the oracle's extra
candidate columns."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U, I = 301, 203
SEED = 42
LOSS_TOL = dict(rtol=1e-5, atol=1e-6)
W_TOL = dict(rtol=2e-3, atol=1e-4)                        # two GPUs, E = 32: test_gpu_twotower_sharded_retrieval.py's
MOVED_SHARE = {True: 1e-2, False: 1e-3}                   # test_gpu_twotower_sharded_retrieval.py's


def _model(dev, E, S, tc, nI=I, **kw):
    from binrec_b200.twoTower import TwoTowerModel
    m = TwoTowerModel(E, nI, U, "u", "i", list(range(U)), list(range(nI)), semb=S, device=dev, tensor_cores=tc, seed=SEED,
                      **kw)
    m.compile("Adagrad", learningRate=0.1)
    return m


def _oracle(m, E, S, tc, tau=None, nI=I):
    from oracle import tf32
    from oracle import twotower_sampled as OS
    o = OS.SampledOracle(U, nI, E, S, seed=SEED, temperature=tau, matmul=tf32.matmul if tc else torch.matmul)
    with torch.no_grad():
        o.t["Eu"].copy_(m.userTower.emb.w.cpu()); o.t["Ei"].copy_(m.itemTower.emb.w.cpu())
        for tw, wn, bn in ((m.userTower, "Wu", "bu"), (m.itemTower, "Wi", "bi")):
            flat = tw.dense.w.view(-1).cpu()
            o.t[wn].copy_(flat[:E * S].view(E, S)); o.t[bn].copy_(flat[E * S:E * S + S])
    return o


def _draws(M, step, replica=0, nI=I, seed=SEED):
    from oracle import twotower_sampled as OS
    return OS.sampled_negatives(M, seed, step, replica, 2, nI + 2)


def _ids(rng, B, nI=I):
    f = lambda n: rng.random(n) ** 2                      # skewed: popular rows repeat, accidental hits
    return (2 + (U * f(B))).astype(np.int32), (2 + (nI * f(B))).astype(np.int32)


class _Trace:
    """BRK_TT_TRACE pointed at a zeroed device buffer: the one-launch step stamps it, the multi-kernel step does not."""

    def __init__(self, dev, monkeypatch):
        self.buf = torch.zeros(16, dtype=torch.int64, device=dev)
        self.mp = monkeypatch

    def __enter__(self):
        self.mp.setenv("BRK_TT_TRACE", hex(self.buf.data_ptr()))

    def __exit__(self, *a):
        self.mp.delenv("BRK_TT_TRACE")

    def stamped(self):
        torch.cuda.synchronize()
        return bool((self.buf[:8] != 0).all().item())


def _call_draw(dev, m, **over):
    """brk_twotower_step_sampled with batch 0: only the draws (and the counter) -- any range, seed and replica."""
    from binrec_b200 import _native as N
    smp = m._smp.c_struct()
    for k, v in over.items():
        setattr(smp, k, v)
    ws = m._workspace(1)
    ut, it = m.userTower.c_struct(), m.itemTower.c_struct()
    loss = torch.ones(1, dtype=torch.float32, device=dev)
    rc = N.lib().brk_twotower_step_sampled(N.ctx(dev), C.byref(ut), C.byref(it), None, None, 0, 0x100, C.byref(ws),
                                           N.ptr(loss), N.stream_ptr(), C.byref(smp), None)
    return rc, loss


@pytest.mark.parametrize("seed,step0,replica,M,lo,hi", [(42, 0, 0, 1, 2, 205), (7, 5, 0, 1000, 2, 205),
                                                         (123456789, 2 ** 32 + 3, 3, 129, 0, 3),
                                                         (0xFFFFFFFF, 2 ** 40, 7, 4096, 100, 101), (1, 9, 1, 2500, 2, 205)])
def test_draws_equal_the_oracle_stream(dev, seed, step0, replica, M, lo, hi):
    from oracle import twotower_sampled as OS
    m = _model(dev, 32, 16, True, sampledNegatives=M)
    m._smp.step.fill_(step0)
    for k in range(2):
        rc, loss = _call_draw(dev, m, seed=seed, replica=replica, lo=lo, hi=hi)
        assert rc == 0
        torch.cuda.synchronize()
        want = OS.sampled_negatives(M, seed, step0 + 1 + k, replica, lo, hi)
        assert np.array_equal(m._smp.ids.cpu().numpy(), want)
        assert int(m._smp.step.item()) == step0 + 1 + k
        assert float(loss.item()) == 0.0
    ids = m._smp.ids.cpu().numpy()
    assert ids.min() >= lo and ids.max() < hi


def test_counter_advances_per_training_step_and_graph_replay_not_on_test_step(dev):
    M, B = 64, 100
    m = _model(dev, 32, 16, True, sampledNegatives=M)
    rng = np.random.default_rng(1)
    batches = []
    for _ in range(6):
        u, i = _ids(rng, B)
        batches.append({"u": [int(x) - 2 for x in u], "i": [int(x) - 2 for x in i]})
    m.train_step(batches[0]); m.train_step(batches[1])
    torch.cuda.synchronize()
    assert int(m._smp.step.item()) == 2
    assert np.array_equal(m._smp.ids.cpu().numpy(), _draws(M, 2))
    m.test_step(batches[2])
    torch.cuda.synchronize()
    assert int(m._smp.step.item()) == 2 and np.array_equal(m._smp.ids.cpu().numpy(), _draws(M, 2))
    m.fit(batches, epochs=2, graph=True)                 # batch 0 eager, batches 1..5 replayed, twice
    torch.cuda.synchronize()
    assert int(m._smp.step.item()) == 2 + 12
    assert np.array_equal(m._smp.ids.cpu().numpy(), _draws(M, 14))
    # the replayed fit trains what eager steps train
    e = _model(dev, 32, 16, True, sampledNegatives=M)
    for _ in range(2):
        for b in batches:
            e.train_step(b)
    g = _model(dev, 32, 16, True, sampledNegatives=M)
    g.fit(batches, epochs=2, graph=True)
    for ta, tb in ((e.userTower.emb, g.userTower.emb), (e.itemTower.emb, g.itemTower.emb), (e.itemTower.dense, g.itemTower.dense)):
        assert (ta.w - tb.w).abs().max().item() <= 1e-3


CASES = [  # B, M, E, S, tensor cores, BRK_TT_NO_FUSED, options, one launch expected
    (1, 1, 32, 16, True, False, {}, True),
    (7, 127, 20, 12, True, False, {}, True),
    (7, 1000, 32, 16, True, True, {}, False),
    (7, 1000, 32, 16, True, False, dict(weightKey="w"), True),
    (200, 128, 32, 16, True, True, dict(temperature=0.5, weightKey="w"), False),
    (200, 129, 32, 16, True, False, dict(temperature=0.5, weightKey="w"), True),
    (200, 129, 20, 12, False, False, {}, False),
    (1000, 1000, 128, 128, True, False, dict(temperature=0.2), True),
    (1000, 129, 128, 128, False, False, dict(weightKey="w"), False),
    (1000, 128, 32, 16, True, True, dict(temperature=2.0, weightKey="w"), False),
    (1536, 1000, 32, 16, True, False, {}, False),        # 12 x 20 score tiles: beyond the SM count, multi-kernel step
]


@pytest.mark.parametrize("B,M,E,S,tc,no_fused,kw,one_launch", CASES)
def test_training_matches_the_oracle(dev, monkeypatch, B, M, E, S, tc, no_fused, kw, one_launch):
    """Three training steps (step + Adagrad in one call: the one launch where max(T Tc, 2 (T + Tc)) <= SM count on the
    tensor cores, else the multi-kernel step): the draws bit for bit, every loss, then weights and Adagrad accumulators;
    rows that occur only as sampled negatives move, with the oracle's accumulators."""
    if no_fused:
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    tr = _Trace(dev, monkeypatch)
    m = _model(dev, E, S, tc, sampledNegatives=M, **kw)
    tau = kw.get("temperature")
    o = _oracle(m, E, S, tc, tau)
    w0 = {k: v.detach().numpy().copy() for k, v in o.t.items()}
    ei0 = w0["Ei"]
    rng = np.random.default_rng(B + M + E)
    batch_rows, sampled_rows = set(), set()
    for t in range(1, 4):
        u, i = _ids(rng, B)
        w = rng.uniform(0.0, 2.0, B).astype(np.float32) if "weightKey" in kw else None
        ex = (None, torch.from_numpy(w).to(dev)) if w is not None else None
        with tr:
            loss = m._train_ids(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev), None, extras=ex).item()
        smp = _draws(M, t)
        assert np.array_equal(m._smp.ids.cpu().numpy(), smp)
        lref = o.step(u, i, cand_ids=i, sample_weight=w, sampled=smp)
        np.testing.assert_allclose(loss, lref, rtol=2e-3)
        batch_rows |= set(i.tolist()); sampled_rows |= set(smp.tolist())
    assert tr.stamped() == one_launch, "the step did not take the expected path"
    # trained state: the difference is held to a share of how far training moved each tensor.  On the tensor cores that is
    # the Frobenius bound of test_gpu_twotower_retrieval.py's gradients (1e-2); single entries are held there by
    # test_gradients_match_the_oracle, not after Adagrad, which divides each entry by the square root of its own
    # accumulator and so passes an entry's TF32 error on unevenly.  fp32: both bounds, 3e-3 and 1e-3.
    mx_share, fro_share = (None, 1e-2) if tc else (3e-3, 1e-3)

    def close(got, want, init, name):
        moved, diff = want - init, got - want
        mx = float(np.abs(diff).max()) / max(float(np.abs(moved).max()), 1e-20)
        fro = float(np.linalg.norm(diff)) / max(float(np.linalg.norm(moved)), 1e-20)
        print(f"{name}: max {mx:.2e} fro {fro:.2e} of the movement")
        assert (mx_share is None or mx <= mx_share) and fro <= fro_share, (name, mx, fro)
    for name, tab in (("Eu", m.userTower.emb), ("Ei", m.itemTower.emb)):
        close(tab.w.cpu().numpy(), o.t[name].detach().numpy(), w0[name], name)
        close(tab.m.cpu().numpy(), o.acc[name].numpy(), np.float32(0.1), name + " accumulator")
    for tw, wn in ((m.userTower, "Wu"), (m.itemTower, "Wi")):
        close(tw.dense.w.view(-1)[:E * S].view(E, S).cpu().numpy(), o.t[wn].detach().numpy(), w0[wn], wn)
    only = np.array(sorted(sampled_rows - batch_rows), dtype=np.int64)
    if len(only):
        ei = m.itemTower.emb.w.cpu().numpy()
        assert (np.abs(ei[only] - ei0[only]).max(axis=1) > 0).all(), "a row drawn only as a negative did not move"
        close(m.itemTower.emb.m.cpu().numpy()[only], o.acc["Ei"].numpy()[only], np.float32(0.1), "sampled-only rows' accumulators")
        assert (m.itemTower.emb.m.cpu().numpy()[only].max(axis=1) > np.float32(0.1)).all()


@pytest.mark.parametrize("B,M,E,S,tc,no_fused,tau", [(1000, 1000, 128, 128, True, False, 0.2),
                                                      (1000, 1000, 128, 128, True, True, 0.2),
                                                      (1000, 129, 128, 128, True, False, 0.2),
                                                      (200, 1000, 32, 16, False, False, 0.2)])
def test_gradients_match_the_oracle(dev, monkeypatch, B, M, E, S, tc, no_fused, tau):
    """One step's loss and gradients with the tolerances of test_gpu_twotower_retrieval.py (loss rtol 2e-3; every gradient
    within 1e-2 of its largest entry, max and Frobenius) at a low temperature, where TF32 rounding of the logits is
    amplified most.  The first two cases are the one launch and the multi-kernel step at the same shape."""
    if no_fused:
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    m = _model(dev, E, S, tc, sampledNegatives=M, temperature=tau, weightKey="w")
    o = _oracle(m, E, S, tc, tau)
    rng = np.random.default_rng(B + M)
    u, i = _ids(rng, B)
    w = rng.uniform(0.0, 2.0, B).astype(np.float32)
    loss = m._step(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev), None, True,
                   extras=(None, torch.from_numpy(w).to(dev))).item()
    lref = o.loss_and_grads(u, i, cand_ids=i, sample_weight=w, sampled=_draws(M, 1))
    np.testing.assert_allclose(loss, float(lref), rtol=2e-3)
    grads = [m.userTower.emb.g, m.itemTower.emb.g, m.userTower.dense.g.view(-1)[:E * S].view(E, S),
             m.itemTower.dense.g.view(-1)[:E * S].view(E, S), m.userTower.dense.g.view(-1)[E * S:E * S + S]]
    for got, name in zip(grads, ("Eu", "Ei", "Wu", "Wi", "bu")):
        g0, g1 = o.t[name].grad.numpy(), got.cpu().numpy()
        scale = max(float(np.abs(g0).max()), 1e-20)
        mx = float(np.abs(g1 - g0).max()) / scale
        fro = float(np.linalg.norm(g1 - g0) / max(np.linalg.norm(g0), 1e-20))
        assert mx <= 1e-2 and fro <= 1e-2, (name, mx, fro)


@pytest.mark.parametrize("B,M", [(1000, 1000), (200, 128)])   # n = B + M a multiple of 4: TF32 products on both paths
def test_one_launch_equals_the_multi_kernel_step(dev, monkeypatch, B, M):
    """The same sampled step as one launch (fused_step<false, true, true>) and as the multi-kernel step
    (BRK_TT_NO_FUSED=1): loss rtol 1e-5, gradients within 5e-4 of the largest entry (the tolerances of
    test_gpu_twotower_retrieval.py's one-launch / multi-kernel comparison)."""
    out = {}
    for path in ("fused", "multi"):
        if path == "multi":
            monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
        tr = _Trace(dev, monkeypatch)
        m = _model(dev, 128, 128, True, sampledNegatives=M, temperature=0.5, weightKey="w")
        rng = np.random.default_rng(3)
        u, i = _ids(rng, B)
        w = torch.from_numpy(rng.uniform(0.0, 2.0, B).astype(np.float32)).to(dev)
        with tr:
            loss = m._step(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev), None, True, extras=(None, w)).item()
        assert tr.stamped() == (path == "fused")
        out[path] = (loss, [m.userTower.emb.g.clone(), m.itemTower.emb.g.clone(), m.userTower.dense.g.clone(),
                            m.itemTower.dense.g.clone()])
    np.testing.assert_allclose(out["fused"][0], out["multi"][0], rtol=1e-5)
    for a, b in zip(out["fused"][1], out["multi"][1]):
        assert (a - b).abs().max().item() <= 5e-4 * b.abs().max().item()


def test_accidental_hits_mask_sampled_copies_of_the_positive(dev):
    """Three-item catalog: most sampled columns are copies of some row's positive; loss and gradients against the oracle,
    and the loss differs from the unmasked one."""
    nI, B, M, E, S = 3, 7, 16, 32, 16
    m = _model(dev, E, S, False, nI=nI, sampledNegatives=M)
    o = _oracle(m, E, S, False, nI=nI)
    u, i = _ids(np.random.default_rng(5), B, nI=nI)
    loss = m._step(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev), None, True).item()
    smp = _draws(M, 1, nI=nI)
    assert np.array_equal(m._smp.ids.cpu().numpy(), smp) and set(smp.tolist()) <= {2, 3, 4}
    assert any(int(s) in set(i.tolist()) for s in smp)
    lref = o.loss_and_grads(u, i, cand_ids=i, sampled=smp)
    np.testing.assert_allclose(loss, float(lref), rtol=1e-5)
    unmasked = o.loss(u, i, cand_ids=None, sampled=smp)
    assert abs(float(unmasked) - float(lref)) > 1e-3 * abs(float(lref))
    for got, name in ((m.userTower.emb.g, "Eu"), (m.itemTower.emb.g, "Ei")):
        np.testing.assert_allclose(got.cpu().numpy(), o.t[name].grad.numpy(), rtol=1e-4, atol=1e-6, err_msg=name)


def test_without_the_option_nothing_is_drawn(dev):
    """A model without sampledNegatives keeps the parent's step: its workspace has no extra rows and a sampled model's
    evaluation loss is the option-free in-batch loss."""
    a = _model(dev, 32, 16, True)
    b = _model(dev, 32, 16, True, sampledNegatives=50)
    assert a._smp is None and a.sampledNegatives == 0
    a._workspace(100); b._workspace(100)
    assert a._bufs["scores"].shape == (100, 100) and b._bufs["scores"].shape == (100, 150)
    u, i = _ids(np.random.default_rng(8), 100)
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    np.testing.assert_allclose(a._step(ud, idd, None, False).item(), b._step(ud, idd, None, False).item(), rtol=1e-6)
    torch.cuda.synchronize()
    assert int(b._smp.step.item()) == 0


def _pair(dev, E, S, G, tc, M, **kw):
    from binrec_b200.sharded import ShardedTwoTowerNet
    ref = _model(dev, E, S, tc, sampledNegatives=M, **kw)
    init = {"user": ref.userTower.emb.w.cpu().numpy(), "item": ref.itemTower.emb.w.cpu().numpy(),
            "user_dense": ref.userTower.dense.w.cpu().numpy(), "item_dense": ref.itemTower.dense.w.cpu().numpy()}
    opts = {k: v for k, v in kw.items() if k == "temperature"}
    sh = ShardedTwoTowerNet(U, I, E, S, learning_rate=0.1, tensor_cores=tc, device=dev, emulate=G, full_init=init,
                            seed=SEED, sampledNegatives=M, **opts)
    sh.init = {k: v.copy() for k, v in init.items()}
    return ref, sh


def _compare_state(ref, sh, share):
    def close(got, want, init, name):
        moved = float(np.abs(want - init).max())
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=max(share * moved, 2e-6), err_msg=name)
    pairs = (("user", sh.user, ref.userTower), ("item", sh.item, ref.itemTower))
    for name, t, tw in pairs:
        close(t.full_weights(), tw.emb.w.cpu().numpy(), sh.init[name], name)
        close(t.full_weights("m"), tw.emb.m.cpu().numpy(), np.float32(0.1), name + " accumulator")
    for (name, _, tw), d in zip(pairs, sh.dense):
        close(d.w.cpu().numpy(), tw.dense.w.cpu().numpy(), sh.init[name + "_dense"].reshape(1, -1), name + " Dense")


@pytest.mark.parametrize("path", ["tc", "no_fused", "fp32"])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_emulated_shards_equal_unsharded_model(dev, monkeypatch, G, path):
    if path == "no_fused":
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    tc = path != "fp32"
    E, S, B, M = 32, 16, 500, 129
    ref, sh = _pair(dev, E, S, G, tc, M, temperature=0.5, weightKey="w")
    rng = np.random.default_rng(10 * G)
    tr = _Trace(dev, monkeypatch)
    for step in range(3):
        u, i = _ids(rng, B)
        ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
        w = torch.from_numpy(rng.uniform(0.0, 2.0, B).astype(np.float32)).to(dev)
        l0 = ref._train_ids(ud, idd, None, extras=(None, w)).item()
        with tr:
            l1 = sh.train_on_batch(ud, idd, weights=w).item()
        np.testing.assert_allclose(l1, l0, **LOSS_TOL)
        assert torch.equal(sh._smp.ids, ref._smp.ids)
    assert int(sh._smp.step.item()) == 3
    assert tr.stamped() == (path == "tc"), "the sharded step did not take the expected path"   # fused_step<true, true, true>
    _compare_state(ref, sh, MOVED_SHARE[tc])


def test_checkpoint_keeps_the_sampler_counter(dev, tmp_path):
    from binrec_b200.sharded import ShardedTwoTowerNet
    E, S, M = 32, 16, 40
    a = ShardedTwoTowerNet(U, I, E, S, device=dev, emulate=3, sampledNegatives=M)
    rng = np.random.default_rng(4)
    for _ in range(2):
        u, i = _ids(rng, 64)
        a.train_on_batch(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev))
    a.save_checkpoint(str(tmp_path / "ck"))
    b = ShardedTwoTowerNet(U, I, E, S, device=dev, emulate=1, seed=5, sampledNegatives=M)
    b.load_checkpoint(str(tmp_path / "ck"))
    assert int(b._smp.step.item()) == 2
    u, i = _ids(rng, 64)
    b.train_on_batch(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev))
    torch.cuda.synchronize()
    assert np.array_equal(b._smp.ids.cpu().numpy(), _draws(M, 3, seed=5))
    plain = ShardedTwoTowerNet(U, I, E, S, device=dev, emulate=3)
    plain.save_checkpoint(str(tmp_path / "plain"))
    b.load_checkpoint(str(tmp_path / "plain"))
    assert int(b._smp.step.item()) == 0


def test_rejections(dev):
    from binrec_b200 import _native as N
    from binrec_b200.sharded import ShardedTwoTowerNet
    for bad in (0, -3, 1.5, True):
        with pytest.raises(ValueError, match="integer >= 1"):
            _model(dev, 32, 16, True, sampledNegatives=bad)
    for kw, msg in ((dict(rdZero=True, resKey="r"), "rdZero"), (dict(global_negatives=True), "global_negatives"),
                    (dict(streamingFrequency=0.1), "streamingFrequency"), (dict(candidateProbKey="p"), "candidate probabilities")):
        with pytest.raises(ValueError, match=msg):
            _model(dev, 32, 16, True, sampledNegatives=8, **kw)
    for kw, msg in ((dict(rdZero=True), "rdZero"), (dict(global_negatives=True), "global_negatives"),
                    (dict(streamingFrequency=True), "streamingFrequency")):
        with pytest.raises(ValueError, match=msg):
            ShardedTwoTowerNet(U, I, 32, 16, device=dev, emulate=2, sampledNegatives=8, **kw)
    sh = ShardedTwoTowerNet(U, I, 32, 16, device=dev, emulate=2, sampledNegatives=8)
    ones = torch.ones(10, dtype=torch.float32, device=dev)
    ids = torch.full((10,), 5, dtype=torch.int32, device=dev)
    with pytest.raises(ValueError, match="candidate probabilities"):
        sh.train_on_batch(ids, ids, cand_prob=ones)

    # C ABI: BRK_E_ARG with a message naming the limit; nothing is drawn
    m = _model(dev, 32, 16, True, sampledNegatives=8)
    lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()
    ws = m._workspace(10)
    ut, it = m.userTower.c_struct(), m.itemTower.c_struct()
    loss = torch.zeros(1, dtype=torch.float32, device=dev)

    def call(which="step", mode=0x100, batch=10, rt_over=None, **over):
        smp = m._smp.c_struct()
        for k, v in over.items():
            setattr(smp, k, v)
        if which == "sharded":
            rt = N.brk_tt_retrieval_sharded(); rt.inv_temperature = 1.0
        else:
            rt = N.brk_tt_retrieval(); rt.inv_temperature = 1.0
        for k, v in (rt_over or {}).items():
            setattr(rt, k, v)
        if which == "step":
            return lib.brk_twotower_step_sampled(ctx, C.byref(ut), C.byref(it), N.ptr(ids), N.ptr(ids), batch, mode, C.byref(ws),
                                                 N.ptr(loss), st, C.byref(smp), C.byref(rt))
        if which == "train":
            return lib.brk_twotower_train_step_sampled(ctx, C.byref(ut), C.byref(it), N.ptr(ids), N.ptr(ids), batch, mode,
                                                       C.byref(ws), 0.1, 1e-7, 1 << 40, N.ptr(loss), st, C.byref(smp),
                                                       C.byref(rt))
        shd = sh._shards()
        return lib.brk_twotower_step_sharded_sampled(ctx, C.byref(sh._towers()[0]), C.byref(sh._towers()[1]), C.byref(shd),
                                                     N.ptr(ids), N.ptr(ids), batch, mode, C.byref(ws), N.ptr(loss), st,
                                                     C.byref(smp), C.byref(rt))

    def rejected(rc, text):
        assert rc == -1, (rc, text)                        # BRK_E_ARG
        msg = lib.brk_last_error().decode()
        assert text in msg, (text, msg)

    est = N.brk_tt_estimator_sharded()
    for which in ("step", "train", "sharded"):
        rejected(call(which, count=0), "sampled count M = 0")
        rejected(call(which, lo=5, hi=5), "empty or outside")
        rejected(call(which, lo=-1), "empty or outside")
        rejected(call(which, hi=I + 3), "outside")
        rejected(call(which, step=None), "step counter")
        rejected(call(which, ids=None), "ids buffer")
        rejected(call(which, mode=0x101), "rdZero")
        rejected(call(which, rt_over=dict(cand_prob=ones.data_ptr())), "candidate probabilities")
        rejected(call(which, rt_over=dict(est=C.pointer(est)) if which == "sharded" else dict(last=ones.data_ptr())),
                 "streaming estimator")
        rejected(call(which, rt_over=dict(inv_temperature=0.0)), "temperature")
        rejected(call(which, batch=40000, count=60000), "2^31")
    rejected(call("step", rows=I + 5, hi=I + 5), "the item table has")
    rejected(lib.brk_twotower_step_sampled(ctx, C.byref(ut), C.byref(it), N.ptr(ids), N.ptr(ids), 10, 0x100, C.byref(ws),
                                           N.ptr(loss), st, None, None), "null sampled")
    torch.cuda.synchronize()
    assert int(m._smp.step.item()) == 0                   # nothing ran
    assert call("step") == 0
    torch.cuda.synchronize()
    assert int(m._smp.step.item()) == 1


# ---- two GPUs ------------------------------------------------------------------------------------------
U2, I2, E2, S2, M2, TAU2 = 1001, 403, 32, 16, 96, 0.5


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _global_batches(world):
    rng = np.random.default_rng(41)
    return [(rng.integers(2, U2 + 2, world * 200).astype(np.int32), rng.integers(2, 60, world * 200).astype(np.int32),
             rng.uniform(0.0, 2.0, world * 200).astype(np.float32)) for _ in range(3)]


def _worker(rank, world, port, init, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", device_id=dev)
    try:
        from binrec_b200.sharded import ShardedTwoTowerNet
        from binrec_b200.twoTower import TwoTowerModel
        out = {}
        net = ShardedTwoTowerNet(U2, I2, E2, S2, device=dev, full_init=init, temperature=TAU2, sampledNegatives=M2)
        mir = TwoTowerModel(E2, I2, U2, "u", "i", list(range(U2)), list(range(I2)), semb=S2, device=dev, tensor_cores=True,
                            temperature=TAU2, weightKey="w", sampledNegatives=M2)
        mir.compile("Adagrad", learningRate=0.1)
        with torch.no_grad():
            mir.userTower.emb.w.copy_(torch.from_numpy(init["user"])); mir.itemTower.emb.w.copy_(torch.from_numpy(init["item"]))
            mir.userTower.dense.w.view(-1).copy_(torch.from_numpy(init["user_dense"]))
            mir.itemTower.dense.w.view(-1).copy_(torch.from_numpy(init["item_dense"]))
        for name, model in (("sharded", net), ("mirrored", mir)):
            losses = []
            for u, i, w in _global_batches(world):
                lo, hi = rank * 200, (rank + 1) * 200
                t = lambda x: torch.from_numpy(x[lo:hi]).to(dev)
                if name == "sharded":
                    losses.append(float(net.train_on_batch(t(u), t(i), weights=t(w)).item()))
                else:
                    losses.append(float(mir._train_ids(t(u), t(i), None, extras=(None, t(w))).item()))
            if name == "sharded":
                net.check()
                out[name] = dict(losses=losses, Eu=net.user.full_weights(), Ei=net.item.full_weights())
            else:
                out[name] = dict(losses=losses, Eu=mir.userTower.emb.w.cpu().numpy(), Ei=mir.itemTower.emb.w.cpu().numpy())
            out[name]["ids"] = (net._smp if name == "sharded" else mir._smp).ids.cpu().numpy()
        ret[rank] = out
    except Exception as e:                                 # pragma: no cover - reported by the parent
        ret[rank] = repr(e)
    finally:
        dist.destroy_process_group()


def test_two_gpus_match_the_oracle_with_replica_keyed_draws():
    """Both models on 2 GPUs against one oracle step per global batch: each replica's slice scored against its own draws
    (Philox keyed by its rank), temperature and weights, Adagrad on the summed gradients."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import tf32
    from oracle import twotower_sampled as OS
    world = 2
    o0 = OS.SampledOracle(U2, I2, E2, S2, seed=42, temperature=TAU2, matmul=tf32.matmul)
    init = {"user": o0.t["Eu"].detach().numpy().copy(), "item": o0.t["Ei"].detach().numpy().copy()}
    for k, (wn, bn) in enumerate((("Wu", "bu"), ("Wi", "bi"))):
        flat = np.concatenate([o0.t[wn].detach().numpy().reshape(-1), o0.t[bn].detach().numpy()])
        init[("user_dense", "item_dense")[k]] = np.pad(flat, (0, (-len(flat)) % 4))
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, init, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
    for r in range(world):
        assert r in ret and not isinstance(ret[r], str), ret.get(r)
    o = OS.SampledOracle(U2, I2, E2, S2, seed=42, temperature=TAU2, matmul=tf32.matmul)
    with torch.no_grad():
        for k in o.t:
            o.t[k].copy_(o0.t[k])
    ref_losses = []
    for t, (u, i, w) in enumerate(_global_batches(world), start=1):
        for v in o.t.values():
            v.grad = None
        parts = [o.loss(u[r * 200:(r + 1) * 200], i[r * 200:(r + 1) * 200], cand_ids=i[r * 200:(r + 1) * 200],
                        sample_weight=w[r * 200:(r + 1) * 200], sampled=OS.sampled_negatives(M2, 42, t, r, 2, I2 + 2))
                 for r in range(world)]
        sum(parts).backward()
        ref_losses.append([float(p) for p in parts])
        with torch.no_grad():
            for k, v in o.t.items():
                g = v.grad if v.grad is not None else torch.zeros_like(v)
                o.acc[k] += g * g
                v -= o.lr * g / (o.acc[k].sqrt() + 1e-7)
    for name in ("sharded", "mirrored"):
        for r in range(world):
            got = ret[r][name]
            assert np.array_equal(got["ids"], OS.sampled_negatives(M2, 42, 3, r, 2, I2 + 2))
            np.testing.assert_allclose(got["losses"], [ls[r] for ls in ref_losses], rtol=2e-3, atol=1e-6)
            np.testing.assert_allclose(got["Eu"], o.t["Eu"].detach().numpy(), **W_TOL)
            np.testing.assert_allclose(got["Ei"], o.t["Ei"].detach().numpy(), **W_TOL)
