"""Size-independent properties at BASELINE.json's full sizes (where the CPU oracle would take minutes to hours):
adjointness / linearity of gather and scatter-add on a 20M x 64 table, sortedness + self-consistency of the
full-catalog top-K at one 8-way item shard of configs[4], "a BPR negative is never a positive" over a whole
ML-1M epoch, lazy Adam touching exactly the rows of the batch, and edge cases (batch of one, every sample hitting
one row, users with every / no item interacted)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def H():
    from binrec_b200 import hotpath
    return hotpath


def test_gather_scatter_adjoint_on_20m_rows(dev):
    # <gather(T, ids), V> == <T, scatter_add(ids, V)> with small-integer values: exact in fp32 -> bit-exact equality
    rows, d, n = 20_000_000, 64, 4_000_000
    g = torch.Generator(device=dev); g.manual_seed(1)
    T = torch.randint(-4, 5, (rows, d), generator=g, device=dev, dtype=torch.int8).float()
    V = torch.randint(-4, 5, (n, d), generator=g, device=dev, dtype=torch.int8).float()
    ids = (rows * torch.rand(n, generator=g, device=dev) ** 2).to(torch.int32).clamp_(0, rows - 1)   # skewed: duplicates
    out = H().gather_rows(T, ids)
    lhs = (out.double() * V.double()).sum()
    acc = torch.zeros(rows, d, device=dev)
    touched = torch.zeros((rows + 31) // 32, dtype=torch.int32, device=dev)
    H().scatter_add_rows(acc, ids, V, touched)
    rhs = (T.double() * acc.double()).sum()
    assert lhs.item() == rhs.item()
    # touched bits == exactly the distinct ids
    bits = torch.zeros(rows, dtype=torch.bool, device=dev); bits[ids.long()] = True
    words = touched.view(torch.int32)
    got = ((words[:, None] >> torch.arange(32, device=dev, dtype=torch.int32)[None, :]) & 1).bool().view(-1)[:rows]
    assert torch.equal(got, bits)


def test_full_catalog_topk_properties_at_shard_size(dev):
    U, I, d, k = 16384, 250_000, 64, 10
    g = torch.Generator(device=dev); g.manual_seed(2)
    Q = torch.randn(U, d, generator=g, device=dev); C = torch.randn(I, d, generator=g, device=dev)
    idx = H().BruteForceIndex(k).index(C)
    vals, ids = idx(Q)
    assert vals.shape == (U, k) and ids.shape == (U, k)
    assert bool((vals[:, :-1] >= vals[:, 1:]).all())                        # sorted descending
    assert bool((ids >= 0).all()) and bool((ids < I).all())
    srt = ids.sort(dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all())                          # no item twice
    # the returned scores are the bf16-operand scores of the returned ids (fp32 accumulation)
    qb, cb = Q.bfloat16().float(), C.bfloat16().float()
    resc = (qb[:, None, :] * cb[ids.long()]).sum(-1)
    torch.testing.assert_close(vals, resc, rtol=1e-5, atol=1e-4)
    # nothing outside the list beats its k-th score (checked exactly on 256 rows)
    rows = torch.arange(0, U, U // 256, device=dev)
    full = qb[rows] @ cb.T
    kth = torch.topk(full, k, dim=1).values[:, -1]
    torch.testing.assert_close(vals[rows, -1], kth, rtol=1e-5, atol=1e-4)
    # idempotence: a second call returns the same lists
    v2, i2 = idx(Q)
    assert torch.equal(ids, i2) and torch.equal(vals, v2)


def test_bpr_negatives_never_positive_over_a_full_epoch(dev):
    from binrec_b200 import synth
    users, items = synth.make_interactions()
    U, I = synth.ML1M_USERS, synth.ML1M_ITEMS
    indptr, sitems = synth.build_csr(users, items, U)
    ud = torch.from_numpy(users).to(dev)
    neg = H().philox_bpr_negatives(ud, 7, 3, I, torch.from_numpy(indptr).to(dev), torch.from_numpy(sitems).to(dev))
    assert bool((neg >= 0).all()) and bool((neg < I).all())
    pos_keys = torch.from_numpy(np.unique(users.astype(np.int64) * I + items)).to(dev)
    q = ud.long() * I + neg.long()
    pos = torch.searchsorted(pos_keys, q).clamp_(max=pos_keys.numel() - 1)
    assert not bool((pos_keys[pos] == q).any())
    # the stream is a function of (seed, epoch, sample index): any slice regenerates identically
    part = H().philox_bpr_negatives(ud[500_000:500_100].contiguous(), 7, 3, I, torch.from_numpy(indptr).to(dev),
                                    torch.from_numpy(sitems).to(dev), first_index=500_000)
    assert torch.equal(part, neg[500_000:500_100])


def test_sampler_edge_users_all_or_no_items(dev):
    from oracle import philox as OP
    I = 37
    pu = np.concatenate([np.zeros(I, np.int32), np.array([2, 2], np.int32)])          # user 0: everything; user 1: nothing
    pi = np.concatenate([np.arange(I, dtype=np.int32), np.array([5, 9], np.int32)])
    indptr, sitems = OP.build_csr(pu, pi, 3)
    q = np.array([0, 1, 2, 1, 0, 2] * 50, dtype=np.int32)
    ref = OP.bpr_negatives(q, 3, 1, I, indptr, sitems, first_index=11)
    got = H().philox_bpr_negatives(torch.from_numpy(q).to(dev), 3, 1, I, torch.from_numpy(indptr).to(dev),
                                   torch.from_numpy(sitems).to(dev), first_index=11)
    assert np.array_equal(got.cpu().numpy(), ref)
    assert not np.isin(ref[q == 2], [5, 9]).any()


def test_bpr_batch_of_one_and_all_samples_on_one_row(dev):
    from oracle import bpr as OB
    U, I, d = 50, 40, 64
    for u, p, n in ((np.array([3], np.int32), np.array([7], np.int32), np.array([9], np.int32)),
                    (np.full(4096, 5, np.int32), np.full(4096, 6, np.int32), np.full(4096, 7, np.int32))):
        orc = OB.BPROracle(U, I, d, seed=42)
        user = H().Table(torch.from_numpy(orc.user.copy()).to(dev)); item = H().Table(torch.from_numpy(orc.item.copy()).to(dev))
        opt = H().Adam(1e-3, device=dev)
        loss = H().bpr_fwd_bwd(user, item, *(torch.from_numpy(x).to(dev) for x in (u, p, n)))
        opt.apply([user, item])
        ref = orc.step(u, p, n)
        np.testing.assert_allclose(loss.item(), ref, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(user.w.cpu().numpy(), orc.user, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(item.w.cpu().numpy(), orc.item, rtol=1e-5, atol=1e-6)


def test_lazy_adam_moves_exactly_the_batch_rows_on_a_large_table(dev):
    rows, d, n = 2_000_000, 64, 65_536
    g = torch.Generator(device=dev); g.manual_seed(3)
    tab = H().Table(torch.empty(rows, d, device=dev).uniform_(-0.05, 0.05, generator=g))
    w0 = tab.w.clone()
    ids = torch.randint(0, rows, (n,), generator=g, device=dev, dtype=torch.int32)
    H().scatter_add_rows(tab.g, ids, torch.ones(n, d, device=dev), tab.touched)
    opt = H().Adam(1e-3, sparse="lazy", device=dev)
    opt.apply([tab])
    moved = (tab.w != w0).any(dim=1)
    hit = torch.zeros(rows, dtype=torch.bool, device=dev); hit[ids.long()] = True
    assert torch.equal(moved, hit)
    assert int(tab.touched.abs().sum().item()) == 0 and float(tab.g.abs().sum().item()) == 0.0
    # first Adam step with g > 0: every coordinate of a hit row moves by -lr (up to rounding)
    step = (tab.w - w0)[hit]
    torch.testing.assert_close(step, torch.full_like(step, -1e-3), rtol=1e-3, atol=1e-7)


def test_bpr_twenty_bench_identical_steps_match_the_oracle(dev):
    """BASELINE.json configs[1] exactly as bench.py runs it: 6040 x 3706, d = 64, batch 16 384, the bench frame, Philox
    negatives (seed 7, epoch 0), twenty Keras-Adam steps from the seeded initial tables -- per-step loss and final tables
    against oracle/bpr.py (fp32: loss rtol 1e-5; tables rtol 1e-4 / atol 2e-5 after 20 Adam steps)."""
    from binrec_b200 import synth
    from binrec_b200.BPRModel import BPRNet
    from oracle import bpr as OB, philox as OP
    users, items = synth.make_interactions()
    U, I, d, B, K = synth.ML1M_USERS, synth.ML1M_ITEMS, 64, 16384, 20
    net = BPRNet(U, I, d, seed=42, learning_rate=1e-3, sparse_adam="keras", device=dev)
    net.set_training_pairs(users, items)
    net.sample_negatives(7, 0)
    losses = net.train_steps(list(range(K)), B).cpu().numpy()
    orc = OB.BPROracle(U, I, d, seed=42)
    indptr, sitems = OP.build_csr(users, items, U)
    neg = OP.bpr_negatives(users[:K * B], 7, 0, I, indptr, sitems)
    assert np.array_equal(net._pairs["n"][:K * B].cpu().numpy(), neg)            # sampled indices: bit-exact
    ref = [orc.step(users[b * B:(b + 1) * B], items[b * B:(b + 1) * B], neg[b * B:(b + 1) * B]) for b in range(K)]
    np.testing.assert_allclose(losses, np.asarray(ref, dtype=np.float32), rtol=1e-5)
    np.testing.assert_allclose(net.user.w.cpu().numpy(), orc.user, rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(net.item.w.cpu().numpy(), orc.item, rtol=1e-4, atol=2e-5)


def test_bench_dump_outputs_hold_the_last_timed_step(dev, tmp_path):
    """bench.py --steps K --warmup W --dump-outputs DIR: K timed steps, and the dumped loss and tables are those after the
    W + K steps over batches 0 .. W + K - 1 of the bench frame, against oracle/bpr.py (tolerances of the test above)."""
    import json
    import os
    import subprocess
    import sys
    from binrec_b200 import synth
    from oracle import bpr as OB, philox as OP
    W, K = 3, 2
    bench = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")
    r = subprocess.run([sys.executable, bench, "--steps", str(K), "--warmup", str(W), "--no-extras", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == K
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("loss", "user_embedding", "item_embedding")}
    assert all(a.dtype == np.float32 for a in got.values())
    users, items = synth.make_interactions()
    U, I, d, B = synth.ML1M_USERS, synth.ML1M_ITEMS, 64, 16384
    orc = OB.BPROracle(U, I, d, seed=42)
    indptr, sitems = OP.build_csr(users, items, U)
    neg = OP.bpr_negatives(users[:(W + K) * B], 7, 0, I, indptr, sitems)
    ref = [orc.step(users[b * B:(b + 1) * B], items[b * B:(b + 1) * B], neg[b * B:(b + 1) * B]) for b in range(W + K)]
    np.testing.assert_allclose(got["loss"], np.float32(ref[-1]).reshape(1), rtol=1e-5)
    np.testing.assert_allclose(got["user_embedding"], orc.user, rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(got["item_embedding"], orc.item, rtol=1e-4, atol=2e-5)


def test_twotower_three_steps_at_baseline_shape_match_the_oracle(dev):
    """BASELINE.json configs[2] shape: 6040 x 3706, E = S = 128, in-batch softmax batch 1000, Adagrad 0.1 -- three fp32 steps."""
    from binrec_b200.twoTower import TwoTowerModel
    from oracle import twotower as OT
    U, I, E, S, B = 6040, 3706, 128, 128, 1000
    m = TwoTowerModel(E, I, U, "u", "i", list(range(U)), list(range(I)), semb=S, device=dev)
    m.compile("Adagrad", learningRate=0.1)
    o = OT.TwoTowerOracle(U, I, E, S, seed=42)
    with torch.no_grad():
        o.t["Eu"].copy_(m.userTower.emb.w.cpu()); o.t["Ei"].copy_(m.itemTower.emb.w.cpu())
        for tw, wn, bn in ((m.userTower, "Wu", "bu"), (m.itemTower, "Wi", "bi")):
            flat = tw.dense.w.view(-1).cpu()
            o.t[wn].copy_(flat[:E * S].view(E, S)); o.t[bn].copy_(flat[E * S:E * S + S])
    rng = np.random.default_rng(0)
    for step in range(3):
        u = rng.integers(2, U + 2, B).astype(np.int32); i = rng.integers(2, I + 2, B).astype(np.int32)
        lref = o.step(u, i, cand_ids=i)
        lgot = m._step(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev), None, True)
        m.optimizer.apply([m.userTower.emb, m.itemTower.emb], dense=[m.userTower.dense, m.itemTower.dense])
        np.testing.assert_allclose(lgot.item(), lref, rtol=1e-5)
    np.testing.assert_allclose(m.userTower.emb.w.cpu().numpy(), o.t["Eu"].detach().numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(m.itemTower.emb.w.cpu().numpy(), o.t["Ei"].detach().numpy(), rtol=1e-4, atol=1e-5)
