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
    rows, d, n = ROWS_SCAN, 64, 65_536
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


# ---- values of the row-sparse optimizers (csrc/optim.cu rows_pass) where its bitmask scan merges slots ---------------
# rows_pass gives each warp up to 32 bitmask words per slot, taken `stride` words apart; a warp owns several slots only
# when the table has more than 32 words per warp of the grid (SMs x 2 CTAs x 8 warps: ~2.4 M rows on a B200).  There it
# prefetches the next slot's words, carries a partial row list (< gpw * 4 rows) into the next slot and flushes on its
# last slot.  6 000 017 rows is past that even at 4 CTAs per SM, and its last bitmask word holds 17 rows.
ROWS_SCAN = 6_000_017


def _pattern(name, rows, gen, dev):
    n = 65_536
    if name == "uniform":                  # sparse slots: their rows are carried into the next slot's list
        return torch.randint(0, rows, (n,), generator=gen, device=dev, dtype=torch.int32)
    if name == "cubic":                    # a crowded neighbourhood that the stride layout spreads over many warps
        return (rows * torch.rand(n, generator=gen, device=dev, dtype=torch.float64) ** 3).to(torch.int32).clamp_(max=rows - 1)
    if name == "all":                      # every slot flushes full 1024-row lists
        return torch.arange(rows, device=dev, dtype=torch.int32)
    if name == "last":                     # the partial last word alone
        return torch.full((1,), rows - 1, device=dev, dtype=torch.int32)
    if name == "uniform+last":
        return torch.cat([_pattern("uniform", rows, gen, dev), _pattern("last", rows, gen, dev)])
    raise ValueError(name)


def _prepare(tab, ids, gen):
    """Random-normal gradients scattered into the accumulator (duplicates summed, rows marked), then the touched rows'
    w / m / v / g gathered to the host in float64 and device copies of the slots, for the untouched rows."""
    H().scatter_add_rows(tab.g, ids, torch.randn(ids.numel(), tab.d, generator=gen, device=tab.w.device), tab.touched)
    rows = torch.unique(ids.long())
    slots = [k for k in "wmv" if getattr(tab, k) is not None]
    host = {k: getattr(tab, k)[rows].double().cpu().numpy() for k in slots + ["g"]}
    return rows, host, {k: getattr(tab, k).clone() for k in slots}


def _check_rows(tab, rows, want, before, tag):
    """Touched rows against the float64 reference, untouched rows bit-identical, accumulator and bitmask left zero."""
    untouched = torch.ones(tab.rows, dtype=torch.bool, device=tab.w.device)
    untouched[rows] = False
    for k in before:
        got = getattr(tab, k)[rows].double().cpu().numpy()
        print(f"{tag} {k}: touched rows {rows.numel()}, max |err| {np.abs(got - want[k]).max():.2e}")
        np.testing.assert_allclose(got, want[k], rtol=1e-5, atol=1e-6, err_msg=f"{tag} {k}")
        assert torch.equal(getattr(tab, k)[untouched], before[k][untouched]), (tag, k)
    assert not tab.g.any().item() and not tab.touched.any().item(), tag


# the hyper-parameters as the kernels hold them (float32, as Keras does): 1 - beta_2 is then 1 - 0.999f = 0.00099998713,
# 1.3e-5 away from 0.001 -- more than rtol 1e-5 wherever v is large
_F32 = lambda x: float(np.float32(x))                                    # noqa: E731
ADAM_HYPER = dict(lr=_F32(1e-3), beta1=_F32(0.9), beta2=_F32(0.999), eps=_F32(1e-7))
ADAGRAD_HYPER = dict(lr=_F32(0.1), eps=_F32(1e-7))


def _lazy_adam_step(opt, tabs, patterns, gen, t, tag):
    """One Adam.apply (one brk_adam_rows call over every table) against oracle/embedding.py adam_rows_lazy at step t."""
    from oracle import embedding as OE
    prep = [_prepare(tab, _pattern(p, tab.rows, gen, tab.w.device), gen) for tab, p in zip(tabs, patterns)]
    opt.apply(tabs)
    assert int(opt.state[0].item()) == t
    for tab, p, (rows, host, before) in zip(tabs, patterns, prep):
        OE.adam_rows_lazy(host["w"], host["m"], host["v"], host["g"], np.arange(rows.numel()), t, **ADAM_HYPER)
        _check_rows(tab, rows, host, before, f"{tag} d={tab.d} {p} t={t}")


@pytest.mark.parametrize("d,first,second", [(4, "all", "last"), (10, "uniform", "cubic"), (64, "cubic", "uniform+last")])
def test_row_sparse_optimizers_match_the_oracle_on_a_large_table(dev, d, first, second):
    """d = 4: one lane per row (float4), a list flushed once 128 rows are waiting; d = 10: the scalar path (rows not a
    multiple of 4 floats); d = 64: 16 lanes per row.  Two lazy-Adam steps (t = 1, 2) with different row sets, then one
    sparse Adagrad step on a fresh table.  Touched rows: w / m / v at rtol 1e-5 / atol 1e-6 of the float64 reference
    computed from the same float32 inputs; untouched rows bit-identical."""
    from oracle import embedding as OE
    gen = torch.Generator(device=dev); gen.manual_seed(d)
    tab = H().Table(torch.empty(ROWS_SCAN, d, device=dev).uniform_(-0.05, 0.05, generator=gen))
    opt = H().Adam(1e-3, sparse="lazy", device=dev)
    _lazy_adam_step(opt, [tab], [first], gen, 1, "lazy Adam")
    _lazy_adam_step(opt, [tab], [second], gen, 2, "lazy Adam")
    del tab, opt
    tab = H().Table(torch.empty(ROWS_SCAN, d, device=dev).uniform_(-0.05, 0.05, generator=gen), slots=1, slot_init=0.1)
    rows, host, before = _prepare(tab, _pattern(first, ROWS_SCAN, gen, dev), gen)
    H().Adagrad(0.1, rows_threshold_bytes=0).apply([tab])
    OE.adagrad_rows(host["w"], host["m"], host["g"], np.arange(rows.numel()), **ADAGRAD_HYPER)
    _check_rows(tab, rows, host, before, f"Adagrad d={d} {first}")


def test_lazy_adam_over_three_tables_of_different_widths_in_one_call(dev):
    """One brk_adam_rows call over three tables: the per-table state of the scan (row list, prefetch) restarts at every
    table.  100 003 x 256: 64 float4 chunks per row, more than a warp's 32 lanes (the chunk loop of the scalar path)."""
    gen = torch.Generator(device=dev); gen.manual_seed(17)
    tabs = [H().Table(torch.empty(r, d, device=dev).uniform_(-0.05, 0.05, generator=gen))
            for r, d in ((ROWS_SCAN, 4), (100_003, 256), (ROWS_SCAN, 64))]
    opt = H().Adam(1e-3, sparse="lazy", device=dev)
    _lazy_adam_step(opt, tabs, ["cubic", "uniform+last", "uniform"], gen, 1, "three tables")
    _lazy_adam_step(opt, tabs, ["uniform+last", "cubic", "last"], gen, 2, "three tables")


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
