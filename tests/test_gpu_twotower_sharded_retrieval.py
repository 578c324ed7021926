"""Sampling-bias-corrected softmax on row-sharded two-tower training (ShardedTwoTowerNet(temperature=,
streamingFrequency=), train_on_batch(cand_prob=, weights=); brk_tt_estimator_update_sharded and
brk_twotower_step_sharded_retrieval).

One GPU: `emulate=G` holds all G shards in one process and trains the whole batch as one replica, so the result must be
the unsharded TwoTowerModel's with the same options, and the estimator state must be bit-equal.  At the C ABI, G emulated
ranks with local shard buffers check the per-replica semantics against oracle/twotower_retrieval.py: every rank's update
of the global batch, then each slice's softmax.  Two GPUs: real peer memory and the cross-GPU barrier between the update
and the step."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U, I = 301, 203                                           # row counts (+2: StringLookup offset) not divisible by G
LOSS_TOL = dict(rtol=1e-5, atol=1e-6)
W_TOL = dict(rtol=1e-4, atol=2e-6)
# test_gpu_twotower_sharded.py: after several steps the weights are held to a share of how far training moved them
MOVED_SHARE = {True: 1e-2, False: 1e-3}
OPTIONS = {                                               # model options, per-call columns (p, w)
    "tau": (dict(temperature=0.5), False, False),
    "p_w": (dict(), True, True),
    "est": (dict(streamingFrequency=0.1), False, False),
    "est_tau_w": (dict(streamingFrequency=0.1, temperature=2.0), False, True),
}
PATHS = {                                                 # batch, tensor cores, BRK_TT_NO_FUSED, one launch
    "one_launch": (1000, True, False, True),
    "b2000": (2000, True, False, False),
    "no_fused": (1000, True, True, False),
    "fp32": (1000, False, False, False),
}


def _pair(dev, E, S, G, tensor_cores=True, **opts):
    from binrec_b200.sharded import ShardedTwoTowerNet
    from binrec_b200.twoTower import TwoTowerModel
    cols = dict(weightKey="w") if "streamingFrequency" in opts else dict(candidateProbKey="p", weightKey="w")
    ref = TwoTowerModel(E, I, U, "u", "i", list(range(U)), list(range(I)), semb=S, device=dev, tensor_cores=tensor_cores,
                        **cols, **opts)
    ref.compile("Adagrad", learningRate=0.1)
    init = {"user": ref.userTower.emb.w.cpu().numpy(), "item": ref.itemTower.emb.w.cpu().numpy(),
            "user_dense": ref.userTower.dense.w.cpu().numpy(), "item_dense": ref.itemTower.dense.w.cpu().numpy()}
    sh = ShardedTwoTowerNet(U, I, E, S, learning_rate=0.1, tensor_cores=tensor_cores, device=dev, emulate=G, full_init=init,
                            **opts)
    sh.init = {k: v.copy() for k, v in init.items()}
    return ref, sh


def _ids(rng, B):
    f = lambda n: rng.random(n) ** 2                      # skewed: popular rows repeat, accidental hits
    return (2 + (U * f(B))).astype(np.int32), (2 + (I * f(B))).astype(np.int32)


def _columns(rng, B, dev, p, w):
    prob = (rng.random(B) ** 4).astype(np.float32)
    prob[rng.integers(0, B, 5)] = 1e-9                    # below the 1e-6 clip
    wt = rng.uniform(0.0, 2.0, B).astype(np.float32)
    wt[rng.integers(0, B, 3)] = 0.0
    return (torch.from_numpy(prob).to(dev) if p else None), (torch.from_numpy(wt).to(dev) if w else None)


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
        close(d.m.cpu().numpy(), tw.dense.m.cpu().numpy(), np.float32(0.1), name + " Dense accumulator")


def _estimator_equal(ref, sh):
    last, gap, step = sh.estimator_state()
    assert np.array_equal(last, ref._freq["last"].cpu().numpy())
    assert np.array_equal(gap.view(np.int32), ref._freq["gap"].cpu().numpy().view(np.int32))
    assert step == int(ref._freq["step"].item())


class _Trace:
    """BRK_TT_TRACE pointed at a zeroed device buffer around the sharded call only."""

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


@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("opt", sorted(OPTIONS))
@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_emulated_shards_equal_unsharded_model_with_options(dev, monkeypatch, G, opt, path):
    B, tc, no_fused, one_launch = PATHS[path]
    kw, has_p, has_w = OPTIONS[opt]
    if no_fused:
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    E, S = 32, 16
    ref, sh = _pair(dev, E, S, G, tensor_cores=tc, **kw)
    rng = np.random.default_rng(100 * G + len(opt))
    tr = _Trace(dev, monkeypatch)
    for step in range(4):
        u, i = _ids(rng, B)
        ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
        p, w = _columns(rng, B, dev, has_p, has_w)
        l0 = ref._train_ids(ud, idd, None, extras=(p, w)).item()
        with tr:
            l1 = sh.train_on_batch(ud, idd, cand_prob=p, weights=w).item()
        np.testing.assert_allclose(l1, l0, **LOSS_TOL)
    assert tr.stamped() == one_launch, "the step did not take the expected path"
    _compare_state(ref, sh, MOVED_SHARE[tc])
    if "streamingFrequency" in kw:
        _estimator_equal(ref, sh)
        assert sh.estimator_state()[2] == 4


def _oracle_from(sh, E, S, tc, tau):
    from oracle import tf32
    from oracle import twotower_retrieval as OR
    o = OR.RetrievalOracle(U, I, E, S, seed=42, temperature=tau, matmul=tf32.matmul if tc else torch.matmul)
    with torch.no_grad():
        o.t["Eu"].copy_(torch.from_numpy(sh.user.full_weights())); o.t["Ei"].copy_(torch.from_numpy(sh.item.full_weights()))
        for d, wn, bn in zip(sh.dense, ("Wu", "Wi"), ("bu", "bi")):
            flat = d.w.view(-1).cpu()
            o.t[wn].copy_(flat[:E * S].view(E, S)); o.t[bn].copy_(flat[E * S:E * S + S])
    return o


@pytest.mark.parametrize("tc", [True, False])
def test_per_replica_softmax_over_the_global_estimator_at_the_c_abi(dev, tc):
    """G = 3 emulated ranks with local shard buffers, one step counter each: every rank's update in rank order, then each
    slice's step.  Against the oracle whose estimator is updated on the global batch and whose softmax is per slice:
    losses per slice, the summed gradients of the first step, the estimator state bit for bit and every counter.  Item 7
    sits in two slices of the same step, slice 0 repeats items, and slice 2 of the last step is empty."""
    from binrec_b200 import _native as N
    from oracle import twotower_retrieval as OR
    G, E, S, tau, alpha = 3, 32, 16, 0.5, 0.2
    _, sh = _pair(dev, E, S, G, tensor_cores=tc, temperature=tau, streamingFrequency=alpha)
    o = _oracle_from(sh, E, S, tc, tau)
    f = OR.StreamingFrequency(I + 2, alpha=alpha)
    lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()
    steps = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(G)]
    rng = np.random.default_rng(4)
    for k in range(3):
        sizes = [300, 250, 200] if k < 2 else [400, 300, 0]
        parts = []
        for r, n in enumerate(sizes):
            u = (2 + rng.integers(0, U, n)).astype(np.int32)
            i = (2 + rng.integers(0, 30 + 20 * r, n)).astype(np.int32)
            if n:
                i[: n // 3] = i[0]                        # duplicates inside one slice
                i[-1] = 7                                  # the same item in several slices
            parts.append((u, i))
        g_items = np.concatenate([i for _, i in parts])
        for r, (_, i) in enumerate(parts):
            est = N.brk_tt_estimator_sharded.from_buffer_copy(sh._est.c)
            est.rank = r
            idd = torch.from_numpy(i).to(dev)
            assert lib.brk_tt_estimator_update_sharded(ctx, C.byref(est), N.ptr(idd) if len(i) else None, len(i), alpha,
                                                       N.ptr(steps[r]), st) == 0, lib.brk_last_error()
        f.update(g_items)
        for t in (sh.user, sh.item):
            for r in range(G):
                t.tables[r].g.zero_(); t.tables[r].touched.zero_()
        for d in sh.dense:
            d.g.zero_()
        for v in o.t.values():
            v.grad = None
        total = 0
        for r, (u, i) in enumerate(parts):
            if not len(i):
                continue
            B = len(i)
            ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
            ws = sh._workspace(B)
            ut, it = sh._towers()
            shards = sh._shards()
            shards.user.rank = shards.item.rank = r
            est = N.brk_tt_estimator_sharded.from_buffer_copy(sh._est.c)
            est.rank = r
            rt = N.brk_tt_retrieval_sharded(None, None, C.pointer(est), 1.0 / tau)
            loss = torch.empty(1, dtype=torch.float32, device=dev)
            assert lib.brk_twotower_step_sharded_retrieval(ctx, C.byref(ut), C.byref(it), C.byref(shards), N.ptr(ud), N.ptr(idd),
                                                           N.ptr(idd), None, B, 0x100 if tc else 0, C.byref(ws), N.ptr(loss),
                                                           st, C.byref(rt)) == 0, lib.brk_last_error()
            lref = o.loss(u, i, cand_ids=i, cand_prob=f.probability(i))
            total = total + lref
            np.testing.assert_allclose(loss.item(), float(lref.detach()), rtol=2e-3 if tc else 1e-5)
        if k == 0:                                         # the summed per-replica gradients
            total.backward()
            for got, name in ((sh.item.full_weights("g"), "Ei"), (sh.user.full_weights("g"), "Eu")):
                g0 = o.t[name].grad.numpy()
                assert np.abs(got - g0).max() <= (1e-2 if tc else 1e-4) * np.abs(g0).max(), name
    last, gap, _ = sh.estimator_state()
    assert np.array_equal(last, f.last)
    assert np.array_equal(gap.view(np.int32), f.gap.view(np.int32))
    assert [int(s.item()) for s in steps] == [3, 3, 3]   # the empty slice's counter advanced too


@pytest.mark.parametrize("B", [1000, 2000])
def test_neutral_options_equal_the_option_free_sharded_step(dev, B):
    """tau = 1, p = 1, w = 1 against the option-free sharded step: loss rtol 1e-6; gradients within 1e-4 of the largest
    entry (the REDs sum in a different order from run to run, see test_gpu_twotower_retrieval.py)."""
    from binrec_b200.sharded import ShardedTwoTowerNet
    G, E, S = 3, 128, 128
    u, i = _ids(np.random.default_rng(7), B)
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    ones = torch.ones(B, dtype=torch.float32, device=dev)
    res = []
    for kw in ({}, dict(temperature=1.0)):
        net = ShardedTwoTowerNet(U, I, E, S, device=dev, emulate=G, seed=3, **kw)
        loss = net.forward_backward(ud, idd, cand_prob=ones if kw else None, weights=ones if kw else None).item()
        res.append((loss, [net.user.full_weights("g"), net.item.full_weights("g")] + [d.g.cpu().numpy() for d in net.dense]))
    np.testing.assert_allclose(res[1][0], res[0][0], rtol=1e-6)
    for a, b in zip(res[1][1], res[0][1]):
        assert np.abs(a - b).max() <= 1e-4 * np.abs(b).max()


@pytest.mark.parametrize("G_from,G_to", [(3, 0), (0, 3)])
def test_checkpoint_with_the_estimator_reshards(dev, tmp_path, G_from, G_to):
    """Saved at G_from (0: one unsharded process), resumed at G_to: the resumed run equals the uninterrupted one, the
    estimator state bit for bit.  A checkpoint without the estimator starts it from zero."""
    from binrec_b200.sharded import ShardedTwoTowerNet
    E, S, B = 32, 16, 500                                  # fp32 products: equal weights differ by RED order only
    kw = dict(learning_rate=0.1, tensor_cores=False, device=dev, temperature=0.5, streamingFrequency=0.2)
    a = ShardedTwoTowerNet(U, I, E, S, emulate=G_from, **kw)
    rng = np.random.default_rng(11)
    batches = [tuple(torch.from_numpy(x).to(dev) for x in _ids(rng, B)) for _ in range(3)]
    for u, i in batches[:2]:
        a.train_on_batch(u, i)
    a.save_checkpoint(str(tmp_path / "ck"))
    saved = a.estimator_state()
    a.train_on_batch(*batches[2])
    b = ShardedTwoTowerNet(U, I, E, S, emulate=G_to, seed=5, **kw)
    b.load_checkpoint(str(tmp_path / "ck"))
    got = b.estimator_state()
    assert np.array_equal(got[0], saved[0]) and np.array_equal(got[1].view(np.int32), saved[1].view(np.int32))
    assert got[2] == saved[2] == 2
    b.train_on_batch(*batches[2])
    la, lb = a.estimator_state(), b.estimator_state()
    assert np.array_equal(la[0], lb[0]) and np.array_equal(la[1].view(np.int32), lb[1].view(np.int32)) and la[2] == lb[2] == 3
    for n in ("user", "item"):
        for w in ("w", "m"):
            np.testing.assert_allclose(getattr(b, n).full_weights(w), getattr(a, n).full_weights(w), **W_TOL)
    for d, e in zip(b.dense, a.dense):
        np.testing.assert_allclose(d.w.cpu().numpy(), e.w.cpu().numpy(), **W_TOL)
    # a checkpoint of a model without the estimator: the estimator starts from zero
    plain = ShardedTwoTowerNet(U, I, E, S, emulate=G_from, learning_rate=0.1, tensor_cores=False, device=dev)
    plain.save_checkpoint(str(tmp_path / "plain"))
    b.load_checkpoint(str(tmp_path / "plain"))
    last, gap, step = b.estimator_state()
    assert step == 0 and not last.any() and not gap.any()


def test_rejections(dev):
    from binrec_b200 import _native as N
    from binrec_b200.sharded import ShardedTwoTowerNet
    E, S = 32, 16
    mk = lambda **kw: ShardedTwoTowerNet(U, I, E, S, device=dev, emulate=2, **kw)
    with pytest.raises(ValueError, match="rdZero"):
        mk(rdZero=True, temperature=0.5)
    with pytest.raises(ValueError, match="global_negatives"):
        mk(global_negatives=True, streamingFrequency=0.1)
    for tau in (0.0, -1.0, float("inf"), float("nan"), 5e-324):
        with pytest.raises(ValueError, match="temperature"):
            mk(temperature=tau)
    for a in (0.0, 1.5, -0.1):
        with pytest.raises(ValueError, match="alpha"):
            mk(streamingFrequency=a)
    B = 64
    u = torch.full((B,), 2, dtype=torch.int32, device=dev)
    ones = torch.ones(B, dtype=torch.float32, device=dev)
    est = mk(streamingFrequency=0.1)
    with pytest.raises(ValueError, match="both"):
        est.train_on_batch(u, u, cand_prob=ones)
    with pytest.raises(ValueError, match="global_negatives"):
        mk(global_negatives=True).train_on_batch(u, u, weights=ones)
    with pytest.raises(ValueError, match="rdZero"):
        mk(rdZero=True).train_on_batch(u, u, labels=ones, weights=ones)
    with pytest.raises(ValueError, match="entries"):
        mk(temperature=0.5).train_on_batch(u, u, cand_prob=ones[:B - 1])
    with pytest.raises(ValueError, match="entries"):
        est.train_on_batch(u, u, weights=torch.ones(B + 1, dtype=torch.float32, device=dev))
    assert est.estimator_state()[2] == 0                   # nothing ran
    # the C ABI
    lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()
    ws = est._workspace(B)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    step = torch.zeros(1, dtype=torch.int64, device=dev)

    def copy_est():
        return N.brk_tt_estimator_sharded.from_buffer_copy(est._est.c)

    def call_step(mode=0x100, est_over=None, **over):
        e = copy_est()
        for k, v in (est_over or {}).items():
            setattr(e, k, v) if not isinstance(v, tuple) else getattr(e, k).__setitem__(*v)
        rt = N.brk_tt_retrieval_sharded(None, None, C.pointer(e), 10.0)
        for k, v in over.items():
            setattr(rt, k, v)
        ut, it = est._towers()
        return lib.brk_twotower_step_sharded_retrieval(ctx, C.byref(ut), C.byref(it), C.byref(est._shards()), N.ptr(u), N.ptr(u),
                                                       N.ptr(u), N.ptr(ones), B, mode, C.byref(ws), N.ptr(loss), st, C.byref(rt))

    def call_update(n=B, alpha=0.1, ids=True, step_ptr=True, **over):
        e = copy_est()
        for k, v in over.items():
            setattr(e, k, v) if not isinstance(v, tuple) else getattr(e, k).__setitem__(*v)
        return lib.brk_tt_estimator_update_sharded(ctx, C.byref(e), N.ptr(u) if ids else None, n, alpha,
                                                   N.ptr(step) if step_ptr else None, st)

    def rejected(rc, msg):
        assert rc == -1
        assert msg in lib.brk_last_error().decode(), lib.brk_last_error()

    rejected(call_step(inv_temperature=0.0), "temperature")
    rejected(call_step(inv_temperature=float("inf")), "temperature")
    rejected(call_step(inv_temperature=float("nan")), "temperature")
    rejected(call_step(cand_prob=ones.data_ptr()), "exclusive")
    rejected(call_step(mode=0x101), "rdZero")
    rejected(call_step(est_over=dict(world=3)), "world")
    rejected(call_step(est_over=dict(world=9)), "world")
    rejected(call_step(est_over=dict(rank=1)), "rank")
    rejected(call_step(est_over=dict(rows=0)), "rows")
    rejected(call_step(est_over=dict(gap=(1, None))), "null gap")
    for alpha in (0.0, 1.5, float("nan")):
        rejected(call_update(alpha=alpha), "alpha")
    rejected(call_update(n=-1), "n = ")
    rejected(call_update(ids=False), "n = ")
    rejected(call_update(step_ptr=False), "null argument")
    rejected(call_update(world=0), "world")
    rejected(call_update(rank=2), "rank")
    rejected(call_update(rows=0), "rows")
    rejected(call_update(last=(0, None)), "null last")
    torch.cuda.synchronize()
    assert int(step.item()) == 0                           # nothing ran
    assert call_update(n=0, ids=False) == 0 and call_update() == 0
    assert call_step() == 0
    torch.cuda.synchronize()
    assert int(step.item()) == 2


# ---- two GPUs ------------------------------------------------------------------------------------------
U2, I2, E2, S2 = 1001, 403, 32, 16
TAU2, ALPHA2 = 0.5, 0.1


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _global_batches(kind, world):
    rng = np.random.default_rng(31 if kind == "one_launch" else 32)
    n = world * 256 if kind == "one_launch" else 1900
    return [(rng.integers(2, U2 + 2, n).astype(np.int32), rng.integers(2, 60, n).astype(np.int32),
             rng.uniform(0.0, 2.0, n).astype(np.float32)) for _ in range(3)]


def _slices(kind, world, n):
    """Local batch 256 each (one-launch path), or 1900 rows on rank 0 (the multi-kernel path) and none on the others."""
    if kind == "one_launch":
        return [(r * 256, (r + 1) * 256) for r in range(world)]
    return [(0, n)] + [(n, n)] * (world - 1)


def _worker(rank, world, port, init, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", device_id=dev)
    try:
        from binrec_b200.sharded import ShardedTwoTowerNet
        out = {}
        for kind in ("one_launch", "ragged"):
            net = ShardedTwoTowerNet(U2, I2, E2, S2, device=dev, full_init=init, temperature=TAU2, streamingFrequency=ALPHA2)
            losses = []
            for u, i, w in _global_batches(kind, world):
                lo, hi = _slices(kind, world, len(u))[rank]
                t = lambda x: torch.from_numpy(x[lo:hi]).to(dev)
                losses.append(float(net.train_on_batch(t(u), t(i), weights=t(w)).item()))
            net.check()
            out[kind] = dict(losses=losses, Eu=net.user.full_weights(), Ei=net.item.full_weights(),
                             dense=[d.w.cpu().numpy() for d in net.dense], est=net.estimator_state())
        ret[rank] = out
    except Exception as e:                                 # pragma: no cover - reported by the parent
        ret[rank] = repr(e)
    finally:
        dist.destroy_process_group()


def test_two_gpus_match_the_oracle_with_options():
    """Temperature, sample weights and the estimator on 2 GPUs against one oracle step per global batch: the estimator
    updated on the global batch, each rank's loss the per-slice loss with those probabilities, Adagrad on the summed
    gradients."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import tf32
    from oracle import twotower_retrieval as OR
    world = 2
    o0 = OR.RetrievalOracle(U2, I2, E2, S2, seed=42, temperature=TAU2, matmul=tf32.matmul)
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
    ltol, wtol = dict(rtol=2e-3), dict(rtol=2e-3, atol=1e-4)
    for kind in ("one_launch", "ragged"):
        o = OR.RetrievalOracle(U2, I2, E2, S2, seed=42, temperature=TAU2, matmul=tf32.matmul)
        f = OR.StreamingFrequency(I2 + 2, alpha=ALPHA2)
        ref_losses = []
        for u, i, w in _global_batches(kind, world):
            sl = _slices(kind, world, len(u))
            f.update(i)
            for v in o.t.values():
                v.grad = None
            parts = [o.loss(u[lo:hi], i[lo:hi], cand_ids=i[lo:hi], cand_prob=f.probability(i[lo:hi]), sample_weight=w[lo:hi])
                     if hi > lo else torch.zeros(()) for lo, hi in sl]
            sum(parts).backward()
            ref_losses.append([float(p) for p in parts])
            with torch.no_grad():
                for k, v in o.t.items():
                    g = v.grad if v.grad is not None else torch.zeros_like(v)
                    o.acc[k] += g * g
                    v -= o.lr * g / (o.acc[k].sqrt() + 1e-7)
        for r in range(world):
            got = ret[r][kind]
            np.testing.assert_allclose(got["losses"], [ls[r] for ls in ref_losses], atol=1e-6, **ltol)
            np.testing.assert_allclose(got["Eu"], o.t["Eu"].detach().numpy(), **wtol)
            np.testing.assert_allclose(got["Ei"], o.t["Ei"].detach().numpy(), **wtol)
            last, gap, step = got["est"]
            assert np.array_equal(last, f.last) and np.array_equal(gap.view(np.int32), f.gap.view(np.int32)) and step == 3
        for a, b in zip(ret[0][kind]["dense"], ret[1][kind]["dense"]):
            assert np.array_equal(a, b)
