"""Global in-batch negatives for data-parallel two-tower training (twoTower.GlobalNegatives, brk_twotower_step_global).

One GPU: ShardedTwoTowerNet(global_negatives=True, emulate=G) splits every batch over G emulated ranks with local_slice
and runs the three phases rank by rank, so the ranks' summed loss and the trained state must be the unsharded
single-GPU TwoTowerModel's on the same global batches.  Two GPUs: real peer memory and barriers, for the row-sharded
and the mirrored model, against one oracle step per global batch."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U, I = 301, 203
LOSS_TOL = {False: dict(rtol=1e-5, atol=1e-6), True: dict(rtol=2e-3, atol=1e-4)}
W_TOL = dict(rtol=1e-4, atol=2e-6)
# The tables and Dense blocks are held to a share of how far training moved them, as in test_gpu_twotower_sharded.py:
# after a few steps a last-bit difference moves an operand across a TF32 rounding boundary, and Adagrad's normalised
# step carries that into the weights.
MOVED_SHARE = {True: 1e-2, False: 1e-3}


def _pair(dev, E, S, G, tensor_cores=True, global_negatives=True):
    from binrec_b200.sharded import ShardedTwoTowerNet
    from binrec_b200.twoTower import TwoTowerModel
    ref = TwoTowerModel(E, I, U, "u", "i", list(range(U)), list(range(I)), semb=S, device=dev, tensor_cores=tensor_cores)
    ref.compile("Adagrad", learningRate=0.1)
    init = {"user": ref.userTower.emb.w.cpu().numpy(), "item": ref.itemTower.emb.w.cpu().numpy(),
            "user_dense": ref.userTower.dense.w.cpu().numpy(), "item_dense": ref.itemTower.dense.w.cpu().numpy()}
    sh = ShardedTwoTowerNet(U, I, E, S, learning_rate=0.1, tensor_cores=tensor_cores, device=dev, emulate=G, full_init=init,
                            global_negatives=global_negatives)
    sh.init = {k: v.copy() for k, v in init.items()}
    return ref, sh


def _ids(rng, B):
    f = lambda n: rng.random(n) ** 2                       # skewed: repeated items, so accidental hits occur
    return (2 + (U * f(B))).astype(np.int32), (2 + (I * f(B))).astype(np.int32)


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


def _train(ref, sh, batches, tc):
    for u, i in batches:
        ud, idd = torch.from_numpy(u).to(sh.device), torch.from_numpy(i).to(sh.device)
        l0 = ref._train_ids(ud, idd, None).item()
        l1 = sh.train_on_batch(ud, idd).item()
        np.testing.assert_allclose(l1, l0, **LOSS_TOL[tc])
    sh.check()
    _compare_state(ref, sh, MOVED_SHARE[tc])


@pytest.mark.parametrize("tc", [True, False])
@pytest.mark.parametrize("E,S", [(32, 16), (128, 128)])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_emulated_global_negatives_equal_unsharded_model(dev, G, E, S, tc):
    ref, sh = _pair(dev, E, S, G, tensor_cores=tc)
    rng = np.random.default_rng(10 * G + E)
    _train(ref, sh, [_ids(rng, 1000) for _ in range(3)], tc)


@pytest.mark.parametrize("tc", [True, False])
@pytest.mark.parametrize("B,G", [(1900, 3), (5, 8), (7, 3)])
def test_ragged_and_empty_slices(dev, B, G, tc):
    """1900 rows over 3 ranks (634 / 633 / 633); 5 rows over 8 ranks (three empty slices)."""
    ref, sh = _pair(dev, 32, 16, G, tensor_cores=tc)
    rng = np.random.default_rng(B + G)
    _train(ref, sh, [_ids(rng, B) for _ in range(3)], tc)


def _hit_batch(B=600):
    """Few distinct items repeated with period 7 over the batch: every slice holds items that other slices hold too."""
    pool = np.array([10, 11, 12, 13, 14, 15, 16], np.int32)
    i = pool[np.arange(B) % len(pool)]
    u = (2 + np.random.default_rng(3).integers(0, U, B)).astype(np.int32)
    return u, i


def test_accidental_hits_masked_across_slices(dev):
    from oracle import twotower as OTT
    G, E, S = 3, 32, 16
    ref, sh = _pair(dev, E, S, G, tensor_cores=False)
    u, i = _hit_batch()
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    l0 = ref._step(ud, idd, None, True).item()
    l1 = sh.forward_backward(ud, idd).item()
    np.testing.assert_allclose(l1, l0, **LOSS_TOL[False])
    np.testing.assert_allclose(sh.user.full_weights("g"), ref.userTower.emb.g.cpu().numpy(), **W_TOL)
    np.testing.assert_allclose(sh.item.full_weights("g"), ref.itemTower.emb.g.cpu().numpy(), **W_TOL)
    for d, tw in zip(sh.dense, (ref.userTower, ref.itemTower)):
        np.testing.assert_allclose(d.g.cpu().numpy(), tw.dense.g.cpu().numpy(), **W_TOL)
    # the oracle at the global batch, hits masked across slices, agrees; the per-replica loss (hits masked inside each
    # slice only, its own slice as negatives) does not
    o = OTT.TwoTowerOracle(U, I, E, S)
    with torch.no_grad():
        for k, t in (("Eu", sh.init["user"]), ("Ei", sh.init["item"])):
            o.t[k].copy_(torch.from_numpy(t))
        for side, (wn, bn) in (("user", ("Wu", "bu")), ("item", ("Wi", "bi"))):
            flat = sh.init[side + "_dense"].reshape(-1)
            o.t[wn].copy_(torch.from_numpy(flat[:E * S].reshape(E, S))); o.t[bn].copy_(torch.from_numpy(flat[E * S:E * S + S]))
        glob = float(o.loss(u, i, cand_ids=i))
        from binrec_b200.distributed import local_slice
        per_replica = sum(float(o.loss(u[lo:hi], i[lo:hi], cand_ids=i[lo:hi])) for lo, hi in
                          (local_slice(len(u), r, G) for r in range(G)))
    np.testing.assert_allclose(l1, glob, rtol=1e-5)
    assert abs(per_replica - glob) > 1e-3 * abs(glob)


def test_flag_changes_the_loss_only_with_more_than_one_replica(dev):
    from oracle import twotower as OTT
    E, S = 32, 16
    u, i = _ids(np.random.default_rng(5), 512)
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    # G = 2: global negatives give the one-GPU loss of the whole batch; per-replica negatives (each half its own
    # candidates) give a different number
    _, sh = _pair(dev, E, S, 2, tensor_cores=False)
    glob = sh.forward_backward(ud, idd).item()
    o = OTT.TwoTowerOracle(U, I, E, S)
    with torch.no_grad():
        o.t["Eu"].copy_(torch.from_numpy(sh.init["user"])); o.t["Ei"].copy_(torch.from_numpy(sh.init["item"]))
        for side, (wn, bn) in (("user", ("Wu", "bu")), ("item", ("Wi", "bi"))):
            flat = sh.init[side + "_dense"].reshape(-1)
            o.t[wn].copy_(torch.from_numpy(flat[:E * S].reshape(E, S))); o.t[bn].copy_(torch.from_numpy(flat[E * S:E * S + S]))
        per_replica = float(o.loss(u[:256], i[:256], cand_ids=i[:256])) + float(o.loss(u[256:], i[256:], cand_ids=i[256:]))
        np.testing.assert_allclose(glob, float(o.loss(u, i, cand_ids=i)), rtol=1e-5)
    assert abs(per_replica - glob) > 1e-2 * abs(glob)
    # one replica: the flag changes nothing -- the same step runs, so the first losses agree bit for bit; the weights
    # (and the losses computed from them) agree to the order of the step's gradient REDs, which differs between runs
    for G in (1, 0):
        _, a = _pair(dev, E, S, G, tensor_cores=False, global_negatives=True)
        _, b = _pair(dev, E, S, G, tensor_cores=False, global_negatives=False)
        assert a._global is None
        assert a.train_on_batch(ud, idd).item() == b.train_on_batch(ud, idd).item()
        np.testing.assert_allclose(a.train_on_batch(ud, idd).item(), b.train_on_batch(ud, idd).item(), **LOSS_TOL[False])
        for n in ("user", "item"):
            np.testing.assert_allclose(getattr(a, n).full_weights(), getattr(b, n).full_weights(), **W_TOL)
        for x, y in zip(a.dense, b.dense):
            np.testing.assert_allclose(x.w.cpu().numpy(), y.w.cpu().numpy(), **W_TOL)


def test_argument_validation(dev):
    from binrec_b200 import _native as N
    from binrec_b200.sharded import ShardedTwoTowerNet
    from binrec_b200.twoTower import TwoTowerModel
    with pytest.raises(ValueError, match="rdZero"):
        ShardedTwoTowerNet(U, I, 32, 16, rdZero=True, device=dev, emulate=2, global_negatives=True)
    with pytest.raises(ValueError, match="rdZero"):
        TwoTowerModel(32, I, U, "u", "i", list(range(U)), list(range(I)), rdZero=True, semb=16, device=dev,
                      global_negatives=True)
    _, sh = _pair(dev, 32, 16, 2)
    u, i = _ids(np.random.default_rng(1), 64)
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    sh.forward_backward(ud, idd)                          # buffers allocated for a 64-row batch
    gn = sh._global
    counts = [32, 32]
    ws = gn._workspace(0, 32, 64)
    loss = torch.empty(1, device=dev)
    lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()

    def call(g, towers=None, shards=True, mode=0x100):
        ut, it = towers or sh._towers()
        s = sh._shards() if shards else None
        return lib.brk_twotower_step_global(ctx, 0, C.byref(ut), C.byref(it), C.byref(s) if s is not None else None,
                                            C.byref(g) if g is not None else None, N.ptr(ud), N.ptr(idd), mode, C.byref(ws),
                                            N.ptr(loss), st)

    assert call(gn._struct(0, counts)) == 0
    assert call(None) == -1
    assert call(gn._struct(0, counts), mode=1) == -1                 # rdZero
    for world in (0, N.BRK_MAX_PEERS + 1):
        g = gn._struct(0, counts); g.world = world
        assert call(g) == -1, world
    g = gn._struct(0, counts); g.rank = 2
    assert call(g) == -1
    g = gn._struct(0, counts); g.offset[1] = 31                      # overlapping slices
    assert call(g) == -1
    g = gn._struct(0, counts); g.offset[0] = 1                       # a gap at the start
    assert call(g) == -1
    g = gn._struct(0, [32, 33]); g.cap = 64                           # n above the slot capacity
    assert call(g) == -1
    g = gn._struct(0, counts); g.cap = 16                            # a count above the block capacity
    assert call(g) == -1
    ut, it = sh._towers(); ut.S = 20
    assert call(gn._struct(0, counts), (ut, it)) == -1               # S mismatch
    for field in ("cand", "ids", "slot"):
        g = gn._struct(0, counts); getattr(g, field)[1] = None
        assert call(g) == -1, field
    for field in ("c_all", "ids_all", "err"):
        g = gn._struct(0, counts); setattr(g, field, None)
        assert call(g) == -1, field
    g = gn._struct(0, counts)
    assert lib.brk_twotower_step_global(ctx, 0, C.byref(sh._towers()[0]), C.byref(sh._towers()[1]), None, C.byref(g), N.ptr(ud),
                                        N.ptr(idd), 0x100, C.byref(ws), N.ptr(loss), st) == -1   # no shards: tables missing
    torch.cuda.synchronize()


def test_a_published_slice_that_differs_from_the_split_is_reported(dev):
    _, sh = _pair(dev, 32, 16, 2)
    u, i = _ids(np.random.default_rng(2), 64)
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    sh.forward_backward(ud, idd)
    sh.check()
    sh._global._bufs[1][1][0] = 31                        # rank 1's header now claims 31 rows, the split says 32
    from binrec_b200 import _native as N
    gn = sh._global
    ws = gn._workspace(0, 32, 64)
    ut, it = sh._towers()
    s = sh._shards()
    N.check(N.lib().brk_twotower_step_global(N.ctx(dev), 1, C.byref(ut), C.byref(it), C.byref(s), C.byref(gn._struct(0, [32, 32])),
                                             N.ptr(ud[:32]), N.ptr(idd[:32]), 0x100, C.byref(ws), None, N.stream_ptr()),
            "brk_twotower_step_global")
    with pytest.raises(RuntimeError, match="rank 1"):
        sh.check()
    sh.check()                                            # reported once


# ---- two GPUs ------------------------------------------------------------------------------------------
U2, I2, E2, S2 = 1001, 403, 32, 16


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _global_batches(kind):
    rng = np.random.default_rng(31 if kind == "equal" else 32)
    n = 512 if kind == "equal" else 1901
    return [(rng.integers(2, U2 + 2, n).astype(np.int32), rng.integers(2, I2 + 2, n).astype(np.int32)) for _ in range(3)]


def _worker(rank, world, port, init, tc, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", device_id=dev)
    try:
        from binrec_b200.distributed import local_slice
        from binrec_b200.sharded import ShardedTwoTowerNet
        from binrec_b200.twoTower import TwoTowerModel
        out = {}
        for kind in ("equal", "ragged"):
            net = ShardedTwoTowerNet(U2, I2, E2, S2, tensor_cores=tc, device=dev, full_init=init, global_negatives=True)
            mir = TwoTowerModel(E2, I2, U2, "u", "i", list(range(U2)), list(range(I2)), semb=S2, device=dev, tensor_cores=tc,
                                global_negatives=True)
            mir.compile("Adagrad", learningRate=0.1)
            with torch.no_grad():
                mir.userTower.emb.w.copy_(torch.from_numpy(init["user"])); mir.itemTower.emb.w.copy_(torch.from_numpy(init["item"]))
                mir.userTower.dense.w.view(-1).copy_(torch.from_numpy(init["user_dense"]))
                mir.itemTower.dense.w.view(-1).copy_(torch.from_numpy(init["item_dense"]))
            losses, mlosses = [], []
            for u, i in _global_batches(kind):
                split = [hi - lo for lo, hi in (local_slice(len(u), r, world) for r in range(world))]
                lo, hi = local_slice(len(u), rank, world)
                ud, idd = torch.from_numpy(u[lo:hi]).to(dev), torch.from_numpy(i[lo:hi]).to(dev)
                losses.append(float(net.train_on_batch(ud, idd, split=split).item()))
                info = {"u": [int(x) - 2 for x in u[lo:hi]], "i": [int(x) - 2 for x in i[lo:hi]]}
                mlosses.append(float(mir.train_step(info, split=split)["loss"].item()))
            net.check()
            mir._global.check()
            out[kind] = dict(losses=losses, Eu=net.user.full_weights(), Ei=net.item.full_weights(),
                             dense=[d.w.cpu().numpy() for d in net.dense], mlosses=mlosses,
                             mEu=mir.userTower.emb.w.cpu().numpy(), mEi=mir.itemTower.emb.w.cpu().numpy(),
                             mdense=[t.dense.w.cpu().numpy() for t in (mir.userTower, mir.itemTower)])
        ret[(tc, rank)] = out
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("tc", [True, False])
def test_two_gpus_match_the_oracle(tc):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import tf32
    from oracle import twotower as OTT
    world = 2
    mm = tf32.matmul if tc else torch.matmul
    o0 = OTT.TwoTowerOracle(U2, I2, E2, S2, seed=42, matmul=mm)
    init = {"user": o0.t["Eu"].detach().numpy().copy(), "item": o0.t["Ei"].detach().numpy().copy()}
    for k, (wn, bn) in enumerate((("Wu", "bu"), ("Wi", "bi"))):
        flat = np.concatenate([o0.t[wn].detach().numpy().reshape(-1), o0.t[bn].detach().numpy()])
        init[("user_dense", "item_dense")[k]] = np.pad(flat, (0, (-len(flat)) % 4))
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, init, tc, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    ltol, wtol = (dict(rtol=2e-3), dict(rtol=2e-3, atol=1e-4)) if tc else (dict(rtol=1e-5), dict(rtol=1e-4, atol=1e-5))
    for kind in ("equal", "ragged"):
        o = OTT.TwoTowerOracle(U2, I2, E2, S2, seed=42, matmul=mm)
        ref = [o.step(u, i, cand_ids=i) for u, i in _global_batches(kind)]
        for pre in ("", "m"):
            got = [ret[(tc, r)][kind] for r in range(world)]
            total = np.sum([g[pre + "losses" if pre else "losses"] for g in got], axis=0)
            np.testing.assert_allclose(total, ref, atol=1e-6, **ltol)
            for g in got:
                np.testing.assert_allclose(g[pre + "Eu"], o.t["Eu"].detach().numpy(), **wtol)
                np.testing.assert_allclose(g[pre + "Ei"], o.t["Ei"].detach().numpy(), **wtol)
                dense = g[pre + "dense"]
                for k, (wn, bn) in enumerate((("Wu", "bu"), ("Wi", "bi"))):
                    np.testing.assert_allclose(dense[k].reshape(-1)[:E2 * S2], o.t[wn].detach().numpy().reshape(-1), **wtol)
                    np.testing.assert_allclose(dense[k].reshape(-1)[E2 * S2:E2 * S2 + S2], o.t[bn].detach().numpy(), **wtol)
            for a, b in zip(got[0][pre + "dense"], got[1][pre + "dense"]):
                assert np.array_equal(a, b)
