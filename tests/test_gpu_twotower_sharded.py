"""Row-sharded two-tower training (sharded.ShardedTwoTowerNet, brk_twotower_step_sharded).

One GPU: all G shards of each table live in one process (`emulate=G`) and the whole batch is one replica, so the
result must be the unsharded single-GPU TwoTowerModel's from the same initial weights.  Both sides use the same
arithmetic (TF32 against TF32, fp32 against fp32); only the order of the gradient REDs differs.  Every case proves
which path ran: the one-launch step stamps BRK_TT_TRACE, the multi-kernel step leaves it zero.
Two GPUs: real NVLink peer memory and cross-GPU barriers against oracle/twotower.py with the replicas' losses summed."""
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
# After several steps the two sides' weights differ by more than RED-order noise: a last-bit difference in an operand
# moves it across a TF32 truncation boundary in the next step's products (2^-10 relative), and Adagrad's normalised
# step carries that into the weights (measured up to 1.4e-4 absolute after three steps, with the losses still equal
# to 1e-5).  So the tables, accumulators and Dense blocks are held to a share of how far training moved them: 1e-2
# with TF32 products (test_gpu_tc.py's bound for TF32 gradients), 1e-3 with fp32 products.  A wrong row or owner
# moves an element by the whole update.
MOVED_SHARE = {True: 1e-2, False: 1e-3}


def _pair(dev, E, S, G, rdZero=False, tensor_cores=True):
    from binrec_b200.sharded import ShardedTwoTowerNet
    from binrec_b200.twoTower import TwoTowerModel
    ref = TwoTowerModel(E, I, U, "u", "i", list(range(U)), list(range(I)), rdZero=rdZero, semb=S, device=dev,
                        tensor_cores=tensor_cores)
    ref.compile("Adagrad", learningRate=0.1)
    init = {"user": ref.userTower.emb.w.cpu().numpy(), "item": ref.itemTower.emb.w.cpu().numpy(),
            "user_dense": ref.userTower.dense.w.cpu().numpy(), "item_dense": ref.itemTower.dense.w.cpu().numpy()}
    sh = ShardedTwoTowerNet(U, I, E, S, learning_rate=0.1, rdZero=rdZero, tensor_cores=tensor_cores, device=dev, emulate=G,
                            full_init=init)
    sh.init = {k: v.copy() for k, v in init.items()}
    return ref, sh


def _ids(rng, B, skew=True):
    f = (lambda n: rng.random(n) ** 2) if skew else rng.random
    return (2 + (U * f(B))).astype(np.int32), (2 + (I * f(B))).astype(np.int32)


def _compare_state(ref, sh, share):
    """Tables, accumulators and Dense blocks: |sharded - reference| <= 1e-4 |reference| + share * max |reference - initial|."""
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


CASES = {                                                  # batch, rdZero, tensor cores, BRK_TT_NO_FUSED, one launch
    "one_launch": (1000, False, True, False, True),
    "no_fused": (1000, False, True, True, False),
    "b2000": (2000, False, True, False, False),           # 16^2 = 256 score tiles: more than the SMs
    "rdzero": (1000, True, True, False, False),
    "fp32": (1000, False, False, False, False),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("E,S", [(32, 16), (128, 128)])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_emulated_shards_equal_unsharded_model(dev, monkeypatch, G, E, S, case):
    B, rdZero, tc, no_fused, one_launch = CASES[case]
    if no_fused:
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    ref, sh = _pair(dev, E, S, G, rdZero=rdZero, tensor_cores=tc)
    rng = np.random.default_rng(100 * G + E)
    tr = _Trace(dev, monkeypatch)
    for step in range(3):
        u, i = _ids(rng, B)
        ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
        lab = torch.from_numpy((rng.random(B) < 0.5).astype(np.float32)).to(dev) if rdZero else None
        l0 = ref._train_ids(ud, idd, lab).item()
        with tr:
            l1 = sh.train_on_batch(ud, idd, lab).item()
        np.testing.assert_allclose(l1, l0, **LOSS_TOL)
    assert tr.stamped() == one_launch, "the step did not take the expected path"
    _compare_state(ref, sh, MOVED_SHARE[tc])


def _bits(words, n):
    w = words.cpu().numpy().view(np.uint32)
    return ((w[:, None] >> np.arange(32, dtype=np.uint32)[None, :]) & 1).astype(bool).reshape(-1)[:n]


@pytest.mark.parametrize("no_fused", [False, True])
def test_touched_bits_at_the_owners_and_row_sparse_adagrad(dev, monkeypatch, no_fused):
    if no_fused:
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    G, E, S, B = 3, 32, 16, 700
    _, sh = _pair(dev, E, S, G)
    u, i = _ids(np.random.default_rng(7), B)
    w0 = {name: [t.tables[r].w.clone() for r in range(G)] for name, t in (("user", sh.user), ("item", sh.item))}
    sh.forward_backward(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev))
    for name, t, ids in (("user", sh.user, u), ("item", sh.item, i)):
        for r in range(G):
            expect = np.zeros(t.local_rows, bool)
            mine = np.unique(ids[ids % G == r])
            expect[mine // G] = True
            assert np.array_equal(_bits(t.tables[r].touched, t.local_rows), expect), (name, r)
            g = t.tables[r].g.cpu().numpy()
            assert not g[~expect].any() and (np.abs(g[expect]).sum(1) > 0).all(), (name, r)
    sh.apply_gradients()
    for name, t, ids in (("user", sh.user, u), ("item", sh.item, i)):
        for r in range(G):
            hit = np.zeros(t.local_rows, bool)
            hit[np.unique(ids[ids % G == r]) // G] = True
            w = t.tables[r].w.cpu().numpy(); before = w0[name][r].cpu().numpy()
            assert np.array_equal(w[~hit], before[~hit]), (name, r)
            assert (w[hit] != before[hit]).any(1).all(), (name, r)
            assert int(t.tables[r].touched.abs().sum().item()) == 0
            assert not t.tables[r].g.cpu().numpy().any()


def test_accidental_hits_across_shards(dev):
    """Few distinct items, repeated so that neighbours in the batch belong to different owners: every row's in-batch
    negatives hold accidental hits whose rows live on other shards."""
    G, E, S, B = 3, 32, 16, 600
    ref, sh = _pair(dev, E, S, G)
    pool = np.array([10, 11, 12, 13, 14, 15, 16], np.int32)     # owners 1, 2, 0, 1, 2, 0, 1
    i = pool[np.arange(B) % len(pool)]
    u = (2 + np.random.default_rng(3).integers(0, U, B)).astype(np.int32)
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    l0 = ref._step(ud, idd, None, True).item()
    l1 = sh.forward_backward(ud, idd).item()
    np.testing.assert_allclose(l1, l0, **LOSS_TOL)
    np.testing.assert_allclose(sh.user.full_weights("g"), ref.userTower.emb.g.cpu().numpy(), **W_TOL)
    np.testing.assert_allclose(sh.item.full_weights("g"), ref.itemTower.emb.g.cpu().numpy(), **W_TOL)
    for d, tw in zip(sh.dense, (ref.userTower, ref.itemTower)):
        np.testing.assert_allclose(d.g.cpu().numpy(), tw.dense.g.cpu().numpy(), **W_TOL)


@pytest.mark.parametrize("G", [2, 3])
def test_score_vectors_bit_identical(dev, G):
    ref, sh = _pair(dev, 64, 32, G)
    rng = np.random.default_rng(G)
    u, i = _ids(rng, 777, skew=False)
    ud, idd = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    q, c = sh.score_vectors(ud, idd)
    assert torch.equal(q, ref._tower_forward(ref.userTower, ud))
    assert torch.equal(c, ref._tower_forward(ref.itemTower, idd))


def test_checkpoint_resharding(dev, tmp_path):
    from binrec_b200.sharded import ShardedTwoTowerNet
    E, S, B = 32, 16, 500                                  # fp32 products: one step from equal weights differs by RED order only
    ref, a = _pair(dev, E, S, 2, tensor_cores=False)
    rng = np.random.default_rng(11)
    batches = [tuple(torch.from_numpy(x).to(dev) for x in _ids(rng, B)) for _ in range(3)]
    for u, i in batches[:2]:
        a.train_on_batch(u, i)
    a.save_checkpoint(str(tmp_path / "ck"))
    saved = {(n, w): getattr(a, n).full_weights(w) for n in ("user", "item") for w in ("w", "m")}
    dense = [(d.w.cpu().numpy(), d.m.cpu().numpy()) for d in a.dense]
    a.train_on_batch(*batches[2])
    for G in (3, 0):                                       # emulated G = 3, and one unsharded process (G = 1)
        b = ShardedTwoTowerNet(U, I, E, S, learning_rate=0.1, tensor_cores=False, device=dev, emulate=G, seed=5)
        b.load_checkpoint(str(tmp_path / "ck"))
        for (n, w), v in saved.items():
            assert np.array_equal(getattr(b, n).full_weights(w), v), (G, n, w)
        for d, (w, m) in zip(b.dense, dense):
            assert np.array_equal(d.w.cpu().numpy(), w) and np.array_equal(d.m.cpu().numpy(), m)
        b.train_on_batch(*batches[2])
        for n in ("user", "item"):
            for w in ("w", "m"):
                np.testing.assert_allclose(getattr(b, n).full_weights(w), getattr(a, n).full_weights(w), **W_TOL)
        for d, e in zip(b.dense, a.dense):
            np.testing.assert_allclose(d.w.cpu().numpy(), e.w.cpu().numpy(), **W_TOL)


def test_argument_validation(dev):
    from binrec_b200 import _native as N
    _, sh = _pair(dev, 32, 16, 2)
    B = 256
    u = torch.full((B,), 2, dtype=torch.int32, device=dev)
    ws = sh._workspace(B)
    loss = torch.empty(1, device=dev)
    lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()

    def call(shards, towers=None):
        ut, it = towers or sh._towers()
        return lib.brk_twotower_step_sharded(ctx, C.byref(ut), C.byref(it), C.byref(shards) if shards is not None else None,
                                             N.ptr(u), N.ptr(u), N.ptr(u), None, B, 0x100, C.byref(ws), N.ptr(loss), st)

    assert call(sh._shards()) == 0
    assert call(None) == -1
    for world in (0, N.BRK_MAX_PEERS + 1):
        s = sh._shards(); s.user.world = world
        assert call(s) == -1, world
    s = sh._shards(); s.item.rank = 2
    assert call(s) == -1
    for field in ("w", "g", "touched"):
        s = sh._shards(); getattr(s.item, field)[1] = None
        assert call(s) == -1, field
    ut, it = sh._towers(); ut.E = 30
    assert call(sh._shards(), (ut, it)) == -1
    torch.cuda.synchronize()


# ---- two GPUs ------------------------------------------------------------------------------------------
U2, I2, E2, S2 = 1001, 403, 32, 16


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _global_batches(kind, world):
    rng = np.random.default_rng(21 if kind == "one_launch" else 22)
    n = world * 256 if kind == "one_launch" else 1900
    return [(rng.integers(2, U2 + 2, n).astype(np.int32), rng.integers(2, I2 + 2, n).astype(np.int32)) for _ in range(3)]


def _slices(kind, world, n):
    """Local batch 256 each (one-launch path), or a ragged split: 1900 rows on rank 0 (above 1536: the multi-kernel
    path), none on the others."""
    if kind == "one_launch":
        return [(r * 256, (r + 1) * 256) for r in range(world)]
    return [(0, n)] + [(n, n)] * (world - 1)


def _worker(rank, world, port, init, tc, ret):
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
            net = ShardedTwoTowerNet(U2, I2, E2, S2, tensor_cores=tc, device=dev, full_init=init)
            losses = []
            for u, i in _global_batches(kind, world):
                lo, hi = _slices(kind, world, len(u))[rank]
                losses.append(float(net.train_on_batch(torch.from_numpy(u[lo:hi]).to(dev), torch.from_numpy(i[lo:hi]).to(dev)).item()))
            net.check()
            out[kind] = dict(losses=losses, Eu=net.user.full_weights(), Ei=net.item.full_weights(),
                             dense=[d.w.cpu().numpy() for d in net.dense])
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
    o0 = OTT.TwoTowerOracle(U2, I2, E2, S2, seed=42, matmul=tf32.matmul if tc else torch.matmul)
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
    for kind in ("one_launch", "ragged"):
        o = OTT.TwoTowerOracle(U2, I2, E2, S2, seed=42, matmul=tf32.matmul if tc else torch.matmul)
        ref_losses = []
        for u, i in _global_batches(kind, world):
            sl = _slices(kind, world, len(u))
            for v in o.t.values():
                v.grad = None
            parts = [o.loss(u[lo:hi], i[lo:hi], cand_ids=i[lo:hi]) if hi > lo else torch.zeros(()) for lo, hi in sl]
            sum(parts).backward()
            ref_losses.append([float(p) for p in parts])
            with torch.no_grad():
                for k, w in o.t.items():
                    g = w.grad if w.grad is not None else torch.zeros_like(w)
                    o.acc[k] += g * g
                    w -= o.lr * g / (o.acc[k].sqrt() + 1e-7)
        for r in range(world):
            got = ret[(tc, r)][kind]
            np.testing.assert_allclose(got["losses"], [ls[r] for ls in ref_losses], atol=1e-6, **ltol)
            np.testing.assert_allclose(got["Eu"], o.t["Eu"].detach().numpy(), **wtol)
            np.testing.assert_allclose(got["Ei"], o.t["Ei"].detach().numpy(), **wtol)
            np.testing.assert_allclose(got["dense"][1][:E2 * S2], o.t["Wi"].detach().numpy().reshape(-1), **wtol)
        for a, b in zip(ret[(tc, 0)][kind]["dense"], ret[(tc, 1)][kind]["dense"]):
            assert np.array_equal(a, b)
