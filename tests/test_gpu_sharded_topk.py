"""Full-catalog top-k of the row-sharded models over item ranges (sharded.ShardedTopKIndex, brk_topk_merge_peer).

One GPU: `emulate=G` holds all G shards in one process, builds the G item-range indexes there and merges their lists
with the same peer-merge kernel a multi-GPU run uses.  After a few sharded training steps the lists must equal, bit
for bit, the single-GPU index over the same full weights (NeuMFNet.topk_index / topk_index_fp32 with the sharded
model's tables, dense block and BatchNorm statistics; BruteForceIndex for BPR and two-tower).  Two GPUs: peer and NCCL
modes in one process per GPU, every rank's lists identical and equal to the single-process index over the gathered
weights with rank 0's BatchNorm statistics."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

NU, NI = 301, 203                                         # row counts not divisible by G


def _batches(U, I, B, steps, seed):
    rng = np.random.default_rng(seed)
    return [((U * rng.random(B) ** 2).astype(np.int32), (I * rng.random(B) ** 2).astype(np.int32),
             (rng.random(B) < 0.25).astype(np.float32)) for _ in range(steps)]


def _train_neumf(net, dev, steps=3, B=500, seed=1, world=1, rank=0):
    from binrec_b200 import distributed as D
    for s, (u, i, y) in enumerate(_batches(net.numUser, net.numItem, world * B, steps, seed)):
        lo, hi = D.local_slice(world * B, rank, world)
        net.train_on_batch(*(torch.from_numpy(x[lo:hi]).to(dev) for x in (u, i, y)), first_index=s * world * B + lo, epoch=1)
    torch.cuda.synchronize()


def _neumf_reference(dev, E, tc, full, dense, bn, U=NU, I=NI):
    """NeuMFNet holding the given full tables, dense block and BatchNorm statistics."""
    from binrec_b200.NeuMFModel import NeuMFNet
    ref = NeuMFNet(U, I, E, dropout=0.0, sparse_adam="lazy", tensor_cores=tc, device=dev)
    for name in ("uMLP", "iMLP", "uMF", "iMF"):
        getattr(ref, name).w.copy_(torch.from_numpy(full[name]))
    ref.dense.w.view(-1)[:len(dense)].copy_(torch.from_numpy(dense))
    ref.bn_moving.copy_(torch.from_numpy(bn))
    return ref


def _neumf_pair(dev, G, E, tc, seed=5):
    from binrec_b200.sharded import ShardedNeuMFNet
    sh = ShardedNeuMFNet(NU, NI, E, dropout=0.2, seed=seed, device=dev, emulate=G, tensor_cores=tc)
    _train_neumf(sh, dev, seed=seed + G)
    assert float(sh.bn_moving[:E].abs().sum().item()) > 0            # the BatchNorm statistics have moved
    full = {n: getattr(sh, n).full_weights() for n in ("uMLP", "iMLP", "uMF", "iMF")}
    ref = _neumf_reference(dev, E, tc, full, sh.dense.w.view(-1).cpu().numpy(), sh.bn_moving.cpu().numpy())
    return sh, ref


def _index(net, tc, items=None):
    return net.topk_index(items) if tc else net.topk_index_fp32(items)


def _same(a, b):
    assert a[0].shape == b[0].shape and a[1].shape == b[1].shape, (a[0].shape, b[0].shape)
    assert torch.equal(a[1], b[1]), (a[1], b[1])
    assert torch.equal(a[0], b[0])


def _users(rng, n=97):
    return torch.from_numpy(np.concatenate([rng.integers(0, NU, n), [3, 3, 0, NU - 1]]).astype(np.int32))


NEUMF_MODELS = [(32, True), (64, True), (8, False), (16, False), (64, False)]


@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("E,tc", NEUMF_MODELS)
def test_neumf_parity(dev, G, E, tc):
    from binrec_b200 import hotpath as H
    sh, ref = _neumf_pair(dev, G, E, tc)
    rng = np.random.default_rng(G * 100 + E)
    users = _users(rng).to(dev)
    a, b = _index(sh, tc), _index(ref, tc)
    for k in (1, 10, 32):
        _same(a(users, k), b(users, k))
    # a permuted subset of the items whose count G does not divide, and exclusions that empty rows below k
    items = rng.permutation(NI)[:NI - 4 - G]
    a, b = _index(sh, tc, items), _index(ref, tc, items)
    _same(a(users, 10), b(users, 10))
    rows = np.concatenate([np.repeat(np.arange(20), 8), np.full(len(items) - 5, 20)])
    cols = np.concatenate([rng.integers(0, len(items), 160), np.arange(5, len(items))])
    csr = H.exclusion_csr(rows, cols, users.numel(), dev)
    got, want = a.query_with_exclusions(users, csr, 10), b.query_with_exclusions(users, csr, 10)
    _same(got, want)
    assert (got[1][20] >= 0).sum().item() == 5 and got[1][20, 5:].eq(-1).all() and torch.isinf(got[0][20, 5:]).all()


@pytest.mark.parametrize("G", [2, 3, 8])
def test_neumf_item_and_user_lists(dev, G):
    sh, ref = _neumf_pair(dev, G, 32, True)
    users = torch.tensor([5, 5, 7, 0, 5], dtype=torch.int32, device=dev)    # duplicate user ids
    for items in ([11, 4, 200][:G - 1], [17, 3, 150, 9, 60]):                # fewer items than ranks; k > len(itemsId)
        a, b = sh.topk_index(items), ref.topk_index(items)
        got = a(users, 10)
        assert got[0].shape == (5, len(items))
        _same(got, b(users, 10))
        assert torch.equal(got[0][0], got[0][1]) and torch.equal(got[1][0], got[1][4])
    v, i = sh.topk_index()(torch.empty(0, dtype=torch.int32, device=dev), 10)
    assert v.shape == (0, 10) and i.shape == (0, 10)
    v, i = sh.topk_index()([], 4)
    assert v.shape == (0, 4)


def test_several_chunks_per_query(dev, monkeypatch):
    """Lists exchanged in many chunks through the two alternating buffers equal a one-chunk query."""
    from binrec_b200.sharded import ShardedTopKIndex
    sh, ref = _neumf_pair(dev, 3, 16, False)
    users = _users(np.random.default_rng(7), 300).to(dev)
    want = ref.topk_index_fp32()(users, 10)
    monkeypatch.setattr(ShardedTopKIndex, "CHUNK_ENTRIES", 10 * 37)
    idx = sh.topk_index_fp32()
    _same(idx(users, 10), want)
    _same(idx(users, 10), want)                                              # the slots keep alternating across queries


def _bpr_pair(dev, G, d=64, steps=3, full_init=None):
    from binrec_b200.sharded import ShardedBPRNet
    sh = ShardedBPRNet(NU, NI, d, device=dev, emulate=G, full_init=full_init)
    rng = np.random.default_rng(G)
    for _ in range(steps):
        u, p, n = (rng.integers(0, NU, 400).astype(np.int32), rng.integers(0, NI, 400).astype(np.int32),
                   rng.integers(0, NI, 400).astype(np.int32))
        sh.train_on_batch(*(torch.from_numpy(x).to(dev) for x in (u, p, n)))
    torch.cuda.synchronize()
    return sh, sh.user.full_weights(), sh.item.full_weights()


def _bf(k, cand, q, dev):
    from binrec_b200 import hotpath as H
    return H.BruteForceIndex(k).index(torch.from_numpy(np.ascontiguousarray(cand)).to(dev))(
        torch.from_numpy(np.ascontiguousarray(q)).to(dev))


@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_bpr_parity(dev, G):
    from binrec_b200 import hotpath as H
    sh, uw, iw = _bpr_pair(dev, G)
    rng = np.random.default_rng(G)
    users = _users(rng).numpy()
    items = rng.permutation(NI)[:NI - 2 - G]
    for k in (1, 10, 100, 128):
        got = sh.topk_index(items, k)(users)
        _same(got, _bf(k, iw[items], uw[users], dev))
    csr = H.exclusion_csr(np.repeat(np.arange(10), 20), rng.integers(0, len(items), 200), len(users), dev)
    ref = H.BruteForceIndex(10).index(torch.from_numpy(iw[items]).to(dev))
    _same(sh.topk_index(items).query_with_exclusions(users, csr),
          ref.query_with_exclusions(torch.from_numpy(uw[users]).to(dev), csr))


@pytest.mark.parametrize("G", [1, 3, 8])
def test_two_tower_parity(dev, G):
    from binrec_b200 import hotpath as H
    from binrec_b200.sharded import ShardedTwoTowerNet
    net = ShardedTwoTowerNet(NU, NI, 32, 64, device=dev, emulate=G)
    rng = np.random.default_rng(G)
    for _ in range(3):
        u, i = rng.integers(0, NU + 2, 256).astype(np.int32), rng.integers(0, NI + 2, 256).astype(np.int32)
        net.train_on_batch(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev))
    users = torch.from_numpy(rng.integers(0, NU + 2, 150).astype(np.int32)).to(dev)
    items = torch.from_numpy(rng.permutation(NI + 2)[:NI - 1].astype(np.int32)).to(dev)
    uv, iv = net.score_vectors(users, items)
    for k in (10, 128):
        _same(net.topk_index(items, k)(users), H.BruteForceIndex(k).index(iv)(uv))
    _, iv_all = net.score_vectors(users, torch.arange(NI + 2, dtype=torch.int32, device=dev))
    _same(net.topk_index()(users), H.BruteForceIndex(10).index(iv_all)(uv))


@pytest.mark.parametrize("G", [2, 3, 8])
def test_ties_across_range_boundaries_go_to_the_lower_position(dev, G):
    """Equal item rows on both sides of every range boundary: the lower position wins, as in the unsharded scan."""
    from binrec_b200 import distributed as D
    rng = np.random.default_rng(G)
    d, I = 64, 64
    item = rng.integers(-2, 3, size=(I, d)).astype(np.float32)
    user = rng.integers(-2, 3, size=(NU, d)).astype(np.float32)
    bounds = [D.local_slice(I, r, G)[0] for r in range(1, G)]
    for b in bounds:
        item[b - 2:b + 2] = item[b - 2]                    # four equal rows straddling the boundary
    from binrec_b200.sharded import ShardedBPRNet
    sh = ShardedBPRNet(NU, I, d, device=dev, emulate=G, full_init={"user": user, "item": item})
    users = np.arange(40)
    got = sh.topk_index(None, 32)(users)
    _same(got, _bf(32, item, user[users], dev))
    ids = got[1].cpu().numpy()
    for b in bounds:                                       # the tied rows appear together, in ascending position
        for r in range(len(users)):
            pos = [j for j in range(32) if b - 2 <= ids[r, j] < b + 2]
            if pos:
                assert list(ids[r, pos]) == sorted(ids[r, pos])


@pytest.mark.parametrize("G", [1, 3])
def test_topk_ratings_and_metrics(dev, G):
    from binrec_b200 import hotpath as H
    from binrec_b200.topKmetrics import topKMetrics, topKRatings
    rng = np.random.default_rng(11)
    users = [int(x) for x in rng.integers(0, NU, 60)]
    items = [int(x) for x in rng.permutation(NI)[:150]]
    positives = [(u, int(i)) for u in users for i in rng.choice(items, 3)]
    exclude = [(u, int(i)) for u in users[:10] for i in rng.choice(items, 5)]
    sh, ref = _neumf_pair(dev, G, 32, True)
    bsh, uw, iw = _bpr_pair(dev, G)

    def lists(vals, idx):
        vals, idx = vals.cpu().numpy(), idx.cpu().numpy()
        return [(u, [(vals[r, j], items[idx[r, j]]) for j in range(idx.shape[1]) if idx[r, j] >= 0])
                for r, u in enumerate(users)]

    from binrec_b200.topKmetrics import exclusion_pairs_csr
    csr = exclusion_pairs_csr(exclude, users, items, dev)
    neumf_idx = ref.topk_index(items)
    bpr_idx = H.BruteForceIndex(10).index(torch.from_numpy(iw[items]).to(dev))
    uq = torch.from_numpy(uw[users]).to(dev)
    for model, mtype, want, want_x in (
            (sh, "NFC", neumf_idx(users, 10), neumf_idx.query_with_exclusions(users, csr, 10)),
            (bsh, None, bpr_idx(uq), bpr_idx.query_with_exclusions(uq, csr))):
        got = topKRatings(10, model, users, items, mtype=mtype)
        assert got == lists(*want)
        assert topKRatings(10, model, users, items, mtype=mtype, exclude=exclude) == lists(*want_x)
        assert topKMetrics(got, positives, users, items, ndcg=True) == topKMetrics(lists(*want), positives, users, items,
                                                                                   ndcg=True)


def test_rejections(dev):
    from binrec_b200.sharded import ShardedBPRNet, ShardedNeuMFNet, ShardedTwoTowerNet
    tc = ShardedNeuMFNet(NU, NI, 32, device=dev, emulate=2, tensor_cores=True)
    fp = ShardedNeuMFNet(NU, NI, 16, device=dev, emulate=2)
    with pytest.raises(ValueError, match="topk_index_fp32"):
        fp.topk_index()
    with pytest.raises(ValueError, match="ShardedNeuMFNet.topk_index"):
        tc.topk_index_fp32()
    with pytest.raises(ValueError, match="no items"):
        tc.topk_index([])
    idx = tc.topk_index()
    users = torch.arange(4, dtype=torch.int32, device=dev)
    for k in (0, 33):
        with pytest.raises(ValueError, match=r"1\.\.32"):
            idx(users, k)
    assert idx(users, 32)[0].shape == (4, 32)
    b = ShardedBPRNet(NU, NI, 64, device=dev, emulate=3)
    with pytest.raises(ValueError, match=r"1\.\.128"):
        b.topk_index(None, 129)
    with pytest.raises(ValueError, match=r"1\.\.128"):
        b.topk_index()(users, 129)
    wide = ShardedBPRNet(NU, NI, 192, device=dev, emulate=2)
    with pytest.raises(ValueError, match=r"1\.\.64"):
        wide.topk_index(None, 65)
    with pytest.raises(ValueError, match=r"1\.\.32"):
        fp.score_all([1, 2], list(range(50)), 40)
    t = ShardedTwoTowerNet(NU, NI, 32, 64, device=dev, emulate=2)
    with pytest.raises(ValueError, match=r"1\.\.128"):
        t.topk_index(None, 200)


# ---- the merge kernel at the C ABI ----------------------------------------------------------------------------------
def _parts(rng, S, U, k, ties):
    """S sorted [U, k] lists (score desc, id asc, (-inf, -1) padded) of random lengths."""
    v = np.full((S, U, k), -np.inf, np.float32)
    ids = np.full((S, U, k), -1, np.int32)
    for s in range(S):
        for u in range(U):
            L = int(rng.integers(0, k + 1))
            ii = rng.integers(0, 1 << 30, L).astype(np.int32)
            if ties:
                ii = rng.integers(0, 3 * k, L).astype(np.int32)      # duplicate ids across and within parts
                vv = rng.integers(0, 3, L).astype(np.float32)
            else:
                vv = rng.standard_normal(L).astype(np.float32)
            o = np.lexsort((ii, -vv))
            v[s, u, :L], ids[s, u, :L] = vv[o], ii[o]
    return v, ids


def _merge_peer(dev, v, ids, hdr, U, k, n_parts=None, err=None):
    from binrec_b200 import _native as N
    S = v.shape[0]
    pv = [torch.from_numpy(np.ascontiguousarray(v[s])).to(dev) for s in range(S)]
    pi = [torch.from_numpy(np.ascontiguousarray(ids[s])).to(dev) for s in range(S)]
    ph = [torch.tensor(h, dtype=torch.int32, device=dev) for h in hdr]
    P = [torch.tensor([t.data_ptr() for t in ts], dtype=torch.int64, device=dev) for ts in (pv, pi, ph)]
    ov = torch.full((max(U, 1), k), 7.0, device=dev)
    oi = torch.full((max(U, 1), k), 7, dtype=torch.int32, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev) if err is None else err
    rc = N.lib().brk_topk_merge_peer(N.ctx(dev), N.ptr(P[0]), N.ptr(P[1]), N.ptr(P[2]), S if n_parts is None else n_parts,
                                     U, k, N.ptr(ov), N.ptr(oi), N.ptr(err), N.stream_ptr())
    torch.cuda.synchronize()
    return rc, ov, oi, int(err.item())


@pytest.mark.parametrize("k", [1, 10, 32, 100, 128])
@pytest.mark.parametrize("S", [1, 3, 8])
@pytest.mark.parametrize("ties", [False, True])
def test_merge_peer_equals_merge(dev, k, S, ties):
    from binrec_b200 import _native as N
    rng = np.random.default_rng(k * 10 + S + ties)
    U = 37
    v, ids = _parts(rng, S, U, k, ties)
    rc, ov, oi, err = _merge_peer(dev, v, ids, [[5, U, k, 0]] * S, U, k)
    assert rc == 0 and err == 0
    pv, pi = torch.from_numpy(v).to(dev), torch.from_numpy(ids).to(dev)
    wv = torch.empty((U, k), device=dev); wi = torch.empty((U, k), dtype=torch.int32, device=dev)
    N.check(N.lib().brk_topk_merge(N.ctx(dev), N.ptr(pv), N.ptr(pi), S, U, k, N.ptr(wv), N.ptr(wi), N.stream_ptr()),
            "brk_topk_merge")
    assert torch.equal(oi, wi) and torch.equal(ov, wv)


def test_merge_peer_headers_and_rejections(dev):
    rng = np.random.default_rng(0)
    U, k, S = 20, 10, 3
    v, ids = _parts(rng, S, U, k, False)
    good = [[9, U, k, 0]] * S
    for s, bad in ((1, [8, U, k, 0]), (2, [9, U + 1, k, 0]), (1, [9, U, k + 1, 0])):   # seq, U, k
        hdr = list(good); hdr[s] = bad
        rc, ov, oi, err = _merge_peer(dev, v, ids, hdr, U, k)
        assert rc == 0 and err == 1 + s
        assert (ov == 7.0).all() and (oi == 7).all()              # no result written
    from binrec_b200 import _native as N
    lib, ctx = N.lib(), N.ctx(dev)
    buf = torch.zeros(64, dtype=torch.int64, device=dev)
    p = N.ptr(buf)
    for args in ((p, p, p, 0, U, k), (p, p, p, 9, U, k), (p, p, p, 3, U, 0), (p, p, p, 3, U, 129), (p, p, p, 3, -1, k),
                 (None, p, p, 3, U, k), (p, p, None, 3, U, k)):
        assert lib.brk_topk_merge_peer(ctx, *args, p, p, p, N.stream_ptr()) == -1
    assert lib.brk_topk_merge_peer(ctx, p, p, p, 3, U, k, p, p, None, N.stream_ptr()) == -1
    assert lib.brk_topk_merge_peer(ctx, p, p, p, 3, 0, k, p, p, p, N.stream_ptr()) == 0     # U = 0 does nothing


# ---- two GPUs -------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


U2, I2 = 1001, 403
QUERY = np.array([0, 5, 5, 999, 400, 17] + list(range(100, 160)), dtype=np.int32)
ITEMS = np.random.default_rng(3).permutation(I2)[:397]


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", device_id=dev)
    try:
        from binrec_b200 import hotpath as H
        from binrec_b200.sharded import ShardedBPRNet, ShardedNeuMFNet, ShardedTopKIndex
        out = {}
        csr = H.exclusion_csr(np.repeat(np.arange(8), 30), np.arange(240) % len(ITEMS), len(QUERY), dev)
        for mode, E, tc in (("peer", 32, True), ("nccl", 16, False)):
            net = ShardedNeuMFNet(U2, I2, E, dropout=0.0, seed=9, device=dev, mode=mode, tensor_cores=tc)
            _train_neumf(net, dev, B=512, seed=4, world=world, rank=rank)
            idx = net.topk_index(ITEMS) if tc else net.topk_index_fp32(ITEMS)
            res = [idx(QUERY, 10), idx.query_with_exclusions(QUERY, csr, 10)]
            ShardedTopKIndex.CHUNK_ENTRIES = 10 * 7                  # several chunks through both slots
            res.append(idx(QUERY, 10))
            ShardedTopKIndex.CHUNK_ENTRIES = 1 << 21
            out[mode] = dict(lists=[(v.cpu().numpy(), i.cpu().numpy()) for v, i in res], bn=idx.bn.cpu().numpy(),
                             dense=net.dense.w.view(-1).cpu().numpy(), peer=idx._bufs is not None,
                             full={n: getattr(net, n).full_weights() for n in ("uMLP", "iMLP", "uMF", "iMF")})
            net.check()
        b = ShardedBPRNet(U2, I2, 64, device=dev)
        rng = np.random.default_rng(21)
        for _ in range(3):
            u, p, n = (rng.integers(0, U2, 2 * 512).astype(np.int32), rng.integers(0, I2, 2 * 512).astype(np.int32),
                       rng.integers(0, I2, 2 * 512).astype(np.int32))
            sl = slice(rank * 512, (rank + 1) * 512)
            b.train_on_batch(*(torch.from_numpy(x[sl]).to(dev) for x in (u, p, n)))
        v, i = b.topk_index(ITEMS, 100)(QUERY)
        out["bpr"] = dict(lists=[(v.cpu().numpy(), i.cpu().numpy())], user=b.user.full_weights(), item=b.item.full_weights())
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def test_two_gpus_peer_nccl_and_bpr():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    dev = torch.device("cuda:0")
    torch.cuda.set_device(0)
    from binrec_b200 import hotpath as H
    r0, r1 = ret[0], ret[1]
    csr = H.exclusion_csr(np.repeat(np.arange(8), 30), np.arange(240) % len(ITEMS), len(QUERY), dev)
    for mode, E, tc in (("peer", 32, True), ("nccl", 16, False)):
        got = r0[mode]
        assert got["peer"] == (mode == "peer")
        for (v0, i0), (v1, i1) in zip(got["lists"], r1[mode]["lists"]):
            assert np.array_equal(v0, v1) and np.array_equal(i0, i1)
        ref = _neumf_reference(dev, E, tc, got["full"], got["dense"], got["bn"], U2, I2)
        idx = ref.topk_index(ITEMS) if tc else ref.topk_index_fp32(ITEMS)
        q = torch.from_numpy(QUERY).to(dev)
        want = [idx(q, 10), idx.query_with_exclusions(q, csr, 10), idx(q, 10)]
        for (v, i), (wv, wi) in zip(got["lists"], want):
            assert np.array_equal(i, wi.cpu().numpy()) and np.array_equal(v, wv.cpu().numpy())
    (v0, i0), = r0["bpr"]["lists"]
    (v1, i1), = r1["bpr"]["lists"]
    assert np.array_equal(v0, v1) and np.array_equal(i0, i1)
    wv, wi = _bf(100, r0["bpr"]["item"][ITEMS], r0["bpr"]["user"][QUERY], dev)
    assert np.array_equal(i0, wi.cpu().numpy()) and np.array_equal(v0, wv.cpu().numpy())
