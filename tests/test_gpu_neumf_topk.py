"""Full-catalog NeuMF top-k in one launch (NeuMFNet.topk_index, brk_neumf_score_topk / _excl, csrc/neumf_topk.cu).

Scores are held to predict_on_batch of the same pairs and to oracle/neumf.py with TF32 products at the tensor-core
prediction tolerance (rtol 2e-3, atol 1e-5); ids are held gap-aware against the full reference score matrix.  Every
claim about which users or items share a call, about k, shards, ties and exclusions is bit-exact: a pair's score
depends on the pair alone."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 2e-3, 1e-5
U_, I_ = 300, 1500

# (numFactor, constructor keywords): the three built instances
INSTANCES = {
    "f32": (32, dict(tensor_cores=True)),
    "f64": (64, dict(tensor_cores=True)),
    "he": (32, dict(mf_dim=8, mf_mode="hadamard", batch_norm=False, hidden=(32, 16, 8))),
}


def _train(net, dev, steps=4, B=1024, seed=3):
    rng = np.random.default_rng(seed)
    for s in range(steps):
        u = torch.from_numpy(rng.integers(0, net.numUser, B).astype(np.int32)).to(dev)
        i = torch.from_numpy(rng.integers(0, net.numItem, B).astype(np.int32)).to(dev)
        y = torch.from_numpy((rng.random(B) < 0.3).astype(np.float32)).to(dev)
        net.train_on_batch(u, i, y, first_index=s * B)
    torch.cuda.synchronize()


@pytest.fixture(scope="module")
def nets(dev):
    """Trained-looking models (a few steps from the seeded init, so the BatchNorm statistics are not identity)."""
    from binrec_b200.NeuMFModel import NeuMFNet
    out = {}
    for name, (E, kw) in INSTANCES.items():
        net = NeuMFNet(U_, I_, E, dropout=0.2, seed=42, device=dev, **kw)
        _train(net, dev)
        out[name] = net
    return out


def _scores(net, users, items):
    """Reference score matrix [len(users), len(items)] from predict_on_batch."""
    dev = net.device
    uu = torch.as_tensor(np.asarray(users, dtype=np.int32)).to(dev)
    it = torch.as_tensor(np.asarray(items, dtype=np.int32)).to(dev)
    out, _ = net.predict_on_batch(uu.repeat_interleave(it.numel()), it.repeat(uu.numel()))
    return out.view(uu.numel(), it.numel()).cpu().numpy()


def _oracle_scores(net, users, items):
    from oracle import neumf as ON
    from oracle import tf32 as OT32
    h = net.hidden
    p = ON.NeuMFParams(net.numUser, net.numItem, net.E, h, mf_dim=net.EMF, mf_mode=net.mf_mode, batch_norm=net.batch_norm)
    for name, t in (("uMLP", net.uMLP), ("iMLP", net.iMLP), ("uMF", net.uMF), ("iMF", net.iMF)):
        p.t[name] = t.w.detach().cpu().clone()
    for name in ON.NeuMFParams.DENSE:
        p.t[name] = net.param(name).detach().cpu().clone()
    bn = net.bn_moving.cpu()
    p.mm1, p.mv1, p.mm2, p.mv2 = bn[:h[0]], bn[h[0]:2 * h[0]], bn[2 * h[0]:2 * h[0] + h[1]], bn[2 * h[0] + h[1]:]
    uu = np.repeat(np.asarray(users), len(items)); ii = np.tile(np.asarray(items), len(users))
    with torch.no_grad():
        out, _ = ON.forward(p, uu, ii, training=False, act="relu", matmul=OT32.matmul)
    return out.numpy().reshape(len(users), len(items))


def _check_gap_aware(vals, ids, ref, k, tol_fn):
    """Every returned id's reference score >= the reference k-th best - tol; where the k-th / (k+1)-th reference gap
    exceeds tol, the id set is exact; returned scores equal the reference scores of their ids."""
    for r in range(ref.shape[0]):
        row = ref[r]
        order = np.argsort(-row, kind="stable")
        kth = row[order[k - 1]]
        tol = tol_fn(kth)
        got = ids[r]
        assert (got >= 0).all()
        assert (row[got] >= kth - tol).all(), r
        np.testing.assert_allclose(vals[r], row[got], rtol=RTOL, atol=ATOL)
        if k < len(row) and kth - row[order[k]] > tol:
            assert set(got.tolist()) == set(order[:k].tolist()), r


@pytest.mark.parametrize("name", list(INSTANCES))
def test_matches_model_and_tf32_oracle(dev, nets, name):
    net = nets[name]
    users = np.arange(0, U_, 3)
    items = np.arange(I_)
    k = 10
    vals, ids = net.topk_index()(users, k)
    vals, ids = vals.cpu().numpy(), ids.cpu().numpy()
    assert (np.diff(vals, axis=1) <= 0).all()
    ref = _scores(net, users, items)
    tol = lambda x: RTOL * abs(x) + 2 * ATOL
    _check_gap_aware(vals, ids, ref, k, tol)
    orc = _oracle_scores(net, users, items)
    for r in range(len(users)):
        np.testing.assert_allclose(vals[r], orc[r, ids[r]], rtol=RTOL, atol=ATOL)


def test_launch_independence(dev, nets):
    from binrec_b200 import hotpath as H
    net = nets["f32"]
    index = net.topk_index()
    users = np.arange(U_, dtype=np.int32)
    v, i = index(users, 10)
    # permuted and duplicated users
    perm = np.random.default_rng(1).permutation(U_)
    dup = np.concatenate([perm, perm[:50]])
    v2, i2 = index(dup, 10)
    assert torch.equal(v2[:U_], v[perm]) and torch.equal(i2[:U_], i[perm])
    assert torch.equal(v2[U_:], v[perm[:50]]) and torch.equal(i2[U_:], i[perm[:50]])
    # subsets
    sub = users[7:20]
    v3, i3 = index(sub, 10)
    assert torch.equal(v3, v[7:20]) and torch.equal(i3, i[7:20])
    # k = 10 against the first 10 of k = 32
    v4, i4 = index(users, 32)
    assert torch.equal(v4[:, :10], v) and torch.equal(i4[:, :10], i)
    # item-range shards with id_offset, merged
    for n in (2, 3, 8):
        bounds = np.linspace(0, I_, n + 1).astype(int)
        pv, pi = [], []
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            a, b = net.topk_index(np.arange(lo, hi), id_offset=int(lo))(users, 10)
            pv.append(a); pi.append(b)
        mv, mi = H.topk_merge(torch.stack(pv), torch.stack(pi))
        assert torch.equal(mv, v) and torch.equal(mi, i), n


def test_ties_go_to_the_lower_id(dev):
    from binrec_b200.NeuMFModel import NeuMFNet
    net = NeuMFNet(64, 400, 32, dropout=0.2, seed=5, device=dev, tensor_cores=True)
    _train(net, dev, steps=2)
    # items 2j and 2j+1 share their iMLP and iMF rows
    with torch.no_grad():
        net.iMLP.w[1::2] = net.iMLP.w[0::2]
        net.iMF.w[1::2] = net.iMF.w[0::2]
    users = np.array([0, 5, 5, 9], dtype=np.int32)
    v, i = net.topk_index()(users, 16)
    v, i = v.cpu().numpy(), i.cpu().numpy()
    for r in range(len(users)):
        for j in range(0, 16, 2):
            assert i[r, j] % 2 == 0 and i[r, j + 1] == i[r, j] + 1 and v[r, j] == v[r, j + 1], (r, j)
    assert (v[1] == v[2]).all() and (i[1] == i[2]).all()


def test_exclusions(dev, nets):
    from binrec_b200 import hotpath as H
    net = nets["he"]
    index = net.topk_index()
    users = np.arange(U_, dtype=np.int32)
    v10, i10 = index(users, 10)
    v32, i32 = index(users, 32)
    # empty lists: the call without exclusions
    empty = H.exclusion_csr([], [], U_, dev)
    ve, ie = index.query_with_exclusions(users, empty, 10)
    assert torch.equal(ve, v10) and torch.equal(ie, i10)
    # lists that remove some of each row's top items (at most 32 - k), plus ids outside the range
    rng = np.random.default_rng(2)
    i32n = i32.cpu().numpy()
    rows, its = [], []
    for r in range(U_):
        drop = rng.choice(20, size=int(rng.integers(0, 21)), replace=False)
        rows += [r] * len(drop); its += i32n[r, drop].tolist()
        rows += [r, r]; its += [I_ + 5, I_ + 1000]                    # outside [0, I): ignored
    csr = H.exclusion_csr(rows, its, U_, dev)
    vx, ix = index.query_with_exclusions(users, csr, 10)
    indptr, xid = csr[0].cpu().numpy(), csr[1].cpu().numpy()
    v32n = v32.cpu().numpy()
    for r in range(U_):
        gone = set(xid[indptr[r]:indptr[r + 1]].tolist())
        keep = [j for j in range(32) if i32n[r, j] not in gone][:10]
        assert ix[r].cpu().numpy().tolist() == i32n[r, keep].tolist(), r
        assert vx[r].cpu().numpy().tolist() == v32n[r, keep].tolist(), r
    # a shard's range: ids of other shards are ignored
    shard = net.topk_index(np.arange(500, 900), id_offset=500)
    vs, is_ = shard(users[:40], 10)
    rows = np.repeat(np.arange(40), 3); its = np.stack([is_[:, 0].cpu().numpy(), np.full(40, 10), np.full(40, 1400)], 1).ravel()
    vsx, isx = shard.query_with_exclusions(users[:40], H.exclusion_csr(rows, its, 40, dev), 10)
    assert torch.equal(isx[:, :9], is_[:, 1:]) and torch.equal(vsx[:, :9], vs[:, 1:])
    # rows left with fewer than k items: padded with (-inf, -1)
    small = net.topk_index(np.arange(12))
    rows = np.repeat(np.arange(4), 5); its = np.tile(np.arange(5), 4)
    vp, ip = small.query_with_exclusions(users[:4], H.exclusion_csr(rows, its, 4, dev), 10)
    assert (ip[:, 7:] == -1).all() and torch.isinf(vp[:, 7:]).all() and (vp[:, 7:] < 0).all()
    assert set(ip[0, :7].cpu().numpy().tolist()) == set(range(5, 12))


@pytest.mark.parametrize("name,U,I", [("f32", 1, 1), ("f32", 129, 37), ("f32", 5, 3), ("he", 257, 131), ("f64", 130, 257)])
def test_shapes(dev, nets, name, U, I):
    net = nets[name]
    users = np.arange(U, dtype=np.int32) % U_
    items = np.arange(I) * 7 % I_
    k = 10
    v, i = net.topk_index(items)(users, k)
    assert v.shape == (U, min(k, I))
    ref = _scores(net, users, items)
    _check_gap_aware(v.cpu().numpy(), i.cpu().numpy(), ref, min(k, I), lambda x: RTOL * abs(x) + 2 * ATOL)


@pytest.mark.parametrize("name,E,kw,U,I", [
    ("ml1m-f32", 32, dict(tensor_cores=True), 6040, 3706),
    ("ml1m-he", 32, dict(mf_dim=8, mf_mode="hadamard", batch_norm=False, hidden=(32, 16, 8)), 6040, 3706),
    ("f64-50k", 64, dict(tensor_cores=True), 1000, 50000),
])
def test_full_size(dev, name, E, kw, U, I):
    from binrec_b200.NeuMFModel import NeuMFNet
    net = NeuMFNet(U, I, E, dropout=0.2, seed=7, device=dev, **kw)
    _train(net, dev, steps=3, B=4096)
    v, i = net.topk_index()(np.arange(U), 10)
    sample = np.random.default_rng(0).choice(U, 24, replace=False)
    ref = _scores(net, sample, np.arange(I))
    _check_gap_aware(v[sample].cpu().numpy(), i[sample].cpu().numpy(), ref, 10, lambda x: RTOL * abs(x) + 2 * ATOL)


def test_rejections(dev, nets):
    from binrec_b200 import _native as N
    from binrec_b200.NeuMFModel import NeuMFNet
    for kw in (dict(), dict(tensor_cores=True, act="sigmoid"), dict(hidden=(32, 8, 8), tensor_cores=False)):
        net = NeuMFNet(16, 40, 32, device=dev, **kw)
        with pytest.raises(ValueError, match="score_all"):
            net.topk_index()
    net = nets["f32"]
    index = net.topk_index()
    with pytest.raises(ValueError, match="score_all"):
        index(np.arange(4), 33)
    # bad arguments at the C ABI
    lib, ctx = N.lib(), N.ctx(dev)
    m = net._c_model()
    A = torch.zeros((4, 32), device=dev); users = torch.zeros(4, dtype=torch.int32, device=dev)
    B = index.item_side; M = index.item_mf
    ov = torch.empty((4, 10), device=dev); oi = torch.empty((4, 10), dtype=torch.int32, device=dev)
    ws_bytes = lib.brk_neumf_topk_workspace_bytes(ctx, 4, B.shape[0], 10)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    args = lambda k, wsb, model: (ctx, C.byref(model), N.ptr(A), N.ptr(users), 4, N.ptr(B), N.ptr(M), B.shape[0], k, 0,
                                  N.ptr(ov), N.ptr(oi), N.ptr(ws), wsb, N.stream_ptr())
    assert lib.brk_neumf_score_topk(*args(10, ws_bytes, m)) == 0
    assert lib.brk_neumf_score_topk(*args(33, ws_bytes, m)) == -1
    assert lib.brk_neumf_score_topk(*args(0, ws_bytes, m)) == -1
    assert lib.brk_neumf_score_topk(*args(10, ws_bytes - 8, m)) == -1
    m2 = net._c_model(); m2.H2 = 8
    assert lib.brk_neumf_score_topk(*args(10, ws_bytes, m2)) == -1
    assert b"built" in lib.brk_last_error()
    m3 = net._c_model(); m3.tensor_cores = 0
    assert lib.brk_neumf_score_topk(*args(10, ws_bytes, m3)) == -1
    assert lib.brk_neumf_score_topk_excl(ctx, C.byref(m), N.ptr(A), N.ptr(users), 4, N.ptr(B), N.ptr(M), B.shape[0], 10, 0,
                                         None, None, N.ptr(ov), N.ptr(oi), N.ptr(ws), ws_bytes, N.stream_ptr()) == -1
    torch.cuda.synchronize()
