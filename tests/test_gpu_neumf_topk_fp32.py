"""Full-catalog top-k of the fp32 NeuMF models in one launch (NeuMFNet.topk_index_fp32, brk_neumf_score_topk_fp32 /
_excl, csrc/neumf_topk_fp32.cu).

Scores are held to predict_on_batch of the same pairs at the fp32 prediction tolerance of test_gpu_neumf.py (rtol
1e-5, atol 1e-6) and to oracle/neumf.py run in float64; ids are held gap-aware against the full predict_on_batch
matrix.  Every claim about which users or items share a call, about k, shards, ties and exclusions is bit-exact: a
pair's score depends on the pair alone."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
U_, I_ = 300, 1500


def _script_kw():
    from binrec_b200.NCFModel import SCRIPT_SPEC
    kw = dict(SCRIPT_SPEC)
    return kw.pop("numFactor"), kw


# (numFactor, constructor keywords): fp32 models of every kind the index serves
INSTANCES = {
    "f32": (32, dict()),                                        # the net NeuMFModel.compileModel builds
    "f64": (64, dict()),
    "f7": (7, dict()),                                          # H3 = 1
    "f20": (20, dict()),                                        # H3 = 5
    "f128": (128, dict()),                                      # at the caps
    "script": _script_kw(),                                     # NFC_plain: sigmoid, (100, 50, 10), head mf_h3
    "had16": (16, dict(mf_dim=8, mf_mode="hadamard", batch_norm=False)),   # not in FUSED_VARIANTS
}


def _train(net, dev, steps=4, B=1024, seed=3):
    rng = np.random.default_rng(seed)
    for s in range(steps):
        u = torch.from_numpy(rng.integers(0, net.numUser, B).astype(np.int32)).to(dev)
        i = torch.from_numpy(rng.integers(0, net.numItem, B).astype(np.int32)).to(dev)
        y = torch.from_numpy((rng.random(B) < 0.3).astype(np.float32)).to(dev)
        net.train_on_batch(u, i, y, first_index=s * B)
    torch.cuda.synchronize()


def _make(dev, name, U=U_, I=I_, seed=42, steps=4, B=1024):
    from binrec_b200.NeuMFModel import NeuMFNet
    E, kw = INSTANCES[name]
    kw = dict(kw)
    kw.setdefault("dropout", 0.2)
    net = NeuMFNet(U, I, E, seed=seed, device=dev, **kw)
    assert not net.tensor_cores
    _train(net, dev, steps=steps, B=B)
    return net


@pytest.fixture(scope="module")
def nets(dev):
    """Trained-looking models (a few steps with dropout from the seeded init, so the BatchNorm statistics are not the
    identity)."""
    return {name: _make(dev, name) for name in INSTANCES}


def _scores(net, users, items):
    """Reference score matrix [len(users), len(items)] from predict_on_batch."""
    dev = net.device
    uu = torch.as_tensor(np.asarray(users, dtype=np.int32)).to(dev)
    it = torch.as_tensor(np.asarray(items, dtype=np.int32)).to(dev)
    out, _ = net.predict_on_batch(uu.repeat_interleave(it.numel()), it.repeat(uu.numel()))
    return out.view(uu.numel(), it.numel()).cpu().numpy()


def _oracle_scores(net, users, items):
    """oracle/neumf.py forward in float64 with the model's act, mf_mode and batch_norm."""
    from oracle import neumf as ON
    h = net.hidden
    p = ON.NeuMFParams(2, 2, net.E, h, dtype=torch.float64, mf_dim=net.EMF, mf_mode=net.mf_mode, batch_norm=net.batch_norm)
    for name, t in (("uMLP", net.uMLP), ("iMLP", net.iMLP), ("uMF", net.uMF), ("iMF", net.iMF)):
        p.t[name] = t.w.detach().cpu().double()
    for name in ON.NeuMFParams.DENSE:
        p.t[name] = net.param(name).detach().cpu().double()
    bn = net.bn_moving.cpu().double()
    p.mm1, p.mv1, p.mm2, p.mv2 = bn[:h[0]], bn[h[0]:2 * h[0]], bn[2 * h[0]:2 * h[0] + h[1]], bn[2 * h[0] + h[1]:]
    uu = np.repeat(np.asarray(users), len(items)); ii = np.tile(np.asarray(items), len(users))
    with torch.no_grad():
        out, _ = ON.forward(p, uu, ii, training=False, act=net.act)
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


TOL = lambda x: RTOL * abs(x) + 2 * ATOL


@pytest.mark.parametrize("name", list(INSTANCES))
def test_matches_model_and_fp64_oracle(dev, nets, name):
    net = nets[name]
    users = np.arange(0, U_, 3)
    items = np.arange(I_)
    k = 10
    vals, ids = net.topk_index_fp32()(users, k)
    vals, ids = vals.cpu().numpy(), ids.cpu().numpy()
    assert (np.diff(vals, axis=1) <= 0).all()
    ref = _scores(net, users, items)
    _check_gap_aware(vals, ids, ref, k, TOL)
    orc = _oracle_scores(net, users, items)
    for r in range(len(users)):
        np.testing.assert_allclose(vals[r], orc[r, ids[r]], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("name", ["f32", "script", "had16"])
def test_launch_independence(dev, nets, name):
    from binrec_b200 import hotpath as H
    net = nets[name]
    index = net.topk_index_fp32()
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
    # item-range shards with id_offset (odd bounds: items change their place in the chunks), merged
    for n in (2, 3, 8):
        bounds = np.linspace(0, I_, n + 1).astype(int)
        bounds[1:-1] += 1
        pv, pi = [], []
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            a, b = net.topk_index_fp32(np.arange(lo, hi), id_offset=int(lo))(users, 10)
            pv.append(a); pi.append(b)
        mv, mi = H.topk_merge(torch.stack(pv), torch.stack(pi))
        assert torch.equal(mv, v) and torch.equal(mi, i), n


@pytest.mark.parametrize("name", ["f32", "script"])
def test_ties_go_to_the_lower_id(dev, name):
    from binrec_b200 import hotpath as H
    net = _make(dev, name, U=64, I=400, seed=5, steps=2)
    # items 2j and 2j+1 share their iMLP and iMF rows; so do 2j+1 and 2j+2 of the shifted index below
    with torch.no_grad():
        net.iMLP.w[1::2] = net.iMLP.w[0::2]
        net.iMF.w[1::2] = net.iMF.w[0::2]
    users = np.array([0, 5, 5, 9], dtype=np.int32)
    v, i = net.topk_index_fp32()(users, 16)
    vn, inn = v.cpu().numpy(), i.cpu().numpy()
    for r in range(len(users)):
        for j in range(0, 16, 2):
            assert inn[r, j] % 2 == 0 and inn[r, j + 1] == inn[r, j] + 1 and vn[r, j] == vn[r, j + 1], (r, j)
    assert (vn[1] == vn[2]).all() and (inn[1] == inn[2]).all()
    # the equal pairs at odd positions (items 1..399 indexed from position 0): each pair shares a kernel step or sits
    # across steps and chunks
    sh = net.topk_index_fp32(np.arange(1, 400), id_offset=1)
    vs, is_ = sh(users, 16)
    vs, is_ = vs.cpu().numpy(), is_.cpu().numpy()
    for r in range(len(users)):
        for j in range(16):
            partner = is_[r, j] ^ 1
            if 1 <= partner < 400 and partner in is_[r]:
                q = list(is_[r]).index(partner)
                assert vs[r, q] == vs[r, j] and (q < j) == (partner < is_[r, j]), (r, j)
    # a tied pair straddling a split boundary: shards [0, 2j+1) and [2j+1, 400), merged
    for cut in (33, 65, 201):
        lo = net.topk_index_fp32(np.arange(0, cut))(users, 16)
        hi = net.topk_index_fp32(np.arange(cut, 400), id_offset=cut)(users, 16)
        mv, mi = H.topk_merge(torch.stack([lo[0], hi[0]]), torch.stack([lo[1], hi[1]]))
        assert torch.equal(mv, v) and torch.equal(mi, i), cut


def test_exclusions(dev, nets):
    from binrec_b200 import hotpath as H
    for name in ("script", "f20"):
        net = nets[name]
        index = net.topk_index_fp32()
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
            rows += [r, r]; its += [I_ + 5, I_ + 1000]                # outside [0, I): ignored
        csr = H.exclusion_csr(rows, its, U_, dev)
        vx, ix = index.query_with_exclusions(users, csr, 10)
        indptr, xid = csr[0].cpu().numpy(), csr[1].cpu().numpy()
        v32n = v32.cpu().numpy()
        for r in range(U_):
            gone = set(xid[indptr[r]:indptr[r + 1]].tolist())
            keep = [j for j in range(32) if i32n[r, j] not in gone][:10]
            assert ix[r].cpu().numpy().tolist() == i32n[r, keep].tolist(), (name, r)
            assert vx[r].cpu().numpy().tolist() == v32n[r, keep].tolist(), (name, r)
        # a shard's range: ids of other shards are ignored
        shard = net.topk_index_fp32(np.arange(500, 900), id_offset=500)
        vs, is_ = shard(users[:40], 10)
        rows = np.repeat(np.arange(40), 3)
        its = np.stack([is_[:, 0].cpu().numpy(), np.full(40, 10), np.full(40, 1400)], 1).ravel()
        vsx, isx = shard.query_with_exclusions(users[:40], H.exclusion_csr(rows, its, 40, dev), 10)
        assert torch.equal(isx[:, :9], is_[:, 1:]) and torch.equal(vsx[:, :9], vs[:, 1:])
        # rows left with fewer than k items: padded with (-inf, -1); a fully excluded row is all (-inf, -1)
        small = net.topk_index_fp32(np.arange(12))
        rows = np.concatenate([np.repeat(np.arange(3), 5), np.full(12, 3)])
        its = np.concatenate([np.tile(np.arange(5), 3), np.arange(12)])
        vp, ip = small.query_with_exclusions(users[:4], H.exclusion_csr(rows, its, 4, dev), 10)
        assert (ip[:3, 7:] == -1).all() and torch.isinf(vp[:3, 7:]).all() and (vp[:3, 7:] < 0).all()
        assert set(ip[0, :7].cpu().numpy().tolist()) == set(range(5, 12))
        assert (ip[3] == -1).all() and torch.isinf(vp[3]).all() and (vp[3] < 0).all()


@pytest.mark.parametrize("name,U,I", [("f32", 1, 1), ("f32", 129, 37), ("f32", 5, 3), ("script", 1, 2000),
                                      ("script", 257, 131), ("f7", 130, 9), ("had16", 200, 257), ("f128", 131, 70)])
def test_shapes(dev, nets, name, U, I):
    net = nets[name]
    users = np.arange(U, dtype=np.int32) % U_
    items = np.arange(I) * 7 % I_
    k = 10
    v, i = net.topk_index_fp32(items)(users, k)
    assert v.shape == (U, min(k, I))
    ref = _scores(net, users, items)
    _check_gap_aware(v.cpu().numpy(), i.cpu().numpy(), ref, min(k, I), TOL)


@pytest.mark.parametrize("name", ["f32", "script"])
def test_full_size(dev, name):
    U, I = 6040, 3706
    net = _make(dev, name, U=U, I=I, seed=7, steps=3, B=4096)
    v, i = net.topk_index_fp32()(np.arange(U), 10)
    sample = np.random.default_rng(0).choice(U, 24, replace=False)
    ref = _scores(net, sample, np.arange(I))
    _check_gap_aware(v[sample].cpu().numpy(), i[sample].cpu().numpy(), ref, 10, TOL)


def test_rejections(dev, nets):
    from binrec_b200 import _native as N
    from binrec_b200.NeuMFModel import NeuMFNet
    # Python: tensor-core nets point to topk_index, widths beyond the caps to score_all, and topk_index keeps
    # rejecting fp32 nets
    tc = NeuMFNet(16, 40, 32, device=dev, tensor_cores=True)
    with pytest.raises(ValueError, match="topk_index"):
        tc.topk_index_fp32()
    for kw in (dict(hidden=(129, 16, 8)), dict(hidden=(32, 65, 8)), dict(hidden=(32, 16, 33)), dict(mf_dim=129)):
        with pytest.raises(ValueError, match="score_all"):
            NeuMFNet(16, 40, 32, device=dev, **kw).topk_index_fp32()
    with pytest.raises(ValueError, match="score_all"):
        nets["f32"].topk_index()
    net = nets["f32"]
    index = net.topk_index_fp32()
    with pytest.raises(ValueError, match="score_all"):
        index(np.arange(4), 33)
    # the C ABI
    lib, ctx = N.lib(), N.ctx(dev)
    m = net._c_model()
    H1 = net.hidden[0]
    A = torch.zeros((4, H1), device=dev); users = torch.zeros(4, dtype=torch.int32, device=dev)
    B = index.item_side; M = index.item_mf
    I = B.shape[0]
    ov = torch.empty((4, 10), device=dev); oi = torch.empty((4, 10), dtype=torch.int32, device=dev)
    ws_bytes = lib.brk_neumf_topk_fp32_workspace_bytes(ctx, C.byref(m), 4, I, 10)
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

    def call(k=10, wsb=ws_bytes, model=m, U=4, I=I, a=A, b=B):
        return lib.brk_neumf_score_topk_fp32(ctx, C.byref(model), N.ptr(a) if a is not None else None, N.ptr(users), U,
                                             N.ptr(b) if b is not None else None, N.ptr(M), I, k, 0, N.ptr(ov), N.ptr(oi),
                                             N.ptr(ws), wsb, N.stream_ptr())

    assert call() == 0
    assert call(U=0) == 0
    assert call(k=33) == -1 and b"k=33" in lib.brk_last_error()
    assert call(k=0) == -1
    assert call(wsb=ws_bytes - 8) == -1 and b"workspace" in lib.brk_last_error()
    assert call(U=-1) == -1
    assert call(I=0) == -1
    assert call(a=None) == -1 and b"null" in lib.brk_last_error()
    assert call(b=None) == -1
    m_tc = net._c_model(); m_tc.tensor_cores = 1
    assert call(model=m_tc) == -1 and b"brk_neumf_score_topk" in lib.brk_last_error()
    for field, value in (("H1", 129), ("H2", 65), ("H3", 33), ("EMF", 129)):
        mw = net._c_model(); setattr(mw, field, value)
        assert call(model=mw) == -1 and b"score_all" in lib.brk_last_error(), field
    assert lib.brk_neumf_score_topk_fp32_excl(ctx, C.byref(m), N.ptr(A), N.ptr(users), 4, N.ptr(B), N.ptr(M), I, 10, 0,
                                              None, None, N.ptr(ov), N.ptr(oi), N.ptr(ws), ws_bytes, N.stream_ptr()) == -1
    assert b"exclusion" in lib.brk_last_error()
    torch.cuda.synchronize()
