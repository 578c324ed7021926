"""Per-row exclusions in full-catalog top-K (BruteForceIndex.query_with_exclusions, brk_score_topk_bf16_excl,
brk_mask_excluded) against a CPU definition of the semantics:

for query row r with excluded global ids X_r, the result is the first k candidates not in X_r whose score is > -inf,
by descending score with ties to the lower id, padded with (-inf, -1).  Ids of X_r outside the call's range
[id_offset, id_offset + I) and duplicates are ignored.

Bit-exact claims use exact-arithmetic inputs (entries j/8, |j| <= 4), as in test_gpu_topk.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import topk as OT


def topk_excluding(S, k, indptr, ids, id_offset=0):
    """(vals [U,k], ids [U,k]) of score rows S [U, I] (local columns; global id = column + id_offset) with row r's
    listed ids ids[indptr[r]:indptr[r+1]] left out; (-inf, -1) pads."""
    S = np.asarray(S, dtype=np.float32)
    U, I = S.shape
    k = min(k, I)
    ov = np.full((U, k), -np.inf, dtype=np.float32)
    oi = np.full((U, k), -1, dtype=np.int32)
    for r in range(U):
        s = S[r].copy()
        lst = np.asarray(ids[indptr[r]:indptr[r + 1]], dtype=np.int64) - id_offset
        s[lst[(lst >= 0) & (lst < I)]] = -np.inf
        order = np.argsort(-s, kind="stable")
        order = order[s[order] > -np.inf][:k]
        ov[r, :len(order)] = s[order]
        oi[r, :len(order)] = order + id_offset
    return ov, oi


def _literal(S, k, indptr, ids, id_offset=0):
    """The definition spelled out: filter the row, then the reference's streaming insertion."""
    U, I = S.shape
    out = []
    for r in range(U):
        X = set(int(x) for x in ids[indptr[r]:indptr[r + 1]])
        row = [(float(S[r, j]), j + id_offset) for j in range(I) if j + id_offset not in X and S[r, j] > -np.inf]
        out.append(OT.topk_insert_reference(row, k) if row else [])
    return out


def test_topk_excluding_matches_the_literal_definition():
    rng = np.random.default_rng(0)
    for U, I, k, off in ((7, 40, 5, 0), (9, 13, 13, 100), (5, 30, 1, 7)):
        S = (rng.integers(-6, 7, size=(U, I)) / 4.0).astype(np.float32)        # heavy ties
        S[0, :3] = -np.inf
        lists = [sorted(set(rng.integers(off - 5, off + I + 5, size=rng.integers(0, I)).tolist())) for _ in range(U)]
        lists[1] = list(range(off, off + I))                                     # everything excluded
        indptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
        ids = np.asarray([x for l in lists for x in l], dtype=np.int32)
        v, i = topk_excluding(S, k, indptr, ids, off)
        for r, ref in enumerate(_literal(S, k, indptr, ids, off)):
            n = len(ref)
            assert [x for _, x in ref] == i[r, :n].tolist() and [x for x, _ in ref] == v[r, :n].tolist()
            assert (i[r, n:] == -1).all() and np.isneginf(v[r, n:]).all()


# ---------------------------------------------------------------------------------------------------------------------
def H():
    from binrec_b200 import hotpath
    return hotpath


def _exact(rng, rows, d):
    return (rng.integers(-4, 5, size=(rows, d)) / 8.0).astype(np.float32)


def _csr(lists):
    indptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
    ids = np.asarray([x for l in lists for x in l] or [0], dtype=np.int32)
    return indptr, ids


def _dev(csr, dev):
    return torch.from_numpy(csr[0]).to(dev), torch.from_numpy(csr[1]).to(dev)


def _patterns(rng, U, I, k, S):
    """Per row: empty, one id, many, all but fewer than k (pads), every item."""
    lists = []
    for r in range(U):
        p = r % 5
        if p == 0:
            lists.append([])
        elif p == 1:
            lists.append([int(np.argmax(S[r]))])                       # the row's best item
        elif p == 2:
            lists.append(sorted(rng.choice(I, size=I // 3, replace=False).tolist()))
        elif p == 3:
            keep = set(rng.choice(I, size=max(k - 1, 0), replace=False).tolist())
            lists.append([j for j in range(I) if j not in keep])
        else:
            lists.append(list(range(I)))
    return lists


def _check(v, i, rv, ri):
    assert np.array_equal(i.cpu().numpy(), ri)
    assert np.array_equal(v.cpu().numpy(), rv)


@pytest.mark.gpu
@pytest.mark.parametrize("U,I,d,k", [(37, 1000, 16, 1), (200, 777, 64, 3), (300, 3706, 128, 10), (5, 5000, 200, 16),
                                     (130, 1030, 64, 32), (257, 2000, 128, 10), (1000, 300, 64, 16), (3, 20000, 16, 32)])
def test_exclusions_bit_exact(dev, U, I, d, k):
    rng = np.random.default_rng(U * 13 + I + k)
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    csr = _csr(_patterns(rng, U, I, k, S))
    rv, ri = topk_excluding(S, k, *csr)
    idx = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev))
    v, i = idx.query_with_exclusions(torch.from_numpy(Q).to(dev), _dev(csr, dev))
    _check(v, i, rv, ri)


@pytest.mark.gpu
def test_excluding_each_rows_own_best(dev):
    """The worst case: every row excludes its own true top-m, so every excluded item beats the running threshold.
    The result is the oracle's ranks m .. m+k-1, padded where the catalog runs out."""
    rng = np.random.default_rng(1)
    U, I, d, k = 150, 1300, 64, 10
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    fv, fi = OT.topk_from_scores(S, I)
    idx = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev))
    Qd = torch.from_numpy(Q).to(dev)
    for m in (1, 5, 40, 600, I - 4):
        csr = _csr([sorted(fi[r, :m].tolist()) for r in range(U)])
        v, i = idx.query_with_exclusions(Qd, _dev(csr, dev))
        n = min(k, I - m)
        rv = np.full((U, k), -np.inf, np.float32); ri = np.full((U, k), -1, np.int32)
        rv[:, :n] = fv[:, m:m + n]; ri[:, :n] = fi[:, m:m + n]
        _check(v, i, rv, ri)


@pytest.mark.gpu
def test_ignored_ids_change_nothing(dev):
    rng = np.random.default_rng(2)
    U, I, d, k = 70, 900, 64, 10
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    base = [sorted(rng.choice(I, size=rng.integers(0, 50), replace=False).tolist()) for _ in range(U)]
    rv, ri = topk_excluding(S, k, *_csr(base))
    noisy = [sorted([-7, -1] + l + l[:3] + [I, I + 5, 1 << 30]) for l in base]      # out of range + duplicates
    idx = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev))
    _check(*idx.query_with_exclusions(torch.from_numpy(Q).to(dev), _dev(_csr(noisy), dev)), rv, ri)
    # an item-range shard ignores ids outside its range
    lo, hi = 300, 700
    sv, si = topk_excluding(S[:, lo:hi], k, *_csr(base), id_offset=lo)
    sh = H().BruteForceIndex(k).index(torch.from_numpy(Cm[lo:hi]).to(dev), id_offset=lo)
    _check(*sh.query_with_exclusions(torch.from_numpy(Q).to(dev), _dev(_csr(noisy), dev)), sv, si)


@pytest.mark.gpu
def test_shards_with_one_global_list_merge_to_the_unsharded_result(dev):
    rng = np.random.default_rng(3)
    U, I, d, k = 333, 2048, 64, 10
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    csr = _csr(_patterns(rng, U, I, k, S))
    rv, ri = topk_excluding(S, k, *csr)
    Qd, ex = torch.from_numpy(Q).to(dev), _dev(csr, dev)
    bounds = [0, 500, 1100, 1101, 2048]
    pv, pi = [], []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        v, i = H().BruteForceIndex(k).index(torch.from_numpy(Cm[lo:hi]).to(dev), id_offset=lo).query_with_exclusions(Qd, ex)
        if v.shape[1] < k:                                              # a shard narrower than k: pad to k for the merge
            v = torch.cat([v, torch.full((U, k - v.shape[1]), float("-inf"), device=dev)], 1)
            i = torch.cat([i, torch.full((U, k - i.shape[1]), -1, dtype=torch.int32, device=dev)], 1)
        pv.append(v); pi.append(i)
    _check(*H().topk_merge(torch.stack(pv), torch.stack(pi)), rv, ri)
    from binrec_b200 import distributed as D
    _check(*D.sharded_topk(Qd, torch.from_numpy(Cm).to(dev), 0, k, exclude=ex), rv, ri)


@pytest.mark.gpu
def test_row_chunks_with_an_indptr_view(dev):
    rng = np.random.default_rng(4)
    U, I, d, k = 400, 1500, 128, 16
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    indptr, ids = _dev(_csr(_patterns(rng, U, I, k, S)), dev)
    idx = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev))
    Qd = torch.from_numpy(Q).to(dev)
    fv, fi = idx.query_with_exclusions(Qd, (indptr, ids))
    for s0, s1 in ((0, 128), (128, 129), (129, 400), (251, 390)):
        v, i = idx.query_with_exclusions(Qd[s0:s1], (indptr[s0:s1 + 1], ids))
        assert torch.equal(v, fv[s0:s1]) and torch.equal(i, fi[s0:s1])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 33])
def test_empty_exclusions_equal_the_plain_call(dev, k):
    rng = np.random.default_rng(5)
    Q = torch.from_numpy(rng.standard_normal((500, 64)).astype(np.float32)).to(dev)
    Cm = torch.from_numpy(rng.standard_normal((3706, 64)).astype(np.float32)).to(dev)
    idx = H().BruteForceIndex(k).index(Cm)
    v0, i0 = idx(Q)
    empty = (torch.zeros(501, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev))
    v, i = idx.query_with_exclusions(Q, empty)
    assert torch.equal(v, v0) and torch.equal(i, i0)


@pytest.mark.gpu
def test_lists_longer_than_32_with_exclusions(dev):
    rng = np.random.default_rng(6)
    U, I, d = 37, 500, 64
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    for k in (33, 100):
        csr = _csr(_patterns(rng, U, I, k, S))
        rv, ri = topk_excluding(S, k, *csr)
        idx = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev))
        _check(*idx.query_with_exclusions(torch.from_numpy(Q).to(dev), _dev(csr, dev)), rv, ri)
        Sd = torch.from_numpy(S).to(dev)
        _check(*H().topk_rows(Sd, k, exclude=_dev(csr, dev)), rv, ri)
        assert torch.equal(Sd, torch.from_numpy(S).to(dev))             # the input is left as it was
    # an offset shard on the materialised route
    csr = _csr(_patterns(rng, U, I, 40, S))
    rv, ri = topk_excluding(S[:, 100:], 40, *csr, id_offset=100)
    idx = H().BruteForceIndex(40).index(torch.from_numpy(Cm[100:]).to(dev), id_offset=100)
    _check(*idx.query_with_exclusions(torch.from_numpy(Q).to(dev), _dev(csr, dev)), rv, ri)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [7, 40])
def test_dense_identifier_form_equals_the_csr_form(dev, k):
    rng = np.random.default_rng(7)
    U, I, d, n = 60, 300, 16, 25
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    idents = torch.from_numpy(rng.permutation(I).astype(np.int64) * 3 + 1000).to(dev)
    cand = np.stack([rng.choice(I, size=n, replace=False) for _ in range(U)])
    cand[::4, 5:] = -1                                                  # -1 padding
    cand[1::4] = -1                                                     # rows with nothing to exclude
    cand[2, 0] = -1
    dense = torch.where(torch.from_numpy(cand).to(dev) >= 0, idents[torch.from_numpy(cand).to(dev).clamp_min(0)], -1)
    dense[2, 0] = 7                                                     # not an identifier of the index: ignored
    rv, ri = topk_excluding(S, k, *_csr([sorted(c for c in row if c >= 0) for row in cand]))
    idx = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev), identifiers=idents)
    v, i = idx.query_with_exclusions(torch.from_numpy(Q).to(dev), dense)
    want = torch.where(torch.from_numpy(ri).to(dev) >= 0, idents[torch.from_numpy(ri).to(dev).clamp_min(0).long()], -1)
    assert torch.equal(i, want) and np.array_equal(v.cpu().numpy(), rv)
    # candidate indices when the index has no identifiers; every item excluded from row 0 -> pads stay pads
    plain = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev))
    dense2 = torch.from_numpy(np.where(cand >= 0, cand, -1)).to(dev)
    dense2 = torch.cat([dense2, torch.full((U, I), -1, dtype=dense2.dtype, device=dev)], 1)
    dense2[0, n:] = torch.arange(I, device=dev)
    v2, i2 = plain.query_with_exclusions(torch.from_numpy(Q).to(dev), dense2)
    assert (i2[0] == -1).all() and torch.isneginf(v2[0]).all()
    assert torch.equal(i2[1:], torch.from_numpy(ri[1:]).to(dev))
    dense3 = dense2.clone()
    dense3[0, n:] = idents                                              # every identifier of the index
    _, i3 = idx.query_with_exclusions(torch.from_numpy(Q).to(dev), dense3)
    assert (i3[0] == -1).all()
    assert torch.equal(i3[1:], idx(torch.from_numpy(Q).to(dev))[1][1:])  # candidate indices are not identifiers here


@pytest.mark.gpu
def test_torch_op_and_ctypes_route_give_equal_bits(dev):
    from binrec_b200 import _native as N, _torchext as T
    o = T.ops()
    assert o is not None
    rng = np.random.default_rng(8)
    U, I, d, k = 300, 2000, 64, 10
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    indptr, ids = _dev(_csr(_patterns(rng, U, I, k, S)), dev)
    qb, cb = o.rows_to_bf16(torch.from_numpy(Q).to(dev)), o.rows_to_bf16(torch.from_numpy(Cm).to(dev))
    v1, i1 = o.score_topk_exclude(qb, cb, k, 5, indptr, ids)
    ctx, lib = N.ctx(dev), N.lib()
    v2 = torch.empty_like(v1); i2 = torch.empty_like(i1)
    wsb = lib.brk_score_topk_workspace_bytes(ctx, U, I, k)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    N.check(lib.brk_score_topk_bf16_excl(ctx, N.ptr(qb), U, N.ptr(cb), I, qb.shape[1], k, 5, N.ptr(indptr), N.ptr(ids),
                                         N.ptr(v2), N.ptr(i2), N.ptr(ws), wsb, N.stream_ptr()), "excl")
    assert torch.equal(v1, v2) and torch.equal(i1, i2)
    rv, ri = topk_excluding(S, k, indptr.cpu().numpy(), ids.cpu().numpy(), 5)
    _check(v1, i1, rv, ri)


@pytest.mark.gpu
def test_bad_exclusion_arguments_raise_before_any_launch(dev):
    from binrec_b200 import _native as N, _torchext as T
    rng = np.random.default_rng(9)
    Q = torch.from_numpy(_exact(rng, 10, 16)).to(dev)
    idx = H().BruteForceIndex(5).index(torch.from_numpy(_exact(rng, 100, 16)).to(dev))
    ip = torch.zeros(11, dtype=torch.int64, device=dev); ids = torch.zeros(3, dtype=torch.int32, device=dev)
    with pytest.raises(TypeError):
        idx.query_with_exclusions(Q, (ip.int(), ids))
    with pytest.raises(TypeError):
        idx.query_with_exclusions(Q, (ip, ids.long()))
    with pytest.raises(ValueError):
        idx.query_with_exclusions(Q, (ip.cpu(), ids))
    with pytest.raises(ValueError):
        idx.query_with_exclusions(Q, (ip[:10], ids))
    with pytest.raises(TypeError):
        idx.query_with_exclusions(Q, torch.zeros((10, 2), dtype=torch.float32, device=dev))
    with pytest.raises(TypeError):
        H().topk_rows(torch.zeros((10, 100), device=dev), 5, exclude=(ip, ids.long()))
    o = T.ops()
    qb, cb = o.rows_to_bf16(Q), o.rows_to_bf16(torch.from_numpy(_exact(rng, 100, 16)).to(dev))
    with pytest.raises(RuntimeError, match="excl_indptr"):
        o.score_topk_exclude(qb, cb, 5, 0, ip[:10], ids)
    with pytest.raises(RuntimeError, match="excl_ids"):
        o.score_topk_exclude(qb, cb, 5, 0, ip, ids.cpu())
    ctx, lib = N.ctx(dev), N.lib()
    out = torch.empty((10, 5), device=dev); oi = torch.empty((10, 5), dtype=torch.int32, device=dev)
    ws = torch.empty(1 << 16, dtype=torch.uint8, device=dev)
    assert lib.brk_score_topk_bf16_excl(ctx, N.ptr(qb), 10, N.ptr(cb), 100, 64, 5, 0, None, N.ptr(ids), N.ptr(out),
                                        N.ptr(oi), N.ptr(ws), ws.numel(), N.stream_ptr()) == -1
    assert lib.brk_score_topk_bf16_excl(ctx, N.ptr(qb), 10, N.ptr(cb), 100, 64, 5, 0, N.ptr(ip), None, N.ptr(out),
                                        N.ptr(oi), N.ptr(ws), ws.numel(), N.stream_ptr()) == -1
    assert lib.brk_mask_excluded(ctx, N.ptr(out), 10, 5, 0, None, N.ptr(ids), N.stream_ptr()) == -1
    assert lib.brk_mask_excluded(ctx, N.ptr(out), 10, 5, 0, N.ptr(ip), None, N.stream_ptr()) == -1


# ---- models ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bpr_predict_for_users_excluding_seen(dev, tmp_path):
    from binrec_b200.BPRModel import BPRModel
    from binrec_b200 import synth
    users, items = synth.make_interactions(num_users=300, num_items=200, num_pos=12000, seed=3)
    m = BPRModel(workDir=str(tmp_path)); m.epochs = 1
    m.train((users, items), None)
    trU, trI = m.trainDf
    seen = {}
    for u, i in zip(trU.tolist(), trI.tolist()):
        seen.setdefault(u, set()).add(i)
    uq = np.unique(trU)
    asked = [int(uq[5]), int(uq[0]), int(uq[17]), int(uq[5]), int(uq[-1]), int(uq[42])]
    got = m.predictForUsers(asked, 10, excludeSeen=True)
    Uw = OT.bf16_round(m.model.user.w.cpu().numpy()); Iw = OT.bf16_round(m.model.item.w.cpu().numpy())
    for u, row in zip(asked, got):
        ids = [int(p) for p, _ in row]
        assert not (set(ids) & seen.get(u, set()))
        s = (Uw[u].astype(np.float64) @ Iw.astype(np.float64).T).astype(np.float32)
        rv, _ = topk_excluding(s[None], 10, np.array([0, len(seen.get(u, ()))]), np.array(sorted(seen.get(u, ())), np.int32))
        n = int((rv[0] > -np.inf).sum())
        assert len(ids) == n
        np.testing.assert_allclose([float(x) for _, x in row], rv[0, :n], rtol=1e-5, atol=1e-6)
        assert (s[ids] >= rv[0, n - 1] - 1e-5).all()
    assert got[0] == got[3]
    plain = m.predictForUsers(asked, 10)
    assert all(len(r) == 10 for r in plain)
    fresh = BPRModel(workDir=str(tmp_path))
    fresh.compileModel(None, 300, 200, 8)
    with pytest.raises(ValueError):
        fresh.predictForUsers([1], 5, excludeSeen=True)


@pytest.mark.gpu
def test_topkratings_with_exclusions_dot_product_and_nfc(dev):
    from binrec_b200.topKmetrics import topKRatings
    from binrec_b200.NeuMFModel import NeuMFNet
    rng = np.random.default_rng(10)
    U, I, d, k = 50, 120, 16, 10
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    usersId = [f"u{j}" for j in range(U)]; itemsId = [1000 + j for j in range(I)]

    class Dot:
        def score_vectors(self, us, its):
            return torch.from_numpy(Q).to(dev), torch.from_numpy(Cm).to(dev)

    S = OT.scores(Q, Cm)
    lists = _patterns(rng, U, I, k, S)
    pairs = [(usersId[r], itemsId[c]) for r, l in enumerate(lists) for c in l] + [("nobody", 1000), ("u1", -5)]
    rv, ri = topk_excluding(S, k, *_csr(lists))
    got = topKRatings(k, Dot(), usersId, itemsId, exclude=pairs)
    for r, (u, lst) in enumerate(got):
        n = int((ri[r] >= 0).sum())
        assert u == usersId[r] and [it for _, it in lst] == [itemsId[c] for c in ri[r, :n]]
        assert [float(s) for s, _ in lst] == rv[r, :n].tolist()
    net = NeuMFNet(U, I, 8, dropout=0.0, device=dev)
    uid = list(range(U)); iid = list(range(I))
    ref = net.score_all(uid, iid, I)                                   # the whole ranking per user
    Sn = np.full((U, I), -np.inf, np.float32)
    np.put_along_axis(Sn, ref[1].cpu().numpy().astype(np.int64), ref[0].cpu().numpy(), 1)
    pairs_n = [(r, c) for r, l in enumerate(lists) for c in l]
    nv, ni = topk_excluding(Sn, k, *_csr(lists))
    got = topKRatings(k, net, uid, iid, mtype="NFC", exclude=pairs_n)
    for r, (u, lst) in enumerate(got):
        n = int((ni[r] >= 0).sum())
        assert [it for _, it in lst] == ni[r, :n].tolist() and [float(s) for s, _ in lst] == nv[r, :n].tolist()


@pytest.mark.gpu
def test_twotower_predict_and_crossvalidation_exclude_training_pairs(dev):
    from binrec_b200.twoTower import TwoTowerModel, crossValidation
    from binrec_b200.topKmetrics import topKMetrics
    rng = np.random.default_rng(11)
    nu, ni = 80, 50
    users = [f"c{j}" for j in range(nu)]; items = [f"m{j}" for j in range(ni)]
    m = TwoTowerModel(16, ni, nu, "CUSTOMER_ID", "MATERIAL", users, items, semb=8, device=dev)
    m.setCandidates(items, 10)
    pairs = [(users[a], items[b]) for a, b in zip(rng.integers(0, nu, 1500), rng.integers(0, ni, 1500))]
    pairs += [(users[3], it) for it in items]                          # user 3: everything excluded
    scores, idents = m.predict(users, batch_size=32, exclude=pairs)
    s0, i0 = m.predict(users, batch_size=32)
    excl = {}
    for u, it in pairs:
        excl.setdefault(u, set()).add(it)
    qv = m._tower_forward(m.userTower, torch.from_numpy(m.userTowerIn(users)).to(dev))
    S = (qv.to(torch.bfloat16).double() @ m.bruteForceLayer._c[:, :m.bruteForceLayer.dim].double().T).float().cpu().numpy()
    for r, u in enumerate(users):
        assert not (set(idents[r]) & excl.get(u, set()))
        left = [j for j in range(ni) if items[j] not in excl.get(u, set())]
        assert len(idents[r]) == min(10, len(left))
        if idents[r]:
            kth = np.sort(S[r, left])[::-1][len(idents[r]) - 1]
            assert all(S[r, items.index(it)] >= kth - 1e-4 for it in idents[r])
    assert idents[3] == [] and np.isneginf(scores[3]).all()
    assert all(len(x) == 10 for x in i0)
    # cross-validation: no training pair in any list; metrics equal the oracle's on the lists returned
    folds = []
    for f in range(3):
        u = rng.integers(0, 40, 600); mm = (u % 5) * 6 + rng.integers(0, 6, 600)
        folds.append({"CUSTOMER_ID": [f"c{j}" for j in u], "MATERIAL": [f"m{j}" for j in mm]})
    import binrec_b200.twoTower as TT
    seen_lists, calls = [], []
    orig = TT.TwoTowerModel.predict

    def spy(self, usersId, batch_size=5000, exclude=None):
        out = orig(self, usersId, batch_size, exclude)
        calls.append((list(usersId), out, exclude))
        return out
    TT.TwoTowerModel.predict = spy
    try:
        res = crossValidation(folds, 10, 0.1, "Adagrad", None, 2, 16, 300, semb=8, excludeTrain=True)
    finally:
        TT.TwoTowerModel.predict = orig
    assert len(calls) == 3
    usersId = list(dict.fromkeys(u for f in folds for u in f["CUSTOMER_ID"]))
    matId = list(dict.fromkeys(x for f in folds for x in f["MATERIAL"]))
    held, full = [], []
    for it, (uids, (sc, idn), exclude) in enumerate(calls):
        train = {(u, x) for j, f in enumerate(folds) if j != it for u, x in zip(f["CUSTOMER_ID"], f["MATERIAL"])}
        assert set(exclude) == train
        preds = [(u, [(sc[r][j], idn[r][j]) for j in range(len(idn[r]))]) for r, u in enumerate(uids)]
        assert not any((u, x) in train for u, l in preds for _, x in l)
        test = folds[it]
        held.append(OT.topk_metrics(preds, list(zip(test["CUSTOMER_ID"], test["MATERIAL"])), usersId, matId))
        full.append(OT.topk_metrics(preds, list(train), usersId, matId))
        assert full[-1]["tp"] == 0
        assert held[-1] == topKMetrics(preds, list(zip(test["CUSTOMER_ID"], test["MATERIAL"])), usersId, matId)
    for key in held[0]:
        assert res[key] == pytest.approx(sum(h[key] for h in held) / 3, rel=1e-12)
    assert res["full_tp"] == 0 and res["full_hitRate"] == 0
