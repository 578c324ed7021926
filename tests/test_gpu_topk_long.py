"""Lists longer than 32 on the fused scorer: score_topk_kernel keeps them as a heap per row in shared memory, for
k up to hotpath.fused_k_cap(dpad) (128 up to dpad 128, 64 at dpad 192 and 256).

Oracles: oracle/topk.py and the exclusion definition `topk_excluding` of test_gpu_topk_exclude.py.  Bit-exact claims
use exact-arithmetic inputs (entries j/8, |j| <= 4: exact in bf16, products and sums exact in fp32).  Random-normal
inputs are held to the bf16-operand oracle at 1e-5 with gap-aware ids, as in test_gpu_topk.py, and to themselves bit
for bit across launches (other users, other k, item shards)."""
import numpy as np
import pytest
import torch

from oracle import topk as OT
from test_gpu_topk_exclude import _csr, _dev, _patterns, topk_excluding

pytestmark = pytest.mark.gpu


def H():
    from binrec_b200 import hotpath
    return hotpath


def _exact(rng, rows, d, lo=-4, hi=4):
    return (rng.integers(lo, hi + 1, size=(rows, d)) / 8.0).astype(np.float32)


def _eq(got, want):
    v, i = got
    rv, ri = want
    assert np.array_equal(i.cpu().numpy(), ri)
    assert np.array_equal(v.cpu().numpy(), rv)


def _gap_aware(v, i, S, k):
    """Scores within 1e-5 of the bf16-operand oracle S; ids equal wherever the oracle's neighbouring ranks are apart."""
    rv, ri = OT.topk_from_scores(S, k + 1)
    np.testing.assert_allclose(v, rv[:, :k], rtol=1e-5, atol=1e-5)
    safe = np.ones((v.shape[0], k), dtype=bool)
    safe[:, 1:] &= (rv[:, :k - 1] - rv[:, 1:k]) > 1e-4
    safe &= (rv[:, :k] - rv[:, 1:k + 1]) > 1e-4
    assert safe.mean() > 0.9
    assert np.array_equal(i[safe], ri[:, :k][safe])
    got = np.take_along_axis(S, i.astype(np.int64), 1)
    assert (got >= rv[:, k - 1:k] - 1e-4).all()                 # every returned id is a genuine top-k member


# ---- 1. bit-exact on exact-arithmetic inputs -------------------------------------------------------------------------
@pytest.mark.parametrize("k,d", [(k, d) for k in (33, 64, 100, 128) for d in (16, 64, 100, 128)] +
                         [(k, d) for k in (33, 64) for d in (160, 256)])
def test_exact_arithmetic_bit_exact(dev, k, d):
    rng = np.random.default_rng(k * 1000 + d)
    Q = _exact(rng, 333, d)
    for I in (k // 2 + 1, k, 3 * 128 + 77, 5 * 128):              # I < k (clamped), I = k, ragged last tile, whole tiles
        C = _exact(rng, I, d)
        idx = H().BruteForceIndex(k).index(torch.from_numpy(C).to(dev))
        for U in (1, 129, 333):
            got = idx(torch.from_numpy(Q[:U]).to(dev))
            assert got[0].shape == (U, min(k, I))
            _eq(got, OT.brute_force_topk(Q[:U], C, k))


# ---- 2. ties ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [40, 100, 128])
def test_ties_keep_the_lower_id_across_chunks_tiles_and_splits(dev, k):
    """Values in {-1, 0, 1}/8 at d = 4: nine distinct scores, so every list ends inside a tie group spread over all
    tiles.  Two query rows alone run on 32 item splits; the same rows among 18 944 (148 m-tiles) run on one."""
    rng = np.random.default_rng(k)
    d, I = 4, 40 * 128 + 5
    C = _exact(rng, I, d, -1, 1)
    Q = _exact(rng, 18944, d, -1, 1)
    Q[:2] = np.array([[1, 1, 1, 1], [1, -1, 0, 1]], np.float32) / 8
    idx = H().BruteForceIndex(k).index(torch.from_numpy(C).to(dev))
    small = idx(torch.from_numpy(Q[:2]).to(dev))
    large = idx(torch.from_numpy(Q).to(dev))
    _eq(small, OT.brute_force_topk(Q[:2], C, k))
    _eq(large, OT.brute_force_topk(Q, C, k))
    # exclusions on the single-split launch (it writes the final lists itself): every 100th row leaves out its top 20
    lists = [sorted(large[1][r, :20].tolist()) if r % 100 == 0 else [] for r in range(len(Q))]
    v, i = idx.query_with_exclusions(torch.from_numpy(Q).to(dev), _dev(_csr(lists), dev))
    rows = np.arange(0, len(Q), 100)
    _eq((v[rows], i[rows]), topk_excluding(OT.scores(Q[rows], C), k, *_csr([lists[r] for r in rows])))
    rest = torch.from_numpy(np.setdiff1d(np.arange(len(Q)), rows)).to(dev)
    assert torch.equal(v[rest], large[0][rest]) and torch.equal(i[rest], large[1][rest])
    # one tie group at the top: items whose id is a multiple of 37 share the best score, everything else scores lower
    C2 = np.zeros((I, d), np.float32); C2[:, 0] = -1 / 8
    C2[::37, 0] = 1 / 8
    C2[:, 1:] = _exact(rng, I, d - 1)                              # Q's other columns are 0: the group stays tied
    q =np.array([[1 / 8, 0, 0, 0]] * 3, np.float32)
    v, i = H().BruteForceIndex(k).index(torch.from_numpy(C2).to(dev))(torch.from_numpy(q).to(dev))
    assert (i.cpu().numpy() == np.arange(k) * 37).all()
    assert (v.cpu().numpy() == 1 / 64).all()


# ---- 3. launch independence ------------------------------------------------------------------------------------------
def test_launch_independence_bit_for_bit(dev):
    rng = np.random.default_rng(3)
    U, I, d = 1000, 20000, 64
    Q = torch.from_numpy(rng.standard_normal((U, d)).astype(np.float32)).to(dev)
    C = torch.from_numpy(rng.standard_normal((I, d)).astype(np.float32)).to(dev)
    idx = H().BruteForceIndex().index(C)
    v128, i128 = idx(Q, 128)
    for k in (100, 64, 32, 10):                                    # k <= 32 runs the register-list instantiations
        v, i = idx(Q, k)
        assert torch.equal(v, v128[:, :k]) and torch.equal(i, i128[:, :k])
    perm = torch.from_numpy(rng.permutation(U)).to(dev)
    v, i = idx(Q[perm], 128)
    assert torch.equal(v, v128[perm]) and torch.equal(i, i128[perm])
    dup = torch.tensor([5, 5, 999, 0, 5, 300], device=dev)
    v, i = idx(Q[dup], 128)
    assert torch.equal(v, v128[dup]) and torch.equal(i, i128[dup])
    v, i = idx(Q[100:229], 128)
    assert torch.equal(v, v128[100:229]) and torch.equal(i, i128[100:229])
    # item-range shards merged by topk_merge against the unsharded call
    v100, i100 = idx(Q, 100)
    bounds = [0, 5000, 12345, 12500, 20000]
    pv, pi = [], []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        v, i = H().BruteForceIndex(100).index(C[lo:hi], id_offset=lo)(Q)
        if v.shape[1] < 100:                                       # a shard narrower than k: pad to k for the merge
            v = torch.cat([v, torch.full((U, 100 - v.shape[1]), float("-inf"), device=dev)], 1)
            i = torch.cat([i, torch.full((U, 100 - i.shape[1]), -1, dtype=torch.int32, device=dev)], 1)
        pv.append(v); pi.append(i)
    v, i = H().topk_merge(torch.stack(pv), torch.stack(pi))
    assert torch.equal(v, v100) and torch.equal(i, i100)


# ---- 4. random-normal accuracy ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("U,I,d,k", [(6040, 3706, 64, 100), (8192, 250000, 64, 128)])
def test_random_normal_against_the_bf16_oracle(dev, U, I, d, k):
    rng = np.random.default_rng(I + k)
    Q = rng.standard_normal((U, d)).astype(np.float32)
    C = rng.standard_normal((I, d)).astype(np.float32)
    v, i = H().BruteForceIndex(k).index(torch.from_numpy(C).to(dev))(torch.from_numpy(Q).to(dev))
    v, i = v.cpu().numpy(), i.cpu().numpy()
    rows = np.arange(U) if U * I <= 1 << 25 else np.unique(np.r_[0, U - 1, rng.choice(U, 190, replace=False)])
    _gap_aware(v[rows], i[rows], OT.scores(Q[rows], C, "bf16"), k)


# ---- 5. exclusions ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [40, 128])
def test_exclusions_against_the_definition(dev, k):
    rng = np.random.default_rng(k + 5)
    U, I, d = 300, 2000, 64
    Q, Cm = _exact(rng, U, d), _exact(rng, I, d)
    S = OT.scores(Q, Cm)
    Qd = torch.from_numpy(Q).to(dev)
    idx = H().BruteForceIndex(k).index(torch.from_numpy(Cm).to(dev))
    # empty, the row's best, long random lists, all but k - 1 items (padding), everything
    lists = _patterns(rng, U, I, k, S)
    csr = _csr(lists)
    _eq(idx.query_with_exclusions(Qd, _dev(csr, dev)), topk_excluding(S, k, *csr))
    # worst case: every row lists its own true top m
    fv, fi = OT.topk_from_scores(S, I)
    for m in (1, 130, I - k // 2):
        csr = _csr([sorted(fi[r, :m].tolist()) for r in range(U)])
        _eq(idx.query_with_exclusions(Qd, _dev(csr, dev)), topk_excluding(S, k, *csr))
    # ids outside the range and duplicates are ignored
    noisy = [sorted([-7, -1] + l[:50] + l[:3] + [I, I + 5, 1 << 30]) for l in lists]
    _eq(idx.query_with_exclusions(Qd, _dev(_csr(noisy), dev)), topk_excluding(S, k, *_csr([l[:50] for l in lists])))
    # an item-range shard with one global list
    lo = 700
    sh = H().BruteForceIndex(k).index(torch.from_numpy(Cm[lo:]).to(dev), id_offset=lo)
    _eq(sh.query_with_exclusions(Qd, _dev(csr, dev)), topk_excluding(S[:, lo:], k, *csr, id_offset=lo))
    # empty lists: the plain call's bits, on random-normal data
    Qn = torch.from_numpy(rng.standard_normal((U, d)).astype(np.float32)).to(dev)
    Cn = H().BruteForceIndex(k).index(torch.from_numpy(rng.standard_normal((I, d)).astype(np.float32)).to(dev))
    empty = (torch.zeros(U + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev))
    v0, i0 = Cn(Qn)
    v, i = Cn.query_with_exclusions(Qn, empty)
    assert torch.equal(v, v0) and torch.equal(i, i0)


# ---- 6. routing ------------------------------------------------------------------------------------------------------
def test_fused_up_to_the_cap_materialised_beyond(dev, monkeypatch):
    h = H()
    calls = []
    orig = h.BruteForceIndex._call_materialised

    def spy(self, queries, k, exclusions=None):
        calls.append(k)
        return orig(self, queries, k, exclusions)
    monkeypatch.setattr(h.BruteForceIndex, "_call_materialised", spy)
    rng = np.random.default_rng(6)
    for d, dpad in ((64, 64), (128, 128), (200, 256)):
        assert h.fused_k_cap(dpad) == (128 if dpad <= 128 else 64)
        cap = h.fused_k_cap(dpad)
        Q, Cm = _exact(rng, 50, d), _exact(rng, 700, d)
        S = OT.scores(Q, Cm)
        idx = h.BruteForceIndex().index(torch.from_numpy(Cm).to(dev))
        assert idx._c.shape[1] == dpad
        Qd = torch.from_numpy(Q).to(dev)
        csr = _csr(_patterns(rng, 50, 700, cap, S))
        for k in sorted({33, 50, cap // 2 + 1, cap}):
            _eq(idx(Qd, k), OT.topk_from_scores(S, k))
            _eq(idx.query_with_exclusions(Qd, _dev(csr, dev), k), topk_excluding(S, k, *csr))
        assert calls == []
        _eq(idx(Qd, cap + 1), OT.topk_from_scores(S, cap + 1))
        _eq(idx.query_with_exclusions(Qd, _dev(csr, dev), cap + 1), topk_excluding(S, cap + 1, *csr))
        assert calls == [cap + 1, cap + 1]
        calls.clear()


# ---- 7. both bindings ------------------------------------------------------------------------------------------------
def test_torch_op_and_ctypes_routes_give_equal_bits(dev, monkeypatch):
    from binrec_b200 import _torchext as T
    assert T.ops() is not None
    rng = np.random.default_rng(7)
    U, I, d, k = 700, 5000, 64, 100
    Q = torch.from_numpy(rng.standard_normal((U, d)).astype(np.float32)).to(dev)
    idx = H().BruteForceIndex(k).index(torch.from_numpy(rng.standard_normal((I, d)).astype(np.float32)).to(dev))
    ex = _dev(_csr([sorted(rng.choice(I, size=rng.integers(0, 300), replace=False).tolist()) for _ in range(U)]), dev)
    a, b = idx(Q), idx.query_with_exclusions(Q, ex)
    monkeypatch.setitem(T._state, "ops", None)                     # what BRK_BINDING=ctypes selects
    assert T.ops() is None
    a2, b2 = idx(Q), idx.query_with_exclusions(Q, ex)
    for x, y in ((a, a2), (b, b2)):
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])


# ---- 8. C ABI rejections ---------------------------------------------------------------------------------------------
def test_c_abi_rejects_before_any_launch(dev):
    from binrec_b200 import _native as N
    lib, ctx = N.lib(), N.ctx(dev)
    rng = np.random.default_rng(8)
    U, I = 10, 300

    def operands(d):
        return (H().rows_to_bf16(torch.from_numpy(_exact(rng, U, d)).to(dev)),
                H().rows_to_bf16(torch.from_numpy(_exact(rng, I, d)).to(dev)))
    ip = torch.zeros(U + 1, dtype=torch.int64, device=dev); xi = torch.zeros(1, dtype=torch.int32, device=dev)
    out = torch.full((U, 129), 7.0, device=dev); oi = torch.full((U, 129), 7, dtype=torch.int32, device=dev)
    ws = torch.empty(1 << 22, dtype=torch.uint8, device=dev)
    st = N.stream_ptr()

    def plain(q, c, k, wsb=ws.numel(), qp=None, cp=None):
        return lib.brk_score_topk_bf16(ctx, N.ptr(q) if qp is None else qp, U, N.ptr(c) if cp is None else cp, I,
                                       q.shape[1], k, 0, N.ptr(out), N.ptr(oi), N.ptr(ws), wsb, st)

    def excl(q, c, k, wsb=ws.numel(), ipp=None, xip=None):
        return lib.brk_score_topk_bf16_excl(ctx, N.ptr(q), U, N.ptr(c), I, q.shape[1], k, 0,
                                            N.ptr(ip) if ipp is None else ipp, N.ptr(xi) if xip is None else xip,
                                            N.ptr(out), N.ptr(oi), N.ptr(ws), wsb, st)

    def rejected(rc, words):
        assert rc == -1
        msg = lib.brk_last_error().decode()
        assert all(w in msg for w in words), msg

    q64, c64 = operands(64)
    q256, c256 = operands(256)
    for f in (plain, excl):
        rejected(f(q64, c64, 0), ["k=0", "128"])
        rejected(f(q64, c64, 129), ["k=129", "128"])
        rejected(f(q256, c256, 65), ["k=65", "dpad=256", "64"])
        for k in (100, 64):
            q, c = (q64, c64) if k == 100 else (q256, c256)
            need = lib.brk_score_topk_workspace_bytes(ctx, U, I, k)
            assert need >= U * k * 8
            rejected(f(q, c, k, need - 8), ["workspace"])
    rejected(plain(q64, c64, 100, qp=0), ["null"])
    rejected(plain(q64, c64, 100, cp=0), ["null"])
    rejected(excl(q64, c64, 100, ipp=0), ["null"])
    rejected(excl(q64, c64, 100, xip=0), ["null"])
    torch.cuda.synchronize()
    assert (out == 7.0).all() and (oi == 7).all()                  # nothing was launched
    # the workspace the size query gives is enough at every cap
    for q, c, k in ((q64, c64, 128), (q256, c256, 64)):
        need = lib.brk_score_topk_workspace_bytes(ctx, U, I, k)
        assert plain(q, c, k, need) == 0 and excl(q, c, k, need) == 0
