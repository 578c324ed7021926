"""The two general dense products against a float64 reference on the same fp32 inputs: brk_sgemm (csrc/twotower.cu,
fp32 on the CUDA cores) and brk_gemm_tf32 (csrc/gemm_tc.cu, tcgen05, TF32 operands, fp32 accumulation; its reference
reads the operands through oracle/tf32.trunc_np).  Both sit under the two-tower step, the tower forward that builds
the retrieval indexes, both halves of the factored NeuMF top-K indexes and BPRModel's full-catalog evaluation.

Two kinds of check:
  exact    operands are small integers over 16, so every partial sum, the alpha scale, the bias and the K-split
           reductions are exact in fp32 and the result must equal the reference bit for bit.  A wrong element, a
           missed or doubled K tile or a bias added by every split is off by a whole unit.
  bounded  random normal operands (already TF32-representable for brk_gemm_tf32, so the operand rule pinned by
           tests/test_gpu_tc.py does not enter): elementwise
               |C - ref| <= (K + splits + 2) 2^-24 (|alpha| |A| |B| + |bias| + |C0|),
           the worst-case bound of K sequential fp32 multiply-adds, the alpha scale, the bias add and one add per K
           split (C0: what C held before an accumulating call).  That tcgen05 accumulates at least as precisely as
           sequential fp32 is an assumption; the largest ratio of error to bound is printed.
Storage: every stored element outside the logical operands is NaN (a product that reads one turns NaN), C has a
sentinel in its padding columns, ahead of an offset base and in a row past M, and the sentinels must survive.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

BRK_E_ARG, BRK_E_ALIGN = -1, -2
SENTINEL = np.float32(-7777.25)
U = 2.0 ** -24                      # unit roundoff of fp32
MN = [1, 63, 64, 65, 127, 129, 1000]
KS = [1, 15, 16, 17, 31, 33, 1000, 4097]
PAIRS = list(zip(MN, MN[1:] + MN[:1]))          # every M and every N value once
GRID_Y_MAX = 65535                              # the row tiles of a product must not be bound by gridDim.y


def _nn():
    from binrec_b200 import _native as Nn
    return Nn


@pytest.fixture(scope="module")
def sm(dev):
    Nn = _nn()
    n = Nn.lib().brk_sm_count(Nn.ctx(dev))
    assert n > 0
    return n


def _cdiv(a, b):
    return -(-a // b)


# ---- the launch arithmetic, restated (csrc/twotower.cu sgemm, csrc/gemm_tc.cu gemm_tf32_run) ----------------------
def sgemm_splits(M, N, K, accumulate, sm):
    """64 x 64 output tiles; an accumulating call splits K (in 16-deep steps) until there are 2 CTAs per SM."""
    splits = 1
    if accumulate:
        splits = max(1, min(2 * sm // (_cdiv(N, 64) * _cdiv(M, 64)), _cdiv(K, 64), 64))
    kps = _cdiv(_cdiv(K, splits), 16) * 16
    return _cdiv(K, kps)


def tf32_plan(M, N, K, accumulate, sm):
    """(BN, splits): 128 x BN tiles, BN the widest of 128 / 64 / 32 that gives a quarter wave of CTAs; an accumulating
    call splits K (in 32-deep chunks) until there is one CTA per SM."""
    row_tiles = _cdiv(M, 128)
    BN = 128
    while BN > 32 and (BN // 2 >= N or row_tiles * _cdiv(N, BN) < sm // 4):
        BN //= 2
    splits = 1
    if accumulate:
        want = sm // (_cdiv(N, BN) * row_tiles)
        splits = 1 if want < 1 else min(want, _cdiv(K, 128), 64)
    kps = _cdiv(_cdiv(K, splits), 32) * 32
    return BN, _cdiv(K, kps)


class Kernel:
    def __init__(self, name):
        self.name, self.tf32 = name, name == "brk_gemm_tf32"

    def fn(self):
        return getattr(_nn().lib(), self.name)

    def ld(self, minimum, padded):
        """brk_gemm_tf32 needs leading dimensions that are multiples of 4; brk_sgemm gets odd ones when padded."""
        if self.tf32:
            return _cdiv(minimum, 4) * 4 + (4 if padded else 0)
        return minimum + 1 + (minimum & 1) if padded else minimum

    def offset(self, padded):
        """Floats by which the operand and C bases are moved off their 16-byte-aligned allocation."""
        return 1 if padded and not self.tf32 else 0

    def splits(self, M, N, K, accumulate, sm):
        return tf32_plan(M, N, K, accumulate, sm)[1] if self.tf32 else sgemm_splits(M, N, K, accumulate, sm)

    def operand(self, x):
        from oracle import tf32
        return tf32.trunc_np(x) if self.tf32 else x

    def __repr__(self):
        return self.name


KERNELS = [Kernel("brk_sgemm"), Kernel("brk_gemm_tf32")]


def _addr(t, off=0):
    return None if t is None else C.c_void_p(t.data_ptr() + 4 * off)


def _store(X, ld, off):
    """X [R, W] row-major with leading dimension ld >= W, `off` floats into a buffer that is NaN everywhere else."""
    R, W = X.shape
    buf = np.full(off + R * ld, np.nan, np.float32)
    buf[off:].reshape(R, ld)[:, :W] = X
    return buf


def run(dev, kern, Al, Bl, ta, tb, alpha=1.0, accumulate=0, bias=None, C0=None, padded=False):
    """C = alpha Al Bl (+ bias) (+ C0 when accumulating) through kern with A stored transposed when ta, B when tb.
    Returns the M x N result; asserts that nothing else in C's storage changed."""
    Nn = _nn()
    M, K = Al.shape
    N = Bl.shape[1]
    lda, ldb = kern.ld(M if ta else K, padded), kern.ld(K if tb else N, padded)
    ldc, off = N + 3 if padded else N, kern.offset(padded)
    As, Bs = _store(Al.T if ta else Al, lda, off), _store(Bl.T if tb else Bl, ldb, off)
    Cs = np.full(off + (M + 1) * ldc, SENTINEL, np.float32)
    Cs[off:off + M * ldc].reshape(M, ldc)[:, :N] = C0 if accumulate else np.nan
    Ad, Bd, Cd = (torch.from_numpy(x).to(dev) for x in (As, Bs, Cs))
    bd = None if bias is None else torch.from_numpy(bias).to(dev)
    Nn.check(kern.fn()(Nn.ctx(dev), _addr(Ad, off), _addr(Bd, off), _addr(Cd, off), _addr(bd), M, N, K, lda, ldb, ldc, ta, tb,
                       alpha, accumulate, Nn.stream_ptr()), kern.name)
    got = Cd.cpu().numpy()
    inside = np.zeros(Cs.shape, bool)
    inside[off:off + M * ldc].reshape(M, ldc)[:, :N] = True
    assert np.array_equal(got[~inside], Cs[~inside]), "the call wrote C outside [M, N]"
    return got[off:off + M * ldc].reshape(M, ldc)[:, :N].copy()


def reference(Al, Bl, alpha, bias, C0):
    """(alpha A B + bias + C0, alpha |A| |B| + |bias| + |C0|) in float64."""
    A64, B64 = Al.astype(np.float64), Bl.astype(np.float64)
    ref, scale = alpha * (A64 @ B64), abs(alpha) * (np.abs(A64) @ np.abs(B64))
    for t in (bias, C0):
        if t is not None:
            ref, scale = ref + t, scale + np.abs(t)
    return ref, scale


def small_ints(rng, shape, den):
    return (rng.integers(-den, den + 1, size=shape) / den).astype(np.float32)


def check_exact(dev, kern, rng, M, N, K, ta, tb, alpha, accumulate, with_bias, padded):
    Al, Bl = small_ints(rng, (M, K), 16), small_ints(rng, (K, N), 16)
    bias = small_ints(rng, N, 4) * 2 if with_bias else None
    C0 = small_ints(rng, (M, N), 2) * 4 if accumulate else None
    got = run(dev, kern, Al, Bl, ta, tb, alpha, accumulate, bias, C0, padded)
    ref, _ = reference(Al, Bl, alpha, bias, C0)
    assert np.array_equal(ref.astype(np.float32).astype(np.float64), ref)        # the premise: ref is an fp32 value
    bad = np.argwhere(got != ref.astype(np.float32))
    assert bad.size == 0, (f"{len(bad)} of {M * N} wrong, first at {tuple(bad[0])}: "
                           f"{got[tuple(bad[0])]} != {ref[tuple(bad[0])]}")


def check_bounded(dev, kern, rng, M, N, K, ta, tb, alpha, accumulate, with_bias, padded, splits):
    """Returns the largest |error| / bound."""
    Al = kern.operand(rng.standard_normal((M, K)).astype(np.float32))
    Bl = kern.operand(rng.standard_normal((K, N)).astype(np.float32))
    bias = rng.standard_normal(N).astype(np.float32) if with_bias else None
    C0 = rng.standard_normal((M, N)).astype(np.float32) if accumulate else None
    got = run(dev, kern, Al, Bl, ta, tb, alpha, accumulate, bias, C0, padded).astype(np.float64)
    ref, scale = reference(Al, Bl, alpha, bias, C0)
    err, bound = np.abs(got - ref), (K + splits + 2) * U * scale
    bad = np.argwhere(~(err <= bound))
    assert bad.size == 0, (f"{len(bad)} of {M * N} outside the bound, first at {tuple(bad[0])}: "
                           f"|{got[tuple(bad[0])]} - {ref[tuple(bad[0])]}| > {bound[tuple(bad[0])]}")
    return float(np.max(err / np.maximum(bound, np.finfo(np.float64).tiny)))


# ---- layouts, edges, storage ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("padded", [False, True], ids=["tight", "padded"])
@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("kern", KERNELS, ids=str)
def test_product_matches_float64_reference(dev, sm, kern, ta, tb, K, padded):
    """M and N from {1, 63, 64, 65, 127, 129, 1000}, every layout, K across the tile depths (16 for brk_sgemm, 32 for
    brk_gemm_tf32).  'tight': minimal leading dimensions (rounded up to 4 for brk_gemm_tf32), ldc = N; 'padded': odd
    leading dimensions and bases one float off alignment for brk_sgemm, leading dimensions 4 past the rounded minimum
    for brk_gemm_tf32, ldc = N + 3 for both.  accumulate = 0 and 1 (K = 4097 with few output tiles splits K), with a
    bias except in the tight accumulate = 0 call."""
    rng = np.random.default_rng(1000 * K + 10 * (2 * ta + tb) + padded + 7 * kern.tf32)
    worst = 0.0
    for M, N in PAIRS:
        for accumulate in (0, 1):
            with_bias = padded or accumulate == 1
            check_exact(dev, kern, rng, M, N, K, ta, tb, -0.5, accumulate, with_bias, padded)
            splits = kern.splits(M, N, K, accumulate, sm)
            worst = max(worst, check_bounded(dev, kern, rng, M, N, K, ta, tb, 0.75, accumulate, with_bias, padded, splits))
    print(f"{kern} ta={ta} tb={tb} K={K} {'padded' if padded else 'tight'}: largest error / bound {worst:.3g}")


@pytest.mark.parametrize("BN", [32, 64, 128])
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_gemm_tf32_every_tile_width(dev, sm, BN, ta, tb):
    """brk_gemm_tf32 picks its tile width from M, N and the SM count; at M = 1000 find the widths N that give each one
    (with 148 SMs: 1000 / 999 -> 128, 300 / 301 -> 64, 127 / 1 -> 32) and check them."""
    kern, M, K = KERNELS[1], 1000, 97
    widths = [N for N in (1000, 999, 300, 301, 129, 127, 1) if tf32_plan(M, N, K, 0, sm)[0] == BN]
    assert widths, f"no N at M = {M} gives BN = {BN} with {sm} SMs"
    rng = np.random.default_rng(BN + 2 * ta + tb)
    worst = 0.0
    for N in widths:
        for accumulate in (0, 1):
            check_exact(dev, kern, rng, M, N, K, ta, tb, 2.0, accumulate, True, True)
            splits = kern.splits(M, N, K, accumulate, sm)
            worst = max(worst, check_bounded(dev, kern, rng, M, N, K, ta, tb, -1.25, accumulate, True, True, splits))
    print(f"BN={BN} at N in {widths}, ta={ta} tb={tb}: largest error / bound {worst:.3g}")


# ---- split-K --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K", [(1, 1, 4097), (64, 64, 4097), (65, 129, 1000), (128, 128, 1000), (3, 300, 2048)])
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("kern", KERNELS, ids=str)
def test_split_k_adds_each_product_and_the_bias_once(dev, sm, kern, M, N, K, ta, tb):
    """Few output tiles and a long K: an accumulating call splits K over CTAs whose partial products are REDs into C,
    and only split 0 adds the bias.  Exact inputs show a split that stores instead of adding, a K tile skipped or
    counted twice, and a bias added by every split."""
    splits = kern.splits(M, N, K, 1, sm)
    assert splits > 1, (kern, M, N, K, splits)
    rng = np.random.default_rng(M + N + K + 2 * ta + tb)
    for padded in (False, True):
        check_exact(dev, kern, rng, M, N, K, ta, tb, 0.5, 1, True, padded)
        ratio = check_bounded(dev, kern, rng, M, N, K, ta, tb, 1.5, 1, True, padded, splits)
        print(f"{kern} M={M} N={N} K={K} ta={ta} tb={tb}: {splits} splits, largest error / bound {ratio:.3g}")


# ---- row independence -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("kern", KERNELS, ids=str)
def test_a_row_does_not_depend_on_the_other_rows_of_the_call(dev, sm, kern, ta, tb):
    """Without accumulation a row of C is the same bits whatever M is and whichever rows share the call: the
    item-range indexes of the sharded top-K are bit-equal to the single-GPU index only so.  The slices are chosen so
    that brk_gemm_tf32 runs them at different tile widths than the whole (with 148 SMs: 128 for the whole, 64 and 32
    for the slices)."""
    Mf, N, K = 20000, 128, 200
    rng = np.random.default_rng(31 + 2 * ta + tb)
    A = rng.standard_normal((Mf, K)).astype(np.float32)          # full mantissas: brk_gemm_tf32 truncates them itself
    B = rng.standard_normal((K, N)).astype(np.float32)
    bias = rng.standard_normal(N).astype(np.float32)
    full = run(dev, kern, A, B, ta, tb, 0.75, 0, bias)
    ref, scale = reference(kern.operand(A), kern.operand(B), 0.75, bias, None)
    assert (np.abs(full - ref) <= (K + 3) * U * scale).all()
    slices = [(3001, 4001), (777, 4877), (19999, 20000), (0, 1), (130, 5130)]
    if kern.tf32:
        widths = {tf32_plan(b - a, N, K, 0, sm)[0] for a, b in slices} | {tf32_plan(Mf, N, K, 0, sm)[0]}
        print("tile widths in play:", sorted(widths))
        assert len(widths) >= 2, widths
    for a, b in slices:
        part = run(dev, kern, A[a:b], B, ta, tb, 0.75, 0, bias)
        assert np.array_equal(part.view(np.uint32), full[a:b].view(np.uint32)), (a, b)
    perm = rng.permutation(Mf)
    shuffled = run(dev, kern, np.ascontiguousarray(A[perm]), B, ta, tb, 0.75, 0, bias)
    assert np.array_equal(shuffled.view(np.uint32), full[perm].view(np.uint32))


# ---- brk_tower_forward ----------------------------------------------------------------------------------------------
def tower_forward(dev, table, dense, E, S, ids):
    Nn = _nn()
    n = len(ids)
    w, d, idd = (torch.from_numpy(x).to(dev) for x in (table, dense, ids))
    emb = torch.full((n, E), float("nan"), device=dev)
    out = torch.full((n, S), float("nan"), device=dev)
    t = Nn.brk_tower(Nn.brk_table(w.data_ptr(), None, None, None, None, table.shape[0], E, 0),
                     Nn.brk_table(d.data_ptr(), None, None, None, None, 1, dense.size, 0), E, S)
    Nn.check(Nn.lib().brk_tower_forward(Nn.ctx(dev), C.byref(t), Nn.ptr(idd), n, Nn.ptr(emb), Nn.ptr(out), Nn.stream_ptr()),
             "brk_tower_forward")
    return emb.cpu().numpy(), out.cpu().numpy()


def check_tower(dev, rng, rows, E, S, ids, exact=False):
    table = (small_ints(rng, (rows, E), 16) if exact else rng.standard_normal((rows, E))).astype(np.float32)
    dense = (small_ints(rng, E * S + S, 16) if exact else rng.standard_normal(E * S + S)).astype(np.float32)
    emb, out = tower_forward(dev, table, dense, E, S, ids)
    assert np.array_equal(emb.view(np.uint32), table[ids].view(np.uint32))
    ref, scale = reference(table[ids], dense[:E * S].reshape(E, S), 1.0, dense[E * S:], None)
    if exact:
        assert np.array_equal(out, ref.astype(np.float32))
    else:
        assert (np.abs(out - ref) <= (E + 3) * U * scale).all()


@pytest.mark.parametrize("E,S,n", [(5, 7, 1000), (13, 33, 1), (64, 128, 777), (3, 1, 129), (128, 128, 2048), (30, 66, 65)])
def test_tower_forward_matches_float64_reference(dev, E, S, n):
    """out = table[ids] W + b: the gathered rows bit for bit, out within the fp32 bound; widths that are not multiples
    of 4 take the scalar gather, ids repeat (n > rows here) and n = 1 is a single row."""
    rng = np.random.default_rng(E * 1000 + S + n)
    ids = rng.integers(0, 300, size=n).astype(np.int32)
    if n > 1:
        ids[-1] = ids[0]                                           # at least one repeat
    check_tower(dev, rng, 300, E, S, ids)
    check_tower(dev, rng, 300, E, S, ids, exact=True)


# ---- more row tiles than gridDim.y allows ---------------------------------------------------------------------------
def test_sgemm_past_65535_row_tiles(dev):
    M, N, K = GRID_Y_MAX * 64 + 65, 4, 4                  # 4 194 305 rows, 65 537 row tiles of 64
    rng = np.random.default_rng(5)
    Al, Bl, bias = small_ints(rng, (M, K), 16), small_ints(rng, (K, N), 16), small_ints(rng, N, 4)
    got = run(dev, KERNELS[0], Al, Bl, 0, 0, 1.0, 0, bias)
    assert np.array_equal(got, reference(Al, Bl, 1.0, bias, None)[0].astype(np.float32))


def test_gemm_tf32_past_65535_row_tiles(dev):
    M, N, K = GRID_Y_MAX * 128 + 129, 4, 4                # 8 388 609 rows, 65 537 row tiles of 128
    rng = np.random.default_rng(6)
    Al, Bl, bias = small_ints(rng, (M, K), 16), small_ints(rng, (K, N), 16), small_ints(rng, N, 4)
    got = run(dev, KERNELS[1], Al, Bl, 0, 0, 1.0, 0, bias)
    assert np.array_equal(got, reference(Al, Bl, 1.0, bias, None)[0].astype(np.float32))


def test_tower_forward_past_65535_row_tiles(dev):
    """Scoring every user of a table above 4.2 M rows in one call (ShardedTwoTowerNet.score_vectors, the retrieval index
    build) runs the tower over that many rows."""
    rng = np.random.default_rng(7)
    ids = rng.integers(0, 5000, size=GRID_Y_MAX * 64 + 65).astype(np.int32)
    check_tower(dev, rng, 5000, 4, 4, ids, exact=True)


# ---- rejections -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["lda", "ldb", "ldc"])
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("kern", KERNELS, ids=str)
def test_leading_dimension_below_its_minimum_is_rejected(dev, kern, which, ta, tb):
    """lda >= (trans_a ? M : K), ldb >= (trans_b ? K : N), ldc >= N, else BRK_E_ARG before any launch, C untouched.
    Each buffer holds its operand at the minimal leading dimension, so no access would leave it even if launched."""
    Nn = _nn()
    M, N, K = 72, 40, 56                                           # distinct, multiples of 4
    ld = {"lda": M if ta else K, "ldb": K if tb else N, "ldc": N}
    ld[which] -= 4 if kern.tf32 else 1                             # still a multiple of 4 for brk_gemm_tf32
    Ad = torch.ones(M * K, device=dev)
    Bd = torch.ones(K * N, device=dev)
    Cd = torch.full((M * N,), float(SENTINEL), device=dev)
    rc = kern.fn()(Nn.ctx(dev), Nn.ptr(Ad), Nn.ptr(Bd), Nn.ptr(Cd), None, M, N, K, ld["lda"], ld["ldb"], ld["ldc"], ta, tb,
                   1.0, 0, Nn.stream_ptr())
    torch.cuda.synchronize()
    assert rc == BRK_E_ARG, rc
    assert "below the stored row length" in Nn.lib().brk_last_error().decode()
    assert bool((Cd == float(SENTINEL)).all())


@pytest.mark.parametrize("what", ["A base", "B base", "lda", "ldb"])
def test_gemm_tf32_misaligned_operands_are_rejected(dev, what):
    """brk_gemm_tf32 copies operands in 16-byte pieces: a base off 16-byte alignment or a leading dimension that is
    not a multiple of 4 floats returns BRK_E_ALIGN (callers then take brk_sgemm), C untouched."""
    Nn = _nn()
    M, N, K = 64, 64, 64
    a_off, b_off = int(what == "A base"), int(what == "B base")
    lda, ldb = K + (what == "lda"), N + (what == "ldb")
    Ad = torch.ones(M * lda + 4, device=dev)
    Bd = torch.ones(K * ldb + 4, device=dev)
    Cd = torch.full((M * N,), float(SENTINEL), device=dev)
    rc = Nn.lib().brk_gemm_tf32(Nn.ctx(dev), _addr(Ad, a_off), _addr(Bd, b_off), Nn.ptr(Cd), None, M, N, K, lda, ldb, N, 0, 0,
                                1.0, 0, Nn.stream_ptr())
    torch.cuda.synchronize()
    assert rc == BRK_E_ALIGN, rc
    assert bool((Cd == float(SENTINEL)).all())
