"""Python face of the C ABI: device-resident embedding tables, the fused kernels and the Keras-named
optimizers the reference's model code asks for.  Each function validates shapes/dtypes (raising, as
Keras would) and forwards raw device pointers to libbrk_b200.so on the current torch stream.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import _torchext as T
from . import synth


def _i32(t, name):
    if t.dtype != torch.int32:
        raise TypeError(f"{name} must be int32 (the reference feeds float32 ids, "
                        f"src/models/BPRModel.py:101-103; this path is int32 end to end)")
    return t.contiguous()


def _f32(t, name):
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32")
    return t.contiguous()


# ----------------------------------------------------------------------------------------------
# K1 / K5
# ----------------------------------------------------------------------------------------------
def gather_rows(table, ids, out=None):
    """out[b,:] = table[ids[b],:]  -- keras Embedding lookup (NeuMFModel.py:58-63 etc.)."""
    table = _f32(table, "table"); ids = _i32(ids, "ids")
    rows, d = table.shape
    n = ids.numel()
    if out is None and T.ops() is not None:
        N.ctx(table.device)
        return T.ops().gather_rows(table, ids)
    if out is None:
        out = torch.empty((n, d), dtype=torch.float32, device=table.device)
    N.check(N.lib().brk_gather_rows(N.ctx(table.device), N.ptr(table), rows, d, N.ptr(ids), n, N.ptr(out),
                                    N.stream_ptr()), "brk_gather_rows")
    return out


def index_skew(ids, sample=8192):
    """Share of the most frequent id among the first `sample` ids (0..1)."""
    smp = ids[:sample].long()
    return float(torch.bincount(smp).max().item()) / float(smp.numel())


def scatter_add_rows(acc, ids, vals, touched=None, mode=0):
    """acc[ids[b],:] += vals[b,:]  -- IndexedSlices gradient accumulation.
    mode 0: vector atomics; 1: per-CTA sort + segment-reduce; "auto": picks by the measured index skew -- the
    share of the most frequent id in a sample of the batch (one small device histogram + one host read): same-row
    REDs serialise in L2, so mode 1 wins once a single row takes >= 1 % of the batch (measured: 6040-row table,
    1 M ids, cubic head: 315 -> 166 us) and loses 25-60 % otherwise."""
    acc = _f32(acc, "acc"); ids = _i32(ids, "ids"); vals = _f32(vals, "vals")
    rows, d = acc.shape
    if mode == "auto":
        mode = 1 if (ids.numel() >= 4096 and index_skew(ids) >= 0.01) else 0
    if T.ops() is not None:
        N.ctx(acc.device)
        T.ops().scatter_add_rows(acc, ids, vals, touched, int(mode))
        return acc
    N.check(N.lib().brk_scatter_add_rows(N.ctx(acc.device), N.ptr(acc), rows, d, N.ptr(ids), ids.numel(),
                                         N.ptr(vals), N.ptr(touched), mode, N.stream_ptr()),
            "brk_scatter_add_rows")
    return acc


# ----------------------------------------------------------------------------------------------
# K10
# ----------------------------------------------------------------------------------------------
def philox4x32_10(ctr, key0, key1):
    ctr = ctr.contiguous()
    out = torch.empty_like(ctr)
    N.check(N.lib().brk_philox4x32_10(N.ctx(ctr.device), N.ptr(ctr), ctr.shape[0], key0 & 0xFFFFFFFF,
                                      key1 & 0xFFFFFFFF, N.ptr(out), N.stream_ptr()), "brk_philox4x32_10")
    return out


def philox_bpr_negatives(users, seed, epoch, num_items, csr_indptr, csr_items, first_index=0, out=None):
    users = _i32(users, "users")
    if csr_indptr.dtype != torch.int64 or csr_items.dtype != torch.int32:
        raise TypeError("csr_indptr must be int64 and csr_items int32")
    if out is None and T.ops() is not None:
        N.ctx(users.device)
        return T.ops().philox_bpr_negatives(users, seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, int(num_items), csr_indptr, csr_items,
                                            int(first_index))
    if out is None:
        out = torch.empty_like(users)
    N.check(N.lib().brk_philox_bpr_negatives(N.ctx(users.device), N.ptr(users), users.numel(), first_index,
                                             seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, num_items,
                                             N.ptr(csr_indptr), N.ptr(csr_items), N.ptr(out), N.stream_ptr()),
            "brk_philox_bpr_negatives")
    return out


def philox_neumf_negatives(pos_users, pos_items, n_neg, seed, epoch, first_index=0):
    pos_users = _i32(pos_users, "pos_users"); pos_items = _i32(pos_items, "pos_items")
    nu = torch.empty(n_neg, dtype=torch.int32, device=pos_users.device)
    ni = torch.empty(n_neg, dtype=torch.int32, device=pos_users.device)
    N.check(N.lib().brk_philox_neumf_negatives(N.ctx(pos_users.device), N.ptr(pos_users), N.ptr(pos_items),
                                               pos_users.numel(), n_neg, first_index, seed & 0xFFFFFFFF,
                                               epoch & 0xFFFFFFFF, N.ptr(nu), N.ptr(ni), N.stream_ptr()),
            "brk_philox_neumf_negatives")
    return nu, ni


# ----------------------------------------------------------------------------------------------
# Tables and optimizers
# ----------------------------------------------------------------------------------------------
class Table:
    """An embedding table (or a flat dense parameter) resident in HBM with its gradient
    accumulator, optimizer slots and touched-row bitmask.  Layout: row-major fp32 [rows, d]."""

    def __init__(self, w, slots=2, touched=True, slot_init=0.0, g=None):
        self.w = _f32(w, "w")
        if self.w.dim() == 1:
            self.w = self.w.view(1, -1)
        self.rows, self.d = self.w.shape
        dev = self.w.device
        # g may be a view into a flat gradient arena shared by several tables (one all-reduce per step)
        self.g = torch.zeros_like(self.w) if g is None else g.view(self.rows, self.d)
        self.m = torch.full_like(self.w, slot_init) if slots >= 1 else None
        self.v = torch.zeros_like(self.w) if slots >= 2 else None
        self.touched = torch.zeros((self.rows + 31) // 32, dtype=torch.int32, device=dev) if touched else None

    def c_struct(self):
        return N.brk_table(self.w.data_ptr(), self.g.data_ptr(),
                           self.m.data_ptr() if self.m is not None else None,
                           self.v.data_ptr() if self.v is not None else None,
                           self.touched.data_ptr() if self.touched is not None else None,
                           self.rows, self.d, 0)

    @property
    def bytes(self):
        return self.w.numel() * 4


def _pack(tables):
    arr = (N.brk_table * len(tables))(*[t.c_struct() for t in tables])
    return arr


class Adam:
    """tf.keras.optimizers.Adam with its defaults (lr 1e-3, beta 0.9/0.999, epsilon 1e-7), as the
    reference constructs it (NeuMFModel.py:89, BPRModel.py:70, bpr.py:201, NFC_plain.py:153).
    sparse='keras' reproduces Keras' dense-equivalent handling of embedding gradients exactly;
    sparse='lazy' updates only the rows hit by the batch (for tables too large for a dense pass)."""

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7, sparse="keras", device=None):
        if sparse not in ("keras", "lazy"):
            raise ValueError("sparse must be 'keras' or 'lazy'")
        self.h = N.brk_adam_hyper(learning_rate, beta_1, beta_2, epsilon)
        self.sparse = sparse
        # device state: [t (int64), beta1^t (double), beta2^t (double)] -- see brk_b200.h
        state = np.zeros(3, dtype=np.int64)
        state[1:] = np.array([1.0, 1.0], dtype=np.float64).view(np.int64)
        self.state = torch.from_numpy(state).to(device or "cuda")

    @property
    def step(self):
        return self.state[0:1]

    def apply(self, tables, dense=()):
        """One optimizer step over embedding `tables` and `dense` parameters (always dense)."""
        lib, ctx, st = N.lib(), N.ctx(self.step.device), N.stream_ptr()
        tables, dense = list(tables), list(dense)
        if self.sparse == "keras":
            allp = tables + dense
            N.check(lib.brk_adam_dense_keras(ctx, _pack(allp), len(allp), self.h, N.ptr(self.state), 1, st),
                    "brk_adam_dense_keras")
        else:
            if dense:
                N.check(lib.brk_adam_dense_keras(ctx, _pack(dense), len(dense), self.h, N.ptr(self.state), 0, st),
                        "brk_adam_dense_keras")
            N.check(lib.brk_adam_rows(ctx, _pack(tables), len(tables), self.h, N.ptr(self.state), 1, st),
                    "brk_adam_rows")


class Adagrad:
    """tf.keras.optimizers.Adagrad defaults (initial accumulator 0.1, epsilon 1e-7); the reference
    uses lr 0.1 (trainers/twoTower.py:278-279).  Untouched rows have g == 0 and do not move, so
    the dense pass and the row-sparse pass give identical results; `rows_threshold_bytes` picks."""

    INITIAL_ACCUMULATOR = 0.1

    def __init__(self, learning_rate=0.001, epsilon=1e-7, rows_threshold_bytes=64 << 20):
        self.lr, self.eps = learning_rate, epsilon
        self.rows_threshold_bytes = rows_threshold_bytes

    def apply(self, tables, dense=(), force_dense=False):
        lib, st = N.lib(), N.stream_ptr()
        tables, dense = list(tables), list(dense)
        big = [] if force_dense else [t for t in tables if t.bytes > self.rows_threshold_bytes and t.touched is not None]
        small = [t for t in tables if t not in big] + dense
        dev = (tables + dense)[0].w.device
        if small:
            N.check(lib.brk_adagrad_dense(N.ctx(dev), _pack(small), len(small), self.lr, self.eps, st),
                    "brk_adagrad_dense")
        if big:
            N.check(lib.brk_adagrad_rows(N.ctx(dev), _pack(big), len(big), self.lr, self.eps, st),
                    "brk_adagrad_rows")


def gather_rows_sharded(shards, d, ids):
    """Rows `ids` of a row-sharded table (row r on rank r % G at local row r // G; `shards`: _native.brk_shards with every
    rank's peer-mapped shard pointers): the all-to-all of looked-up rows as plain peer loads (brk_gather_rows_sharded)."""
    ids = _i32(ids, "ids")
    out = torch.empty((ids.numel(), d), dtype=torch.float32, device=ids.device)
    N.check(N.lib().brk_gather_rows_sharded(N.ctx(ids.device), C.byref(shards), d, N.ptr(ids), ids.numel(), N.ptr(out),
                                            N.stream_ptr()), "brk_gather_rows_sharded")
    return out


def scatter_add_rows_sharded(shards, d, ids, values):
    """values[b, :] added to the OWNER's accumulator row of ids[b] (16-byte REDs over NVLink, owner's touched bit set)."""
    ids = _i32(ids, "ids"); values = _f32(values, "values")
    N.check(N.lib().brk_scatter_add_rows_sharded(N.ctx(ids.device), C.byref(shards), d, N.ptr(ids), ids.numel(), N.ptr(values),
                                                 N.stream_ptr()), "brk_scatter_add_rows_sharded")


# ----------------------------------------------------------------------------------------------
# Fused BPR
# ----------------------------------------------------------------------------------------------
def bpr_fwd_bwd(user, item, u, p, n, loss_out=None, global_batch=0):
    """Fused triplet forward/backward (BPRModel.py:49-74,124-144); returns the device loss scalar."""
    u = _i32(u, "u"); p = _i32(p, "p"); n = _i32(n, "n")
    if not (u.numel() == p.numel() == n.numel()):
        raise ValueError("u, p, n must have the same length")
    if loss_out is None:
        loss_out = torch.empty(1, dtype=torch.float32, device=user.w.device)
    us, it = user.c_struct(), item.c_struct()
    N.check(N.lib().brk_bpr_fwd_bwd(N.ctx(user.w.device), C.byref(us), C.byref(it), N.ptr(u), N.ptr(p),
                                    N.ptr(n), u.numel(), global_batch, N.ptr(loss_out), N.stream_ptr()), "brk_bpr_fwd_bwd")
    return loss_out


def bpr_scores(user_w, item_w, u, p, n):
    u = _i32(u, "u"); p = _i32(p, "p"); n = _i32(n, "n")
    out = torch.empty(u.numel(), dtype=torch.float32, device=user_w.device)
    N.check(N.lib().brk_bpr_scores(N.ctx(user_w.device), N.ptr(_f32(user_w, "user_w")),
                                   N.ptr(_f32(item_w, "item_w")), user_w.shape[1], N.ptr(u), N.ptr(p),
                                   N.ptr(n), u.numel(), N.ptr(out), N.stream_ptr()), "brk_bpr_scores")
    return out


def keras_embedding_init(rows, dim, rng):
    """Keras Embedding default initializer U(-0.05, 0.05), generated on the host so that the
    oracle and the device start from identical weights."""
    return rng.uniform(-0.05, 0.05, size=(rows, dim)).astype(np.float32)


# ----------------------------------------------------------------------------------------------
# K7 / K8: full-catalog scoring + top-K (tcgen05 GEMM with a top-K epilogue)
# ----------------------------------------------------------------------------------------------
def rows_to_bf16(x):
    """fp32 [rows, d] -> bf16 [rows, dpad] (zero padded to a multiple of 64 columns)."""
    x = _f32(x, "x")
    rows, d = x.shape
    if T.ops() is not None:
        N.ctx(x.device)
        return T.ops().rows_to_bf16(x)
    dpad = N.lib().brk_bf16_padded_dim(d)
    out = torch.empty((rows, dpad), dtype=torch.bfloat16, device=x.device)
    N.check(N.lib().brk_rows_to_bf16(N.ctx(x.device), N.ptr(x), rows, d, N.ptr(out), dpad, N.stream_ptr()),
            "brk_rows_to_bf16")
    return out


MAX_FUSED_K = 32          # longest list of topk_rows and of the NeuMF top-K indexes (register lists per row)


def fused_k_cap(dpad):
    """Longest list the fused scorer (brk_score_topk_bf16 / _excl) selects for candidates of padded width `dpad`: 128
    up to dpad 128, 64 at dpad 192 and 256 (csrc/topk.cu kHeapCap / kHeapCapWide: lists beyond 32 keep a heap per row
    in shared memory beside the query tile).  BruteForceIndex takes longer lists through _call_materialised."""
    return 128 if dpad <= 128 else 64


class BruteForceIndex:
    """tfrs.layers.factorized_top_k.BruteForce as the reference uses it (trainers/twoTower.py:64-69,
    src/origin_models/svd/SVD.py:424-432): index(candidates, identifiers) once, then call(queries)
    -> (scores [U,k], identifiers [U,k]) sorted by descending score, ties -> lower candidate index."""

    def __init__(self, k=10):
        self.k = int(k)
        self._c = None
        self._identifiers = None
        self.id_offset = 0

    def index(self, candidates, identifiers=None, id_offset=0):
        self.num_candidates, self.dim = candidates.shape
        self._c = rows_to_bf16(candidates)
        self._identifiers = identifiers
        self.id_offset = int(id_offset)
        return self

    def _identify(self, ids):
        """Global candidate ids -> identifiers (when index() was given some); -1 pads stay -1."""
        if self._identifiers is None:
            return ids
        return self._identifiers[(ids - self.id_offset).clamp_min(0).long()].masked_fill(ids < 0, -1)

    def __call__(self, queries, k=None):
        if self._c is None:
            raise RuntimeError("BruteForceIndex: call index(candidates) first")
        k = min(int(k or self.k), self.num_candidates)
        if k > fused_k_cap(self._c.shape[1]):
            # lists beyond the fused kernel's cap take the materialised route: fp32 scores of a chunk of users
            # (brk_sgemm) + the multi-pass row top-k below
            return self._call_materialised(queries, k)
        if queries.shape[1] != self.dim:
            raise ValueError(f"query dim {queries.shape[1]} != candidate dim {self.dim}")
        U = queries.shape[0]
        dev = queries.device
        vals = torch.empty((U, k), dtype=torch.float32, device=dev)
        ids = torch.empty((U, k), dtype=torch.int32, device=dev)
        if U == 0:
            return vals, ids
        q = rows_to_bf16(queries)
        if T.ops() is not None:
            vals, ids = T.ops().score_topk(q, self._c, k, self.id_offset)
            return vals, self._identify(ids)
        lib, ctx = N.lib(), N.ctx(dev)
        ws_bytes = lib.brk_score_topk_workspace_bytes(ctx, U, self.num_candidates, k)
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        N.check(lib.brk_score_topk_bf16(ctx, N.ptr(q), U, N.ptr(self._c), self.num_candidates, q.shape[1], k,
                                        self.id_offset, N.ptr(vals), N.ptr(ids), N.ptr(ws), ws_bytes,
                                        N.stream_ptr()), "brk_score_topk_bf16")
        return vals, self._identify(ids)

    def query_with_exclusions(self, queries, exclusions, k=None):
        """TFRS TopK.query_with_exclusions: the call's (scores, identifiers) [U, k] with each query row's excluded
        candidates left out.  `exclusions` is either a dense int tensor [U, n] of identifiers (candidate indices when
        index() got no identifiers; entries not in the index, such as -1 padding, are ignored) or a CSR
        (indptr int64 [>= U+1], ids int32) of global candidate ids (index + id_offset), ascending within each row --
        see exclusion_csr.  Rows with fewer than k remaining candidates are padded with (-inf, -1)."""
        if self._c is None:
            raise RuntimeError("BruteForceIndex: call index(candidates) first")
        if queries.shape[1] != self.dim:
            raise ValueError(f"query dim {queries.shape[1]} != candidate dim {self.dim}")
        k = min(int(k or self.k), self.num_candidates)
        U, dev = queries.shape[0], queries.device
        if isinstance(exclusions, torch.Tensor):
            exclusions = self._dense_exclusions(exclusions, U)
        indptr, xids = _check_csr(exclusions, U, dev)
        if k > fused_k_cap(self._c.shape[1]):
            return self._call_materialised(queries, k, (indptr, xids))
        vals = torch.empty((U, k), dtype=torch.float32, device=dev)
        ids = torch.empty((U, k), dtype=torch.int32, device=dev)
        if U == 0:
            return vals, ids
        q = rows_to_bf16(queries)
        if T.ops() is not None:
            vals, ids = T.ops().score_topk_exclude(q, self._c, k, self.id_offset, indptr, xids)
            return vals, self._identify(ids)
        lib, ctx = N.lib(), N.ctx(dev)
        ws_bytes = lib.brk_score_topk_workspace_bytes(ctx, U, self.num_candidates, k)
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        N.check(lib.brk_score_topk_bf16_excl(ctx, N.ptr(q), U, N.ptr(self._c), self.num_candidates, q.shape[1], k,
                                             self.id_offset, N.ptr(indptr), N.ptr(xids), N.ptr(vals), N.ptr(ids),
                                             N.ptr(ws), ws_bytes, N.stream_ptr()), "brk_score_topk_bf16_excl")
        return vals, self._identify(ids)

    def _dense_exclusions(self, E, U):
        """Dense [U, n] identifiers -> CSR of global candidate ids (device plumbing: sort + searchsorted)."""
        if E.dim() != 2 or E.shape[0] != U or E.dtype.is_floating_point or E.dtype == torch.bool:
            raise TypeError(f"dense exclusions must be an integer tensor [{U}, n]")
        E = E.to(self._c.device)
        I = self.num_candidates
        if self._identifiers is None:
            hit = (E >= 0) & (E < I)
            cand = E.long()
        else:
            ident = torch.as_tensor(self._identifiers, device=E.device)
            sv, perm = torch.sort(ident)
            pos = torch.searchsorted(sv, E.to(sv.dtype)).clamp_max(I - 1)
            hit = sv[pos] == E.to(sv.dtype)
            cand = perm[pos]
        big = torch.iinfo(torch.int64).max
        cand = torch.where(hit, cand + self.id_offset, big).sort(dim=1).values
        n_row = hit.sum(dim=1)
        indptr = torch.zeros(U + 1, dtype=torch.int64, device=E.device)
        torch.cumsum(n_row, 0, out=indptr[1:])
        ids = cand[torch.arange(cand.shape[1], device=E.device) < n_row[:, None]].to(torch.int32)
        return indptr, ids


def sgemm(a, b, trans_b=False):
    """fp32 product a [M, K] @ b ([K, N], or [N, K] with trans_b) on the CUDA cores (csrc/twotower.cu brk_sgemm)."""
    a = _f32(a, "a"); b = _f32(b, "b")
    M, K = a.shape
    Nn = b.shape[0] if trans_b else b.shape[1]
    if (b.shape[1] if trans_b else b.shape[0]) != K:
        raise ValueError("sgemm: inner dimensions differ")
    out = torch.empty((M, Nn), dtype=torch.float32, device=a.device)
    N.check(N.lib().brk_sgemm(N.ctx(a.device), N.ptr(a), N.ptr(b), N.ptr(out), None, M, Nn, K, a.shape[1], b.shape[1], Nn, 0,
                              1 if trans_b else 0, 1.0, 0, N.stream_ptr()), "brk_sgemm")
    return out


def _bruteforce_materialised(self, queries, k, exclusions=None):
    """k above the fused cap (fused_k_cap): bf16-rounded operands like the fused kernel (so shorter and longer lists
    agree on their common prefix up to fp32 summation order), scores of <= 2^24 pairs at a time, multi-pass top-k.  `exclusions`: a checked CSR of
    global ids, masked out of each chunk's scores."""
    U, I = queries.shape[0], self.num_candidates
    dev = queries.device
    C = self._c[:, :self.dim].float().contiguous()
    vals = torch.empty((U, k), dtype=torch.float32, device=dev)
    ids = torch.empty((U, k), dtype=torch.int32, device=dev)
    chunk = max(1, (1 << 24) // max(I, 1))
    for s0 in range(0, U, chunk):
        q = _f32(queries[s0:s0 + chunk], "queries").to(torch.bfloat16).float().contiguous()
        S = sgemm(q, C, trans_b=True)
        if exclusions is not None:
            mask_excluded(S, exclusions[0][s0:s0 + S.shape[0] + 1], exclusions[1], self.id_offset)
        v, ix = topk_rows(S, k)
        vals[s0:s0 + chunk] = v; ids[s0:s0 + chunk] = torch.where(ix >= 0, ix + self.id_offset, ix)
    return vals, self._identify(ids)


BruteForceIndex._call_materialised = _bruteforce_materialised


def topk_merge(part_vals, part_ids):
    """Merges [S, U, k] partial lists (global ids) into [U, k]: score desc, id asc."""
    part_vals = _f32(part_vals, "part_vals"); part_ids = _i32(part_ids, "part_ids")
    S, U, k = part_vals.shape
    if T.ops() is not None:
        N.ctx(part_vals.device)
        return T.ops().topk_merge(part_vals, part_ids)
    vals = torch.empty((U, k), dtype=torch.float32, device=part_vals.device)
    ids = torch.empty((U, k), dtype=torch.int32, device=part_vals.device)
    N.check(N.lib().brk_topk_merge(N.ctx(part_vals.device), N.ptr(part_vals), N.ptr(part_ids), S, U, k,
                                   N.ptr(vals), N.ptr(ids), N.stream_ptr()), "brk_topk_merge")
    return vals, ids


def exclusion_csr(rows, items, num_rows, device):
    """Exclusion lists from (row, item) pairs: device (indptr int64 [num_rows + 1], ids int32), each row's items
    distinct and ascending (synth.build_csr).  Pairs with a row outside [0, num_rows) or a negative item are dropped."""
    rows = np.asarray(rows, dtype=np.int64); items = np.asarray(items, dtype=np.int64)
    keep = (rows >= 0) & (rows < num_rows) & (items >= 0)
    indptr, ids = synth.build_csr(rows[keep], items[keep], num_rows)
    if len(ids) == 0:
        ids = np.zeros(1, dtype=np.int32)          # the kernels take an address even for empty lists
    return torch.from_numpy(indptr).to(device), torch.from_numpy(ids).to(device)


def _check_csr(csr, rows, device):
    """Validates an exclusion CSR for `rows` query rows before anything is launched: types, device, shapes.  The
    offsets themselves stay on the device unread (no synchronisation); they must lie within ids."""
    indptr, ids = csr
    if not (isinstance(indptr, torch.Tensor) and isinstance(ids, torch.Tensor)):
        raise TypeError("exclusions must be a tensor or an (indptr, ids) pair of tensors")
    if indptr.dtype != torch.int64 or ids.dtype != torch.int32:
        raise TypeError("exclusion indptr must be int64 and ids int32")
    if indptr.device != torch.device(device) or ids.device != torch.device(device):
        raise ValueError(f"exclusion CSR must be on {device}")
    if indptr.dim() != 1 or indptr.numel() < rows + 1:
        raise ValueError(f"exclusion indptr has {indptr.numel()} entries, {rows + 1} needed")
    if ids.dim() != 1 or not indptr.is_contiguous() or not ids.is_contiguous():
        raise ValueError("exclusion indptr and ids must be contiguous 1-D tensors")
    if ids.numel() == 0:
        ids = torch.zeros(1, dtype=torch.int32, device=device)
    return indptr, ids


def mask_excluded(scores, indptr, ids, col_offset=0):
    """In place: scores[r, id - col_offset] = -inf for each listed id of row r inside the matrix (brk_mask_excluded)."""
    R, I = scores.shape
    indptr, ids = _check_csr((indptr, ids), R, scores.device)
    N.check(N.lib().brk_mask_excluded(N.ctx(scores.device), N.ptr(scores), R, I, int(col_offset), N.ptr(indptr), N.ptr(ids),
                                      N.stream_ptr()), "brk_mask_excluded")
    return scores


def topk_rows(scores, k, exclude=None):
    """Top-k per row of a score matrix [R, I] (score desc, ties -> lower column).  `exclude`: an (indptr, ids) CSR
    of columns to leave out per row (the input is not modified); rows left short are padded with (-inf, -1)."""
    scores = _f32(scores, "scores")
    R, I = scores.shape
    if exclude is not None:
        scores = mask_excluded(scores.clone(), exclude[0], exclude[1], 0)
    k = min(int(k), I)
    if k > MAX_FUSED_K:
        # the kernel selects at most 32 per pass: take 32, strike them out of a copy, repeat (the tie rule carries over:
        # every pass prefers the lower column among equal scores)
        work = scores.clone()
        vs, js = [], []
        for k0 in range(0, k, MAX_FUSED_K):
            v, j = topk_rows(work, min(MAX_FUSED_K, k - k0))
            vs.append(v); js.append(j)
            work.scatter_(1, j.long().clamp_min(0), float("-inf"))      # a -1 pad: the row has nothing left above -inf
        return torch.cat(vs, 1), torch.cat(js, 1)
    vals = torch.empty((R, k), dtype=torch.float32, device=scores.device)
    ids = torch.empty((R, k), dtype=torch.int32, device=scores.device)
    N.check(N.lib().brk_topk_rows(N.ctx(scores.device), N.ptr(scores), R, I, k, N.ptr(vals), N.ptr(ids),
                                  N.stream_ptr()), "brk_topk_rows")
    return vals, ids
