"""Top-K scoring and ranking metrics -- drop-in mirror of the reference's trainers/topKmetrics.py
(topKRatings, topKMetrics) and src/origin_models/svd/topKMetrics.py (getAverage).

The reference scores one (user, item) pair per model.predict call and keeps the best k with a
Python insertion loop (topKmetrics.py:17-72), then probes a Python set per recommendation
(:74-99).  Here topKRatings is one fused scoring + top-K kernel launch over all users (csrc/topk.cu)
and topKMetrics one counting kernel (csrc/metrics.cu).  Return formats are the reference's:
topKRatings -> [(user, [(score, item), ... k]), ...]; topKMetrics -> the same 7-key dict.

Reference defects not reproduced (SURVEY.md section 0.5): the non-"NFC" branch of topKRatings builds
an empty list and raises IndexError; __topk raises for k == 1 and k > len(items).
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import hotpath as H
from . import synth


def device_topk(user_vectors, item_vectors, k):
    """(scores [U,k], item rows [U,k]) for dot-product models -- BruteForce semantics."""
    return H.BruteForceIndex(k).index(item_vectors)(user_vectors)


def exclusion_pairs_csr(pairs, usersId, itemsId, device):
    """(user, item) pairs in the caller's id space -> exclusion CSR (hotpath.exclusion_csr) over the positions of
    usersId (rows) and itemsId (columns).  Pairs whose user or item is not listed are ignored; an id listed twice
    gets the pair at each of its positions."""
    upos, ipos = {}, {}
    for r, u in enumerate(usersId):
        upos.setdefault(u, []).append(r)
    for c, i in enumerate(itemsId):
        ipos.setdefault(i, []).append(c)
    rows, cols = [], []
    for u, i in pairs:
        ru, ci = upos.get(u), ipos.get(i)
        if ru is not None and ci is not None:
            for r in ru:
                rows.extend([r] * len(ci)); cols.extend(ci)
    return H.exclusion_csr(np.asarray(rows, dtype=np.int64), np.asarray(cols, dtype=np.int64), len(usersId), device)


def topKRatings(k, model, usersId, itemsId, mtype=None, exclude=None):
    """Top-k (score, item) lists for every user in usersId over the catalog itemsId.
    `model` must offer score_vectors(usersId, itemsId) -> (user_vectors, item_vectors) for dot-product
    models (BPR, two-tower), or score_all(usersId, itemsId, k) for models with a non-factorised
    scorer (mtype == "NFC": NeuMF, reference topKmetrics.py:29-33).  `exclude`: (user, item) pairs to leave out of
    that user's list, such as the training interactions; pairs outside usersId / itemsId are ignored.  A user with
    fewer than k items left gets a shorter list."""
    usersId = list(usersId); itemsId = list(itemsId)
    dev = torch.device("cuda", torch.cuda.current_device())
    csr = None if exclude is None else exclusion_pairs_csr(exclude, usersId, itemsId, getattr(model, "device", dev))
    if mtype == "NFC" or not hasattr(model, "score_vectors"):
        if csr is None:
            vals, idx = model.score_all(usersId, itemsId, k)
        else:
            vals, idx = model.score_all(usersId, itemsId, k, exclude=csr)
    else:
        uv, iv = model.score_vectors(usersId, itemsId)
        if csr is None:
            vals, idx = device_topk(uv, iv, k)
        else:
            csr = (csr[0].to(uv.device), csr[1].to(uv.device))
            vals, idx = H.BruteForceIndex(k).index(iv).query_with_exclusions(uv, csr)
    vals = vals.cpu().numpy(); idx = idx.cpu().numpy()
    return [(u, [(vals[r, j], itemsId[idx[r, j]]) for j in range(idx.shape[1]) if idx[r, j] >= 0])
            for r, u in enumerate(usersId)]


def topk_counts(ids, user_rows, pos_users, pos_items, num_users):
    """Device counting core: ids [U,k] int32 item ids (device), user_rows [U] int32 user ids or None,
    positives as int arrays.  Returns (tp, hits, ndcg_sum, n_distinct_positives)."""
    dev = ids.device
    pu = np.asarray(pos_users, dtype=np.int64); pi = np.asarray(pos_items, dtype=np.int64)
    n_items_key = int(pi.max()) + 1 if len(pi) else 1
    key = np.unique(pu * n_items_key + pi)                       # set() semantics: distinct pairs
    pu, pi = (key // n_items_key).astype(np.int32), (key % n_items_key).astype(np.int32)
    csr_users = max(int(num_users), int(pu.max()) + 1 if len(pu) else 1)
    indptr, sitems = synth.build_csr(pu, pi, csr_users)
    indptr_d = torch.from_numpy(indptr).to(dev)
    sitems_d = torch.from_numpy(sitems if len(sitems) else np.zeros(1, np.int32)).to(dev)
    counts = torch.zeros(2, dtype=torch.int64, device=dev)
    ndcg = torch.zeros(1, dtype=torch.float64, device=dev)
    ids = ids.contiguous()
    U, k = ids.shape
    N.check(N.lib().brk_topk_metrics(N.ctx(dev), N.ptr(ids), U, k, N.ptr(user_rows) if user_rows is not None else None,
                                     N.ptr(indptr_d), N.ptr(sitems_d), csr_users, N.ptr(counts), N.ptr(ndcg),
                                     N.stream_ptr()), "brk_topk_metrics")
    c = counts.cpu().numpy()
    return int(c[0]), int(c[1]), float(ndcg.item()), len(key)


def topKMetrics(predictions, positives, usersId, itemsId, ndcg=False):
    """Same contract as the reference (topKmetrics.py:74-99): predictions is the topKRatings list,
    positives an iterable of (user, item).  Ids of any hashable type are mapped to dense ints on the
    host; the counting runs on the device.  Raises ZeroDivisionError like the reference when there
    are no positives.  ndcg=True adds the 'ndcg' key (not in the reference)."""
    usersId = list(usersId); itemsId = list(itemsId)
    nbrUser, nbrItem = len(usersId), len(itemsId)
    umap, imap = {}, {}

    def uid(u):
        return umap.setdefault(u, len(umap))

    def iid(i):
        return imap.setdefault(i, len(imap))

    k = max((len(t) for _, t in predictions), default=0)
    ids = np.full((len(predictions), max(k, 1)), -1, dtype=np.int32)
    rows = np.empty(len(predictions), dtype=np.int32)
    for r, (u, topk) in enumerate(predictions):
        rows[r] = uid(u)
        for j, (_, i) in enumerate(topk):
            ids[r, j] = iid(i)
    real = set(positives)
    pu = np.fromiter((uid(u) for u, _ in real), dtype=np.int64, count=len(real))
    pi = np.fromiter((iid(i) for _, i in real), dtype=np.int64, count=len(real))
    n_rec = int((ids >= 0).sum())
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    tp, hits, ndcg_sum, n_real = topk_counts(torch.from_numpy(ids).to(dev), torch.from_numpy(rows).to(dev), pu, pi,
                                             len(umap))
    fp = n_rec - tp
    fn = n_real - tp
    tn = nbrUser * nbrItem - tp - fp - fn
    out = {"tp": tp, "tn": tn, "fp": fp, "fn": fn, "precision": tp / (tp + fp), "recall": tp / (tp + fn),
           "hitRate": hits / nbrUser}
    if ndcg:
        out["ndcg"] = ndcg_sum / nbrUser
    return out


def getAverage(results):
    """src/origin_models/svd/topKMetrics.py:101-110."""
    average = {}
    for key in results[0]:
        average[key] = 0
        for result in results:
            average[key] += result[key]
        average[key] /= len(results)
    return average


# ---- the reference's module-private helpers (trainers/topKmetrics.py:45-72), kept for callers that reach for them ------
var = {"__currentModel": None, "__currentUserId": None}


def __predictForCurrentUser(i):
    """(prediction, item) of the current model / user for one item (:45-49): one model.predict call per pair -- the
    slow path the fused kernels replace; kept for models that only offer predict([users], [items])."""
    return (var["__currentModel"].predict([np.array([var["__currentUserId"]]), np.array([i])]), i)


def __topk(l, k):
    """The k best (score, item) entries of l, best first; among equal scores the earlier entry wins -- what the
    reference's insertion loop (:51-72) computes (held to its executed outputs: tests/golden/topk_golden.json).
    Python's sort is stable, and stays so under reverse=True."""
    return sorted(l, key=lambda x: x[0], reverse=True)[:k]


def __insertSorted(l, val):
    """Inserts val into the descending list l behind every entry that is not smaller (:63-72)."""
    i = len(l)
    while i > 0 and l[i - 1][0] < val[0]:
        i -= 1
    l.insert(i, val)

