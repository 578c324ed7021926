"""Cost of per-row exclusions in full-catalog top-K (BruteForceIndex.query_with_exclusions), one GPU command, one JSON
file (argv[1], default topk_exclude.json in the working directory).

W1, ML-1M shape (bench.py's topk_ml1m): 6040 users x 3706 items, d = 128, k = 10.  Exclusions: the 1 000 209 pairs of
synth.make_interactions() (power-law, ~166 per user).  Cases: no exclusions; the pairs on random Q / C; the adversarial
case where each user's n_u excluded items are its n_u best under the bf16 scores (every excluded item beats every
threshold).  Baseline: today's workaround, BruteForceIndex(k + max n_u) (the materialised route) and a device-side
filter of its lists.
W2, one 8-way item shard of configs[4]: 65 536 users x 250 000 items, d in {64, 128}, k = 10, 128 excluded ids per
user: random ids, and popularity-skewed (128 items with a large component along a direction every query shares,
excluded for every user, so they beat every threshold).

Timing as bench.py's topk_* legs: CUDA events around back-to-back calls after warm-up; a call includes the query bf16
conversion.  L2 is warm: the item index (<= 64 MB) and the lists stay resident between calls; nothing is flushed."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from binrec_b200 import hotpath as H, synth  # noqa: E402


def timed(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def filtered(idx, Q, K, k, keys, I):
    """The workaround: top-(k + max n_u) lists, then the first k entries whose (user, item) is not excluded."""
    v, i = idx(Q)
    U = Q.shape[0]
    key = torch.arange(U, device=Q.device, dtype=torch.int64)[:, None] * I + i.long()
    pos = torch.searchsorted(keys, key).clamp_max(keys.numel() - 1)
    keep = keys[pos] != key
    rank = torch.cumsum(keep.int(), 1)
    sel = keep & (rank <= k)
    col = torch.where(sel, rank - 1, k)                     # dropped entries land in a spill column
    ov = torch.full((U, k + 1), float("-inf"), device=Q.device).scatter_(1, col, v)[:, :k]
    oi = torch.full((U, k + 1), -1, dtype=torch.int32, device=Q.device).scatter_(1, col, i)[:, :k]
    return ov, oi


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "topk_exclude.json"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    res = {"nvidia_smi": smi, "l2": "warm (index and lists resident across calls, no flush)",
           "timing": "CUDA events over back-to-back calls after warm-up, query bf16 conversion included"}
    g = torch.Generator(device=dev); g.manual_seed(7)

    # ---- W1 ----
    U, I, d, k = synth.ML1M_USERS, synth.ML1M_ITEMS, 128, 10
    pu, pi = synth.make_interactions()
    indptr, ids = H.exclusion_csr(pu, pi, U, dev)
    n_u = np.diff(indptr.cpu().numpy())
    Q = torch.randn(U, d, generator=g, device=dev); Cm = torch.randn(I, d, generator=g, device=dev)
    idx = H.BruteForceIndex(k).index(Cm)
    w1 = {"shape": f"{U} x {I}, d={d}, k={k}", "pairs": int(n_u.sum()), "mean_n_u": float(n_u.mean()),
          "max_n_u": int(n_u.max())}
    w1["none_ms"] = timed(lambda: idx(Q), 50)
    w1["random_ms"] = timed(lambda: idx.query_with_exclusions(Q, (indptr, ids)), 50)
    # adversarial: user u excludes its n_u best items under the bf16 scores
    S = (Q.to(torch.bfloat16).float() @ Cm.to(torch.bfloat16).float().T)
    order = torch.argsort(S, dim=1, descending=True, stable=True)
    cols = torch.arange(I, device=dev)[None, :] < torch.from_numpy(n_u).to(dev)[:, None]
    adv = torch.where(cols, order, torch.iinfo(torch.int64).max).sort(dim=1).values
    adv_ids = adv[cols].to(torch.int32)                    # row-major: row u's n_u ids, ascending
    w1["adversarial_ms"] = timed(lambda: idx.query_with_exclusions(Q, (indptr, adv_ids)), 50)
    K = k + int(n_u.max())
    wide = H.BruteForceIndex(K).index(Cm)
    keys_rand = (torch.from_numpy(pu.astype(np.int64)).to(dev) * I + torch.from_numpy(pi.astype(np.int64)).to(dev)).sort().values
    rows = torch.repeat_interleave(torch.arange(U, device=dev), torch.from_numpy(n_u).to(dev))
    keys_adv = (rows * I + adv_ids.long()).sort().values
    w1["workaround_k"] = K
    w1["workaround_random_ms"] = timed(lambda: filtered(wide, Q, K, k, keys_rand, I), 10)
    w1["workaround_adversarial_ms"] = timed(lambda: filtered(wide, Q, K, k, keys_adv, I), 10)
    # the workaround and the fused call agree (ids; scores up to fp32 summation order of the two routes)
    for name, csr, keys in (("random", (indptr, ids), keys_rand), ("adversarial", (indptr, adv_ids), keys_adv)):
        a = idx.query_with_exclusions(Q, csr); b = filtered(wide, Q, K, k, keys, I)
        w1[f"{name}_ids_agree_with_workaround"] = float((a[1] == b[1]).float().mean().item())
        w1[f"{name}_max_score_diff"] = float((a[0] - b[0]).abs().max().item())
    res["W1"] = w1
    del S, order, adv, wide

    # ---- W2 ----
    Ub, Ib, n_ex = 65536, 250000, 128
    w2 = {"shape": f"{Ub} x {Ib}, k={k}, {n_ex} excluded per user"}
    rng = np.random.default_rng(3)
    w = Ib // n_ex                                         # one id per stratum of w items: distinct and ascending
    rnd = (np.arange(n_ex) * w)[None, :] + rng.integers(0, w, size=(Ub, n_ex))
    ip = torch.arange(0, Ub * n_ex + 1, n_ex, dtype=torch.int64, device=dev)
    rnd_ids = torch.from_numpy(rnd.reshape(-1).astype(np.int32)).to(dev)
    hot = np.sort(rng.choice(Ib, n_ex, replace=False)).astype(np.int32)
    hot_ids = torch.from_numpy(np.tile(hot, Ub)).to(dev)
    for dd in (64, 128):
        Q = torch.randn(Ub, dd, generator=g, device=dev); Cm = torch.randn(Ib, dd, generator=g, device=dev)
        Q[:, 0] = Q[:, 0].abs() + 3.0                      # a direction every query shares
        idx = H.BruteForceIndex(k).index(Cm)
        r = {"none_ms": timed(lambda: idx(Q), 5, warm=1),
             "random_ms": timed(lambda: idx.query_with_exclusions(Q, (ip, rnd_ids)), 5, warm=1)}
        Cs = Cm.clone(); Cs[torch.from_numpy(hot).long().to(dev), 0] = 60.0
        idx_s = H.BruteForceIndex(k).index(Cs)
        r["skewed_none_ms"] = timed(lambda: idx_s(Q), 5, warm=1)
        r["skewed_excluded_ms"] = timed(lambda: idx_s.query_with_exclusions(Q, (ip, hot_ids)), 5, warm=1)
        v, i = idx_s(Q)
        r["skewed_hot_items_fill_plain_lists"] = bool(np.isin(i.cpu().numpy(), hot).all())
        v, i = idx_s.query_with_exclusions(Q, (ip, hot_ids))
        r["skewed_no_hot_item_in_excluded_lists"] = bool(not np.isin(i.cpu().numpy(), hot).any())
        w2[f"d{dd}"] = r
        del Q, Cm, Cs, idx, idx_s
    res["W2"] = w2
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
