"""Long top-K lists (33 <= k <= 128) on the fused scorer against the materialised route they took before, one GPU
command, one JSON file (argv[1], default topk_long.json in the working directory).

W1, ML-1M shape: 6040 users x 3706 items, d = 64, k in {32, 50, 100, 128}; and k = 100 with the 1 000 209 pairs of
synth.make_interactions() as exclusions.
W2, one 8-way item shard of configs[4]: 65 536 users x 250 000 items, d in {64, 128}, k in {32, 64, 100, 128}.  The
materialised route (BruteForceIndex._call_materialised: brk_sgemm scores of <= 2^24 pairs at a time + multi-pass
brk_topk_rows) is timed on the first 512 users and scaled linearly to 65 536 ("scaled" in the keys).
W3, few users (U in {1, 128}, I in {3706, 250 000}, d = 64, k = 100): many item splits per user, so the merge counts.
k = 32 is the register-list kernel: the floor of the fused times.  At k = 128, torch.profiler (after the timed runs)
splits fused calls into the scorer and its warp-per-user merge; brk_topk_merge (thread per user, the shard merge of
sharded_topk) is timed alone at k = 128.

Outputs are compared with the materialised route on the timed rows (all of W1, the 512 users of W2): ids where the
materialised scores of neighbouring ranks are more than 1e-4 apart, and the largest score difference (the two routes
sum in different orders).

Timing: CUDA events around back-to-back calls after warm-up; a call includes the query bf16 conversion.  L2 is warm:
the item index (<= 64 MB) stays resident between calls; nothing is flushed."""
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


def agreement(fused, old):
    """ids equal where the old route's ranks are > 1e-4 apart (share of those entries, and of all), max |score diff|.
    `old` holds one rank more than `fused`, for the gap of the last entry."""
    (v, i), (rv, ri) = fused, old
    k = v.shape[1]
    gap = rv[:, :-1] - rv[:, 1:]
    safe = gap > 1e-4
    safe[:, 1:] &= gap[:, :-1] > 1e-4
    rv, ri = rv[:, :k], ri[:, :k]
    same = i == ri
    return {"ids_equal_where_gap_gt_1e-4": float(same[safe].float().mean().item()),
            "ids_equal_all": float(same.float().mean().item()),
            "max_abs_score_diff": float((v - rv).abs().max().item())}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "topk_long.json"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    res = {"nvidia_smi": smi, "l2": "warm (item index resident across calls, no flush)",
           "timing": "CUDA events over back-to-back calls after warm-up, query bf16 conversion included"}
    g = torch.Generator(device=dev); g.manual_seed(8)

    # ---- W1: ML-1M ----
    U, I, d = synth.ML1M_USERS, synth.ML1M_ITEMS, 64
    Q = torch.randn(U, d, generator=g, device=dev); Cm = torch.randn(I, d, generator=g, device=dev)
    idx = H.BruteForceIndex().index(Cm)
    w1 = {"shape": f"{U} x {I}, d={d}"}
    for k in (32, 50, 100, 128):
        r = {"fused_ms": timed(lambda: idx(Q, k), 50)}
        if k > H.MAX_FUSED_K:
            r["materialised_ms"] = timed(lambda: idx._call_materialised(Q, k), 5, warm=1)
            r["speedup"] = r["materialised_ms"] / r["fused_ms"]
            r.update(agreement(idx(Q, k), idx._call_materialised(Q, k + 1)))
        w1[f"k{k}"] = r
    pu, pi = synth.make_interactions()
    ex = H.exclusion_csr(pu, pi, U, dev)
    k = 100
    r = {"pairs": int(len(pu)), "fused_ms": timed(lambda: idx.query_with_exclusions(Q, ex, k), 50),
         "materialised_ms": timed(lambda: idx._call_materialised(Q, k, ex), 5, warm=1)}
    r["speedup"] = r["materialised_ms"] / r["fused_ms"]
    r.update(agreement(idx.query_with_exclusions(Q, ex, k), idx._call_materialised(Q, k + 1, ex)))
    w1["k100_exclusions"] = r
    res["W1"] = w1
    del Q, Cm, idx

    # ---- W2: 65 536 x 250 000 ----
    Ub, Ib, sub = 65536, 250000, 512
    w2 = {"shape": f"{Ub} x {Ib}", "materialised_timed_on_users": sub, "materialised_scale": Ub / sub}
    for dd in (64, 128):
        Q = torch.randn(Ub, dd, generator=g, device=dev); Cm = torch.randn(Ib, dd, generator=g, device=dev)
        idx = H.BruteForceIndex().index(Cm)
        rd = {}
        for k in (32, 64, 100, 128):
            r = {"fused_ms": timed(lambda: idx(Q, k), 5, warm=2)}
            r["fused_tflops"] = 2.0 * dd * Ub * Ib / (r["fused_ms"] * 1e-3) / 1e12
            if k > H.MAX_FUSED_K:
                ms = timed(lambda: idx._call_materialised(Q[:sub], k), 2, warm=1)
                r["materialised_ms_scaled"] = ms * Ub / sub
                r["speedup_vs_scaled"] = r["materialised_ms_scaled"] / r["fused_ms"]
                fused = idx(Q, k)
                r.update(agreement((fused[0][:sub], fused[1][:sub]), idx._call_materialised(Q[:sub], k + 1)))
            rd[f"k{k}"] = r
        w2[f"d{dd}"] = rd
        del Q, Cm, idx
    res["W2"] = w2

    # ---- W3: few users (single-user serving requests, small evaluation batches), k = 100 ----
    w3 = {}
    for U, I in ((1, 3706), (128, 3706), (1, 250000), (128, 250000)):
        Q = torch.randn(U, 64, generator=g, device=dev); Cm = torch.randn(I, 64, generator=g, device=dev)
        idx = H.BruteForceIndex().index(Cm)
        r = {"fused_ms": timed(lambda: idx(Q, 100), 50), "materialised_ms": timed(lambda: idx._call_materialised(Q, 100), 20)}
        r["speedup"] = r["materialised_ms"] / r["fused_ms"]
        r.update(agreement(idx(Q, 100), idx._call_materialised(Q, 101)))
        w3[f"U{U}_I{I}"] = r
    res["W3_few_users_d64_k100"] = w3

    # ---- kernel times inside fused calls (torch.profiler): scorer and merge at k = 128 ----
    kern = {}
    for U, I in ((128, 250000), (6040, 3706), (65536, 250000)):
        Q = torch.randn(U, 64, generator=g, device=dev); Cm = torch.randn(I, 64, generator=g, device=dev)
        idx = H.BruteForceIndex().index(Cm)
        idx(Q, 128); torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                idx(Q, 128)
            torch.cuda.synchronize()
        r = {}
        for e in prof.key_averages():
            for name in ("score_topk_kernel", "topk_merge_warp_kernel"):
                if name in e.key:
                    total = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                    r[name + "_ms"] = total / e.count / 1e3
        kern[f"U{U}_I{I}"] = r
    res["kernels_k128_d64"] = kern

    # ---- brk_topk_merge (thread per user; the shard merge of sharded_topk) alone, k = 128 ----
    merge = {}
    for S, U in ((4, 6040), (32, 128), (1, 65536), (8, 65536)):
        pv = torch.randn(S, U, 128, generator=g, device=dev).sort(dim=2, descending=True).values
        pi = torch.randint(0, 1 << 20, (S, U, 128), generator=g, device=dev, dtype=torch.int32)
        merge[f"S{S}_U{U}_ms"] = timed(lambda: H.topk_merge(pv, pi), 20)
    res["brk_topk_merge_k128"] = merge
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
