"""Full-catalog NeuMF top-k: the fused index (NeuMFNet.topk_index, csrc/neumf_topk.cu) against score_all (the forward
over every pair + materialised scores + brk_topk_rows), one GPU command, one JSON file (argv[1], default
r06_neumf_topk.json in the working directory).  The card's name and power limit are read in the same run.

W1, ML-1M shape: 6040 users x 3706 items, k = 10, for the tensor-core class graph at numFactor 32 and the He et al.
variant (E 32, mf_dim 8, Hadamard, no BatchNorm): index call and score_all on the same model in the same process,
alternated; then with the 1 000 209 synthetic interactions (synth.make_interactions) as exclusions.
W2, one configs[4]-sized item shard at numFactor 64: 65 536 users x 250 000 items, k = 10.  score_all is timed on a
subsample of the users only (SUB users; its cost is linear in the users), and the script says so in the output.

CUDA events around back-to-back calls after warm-up; L2 warm (the item side, <= 128 MB, stays resident between
calls).  The index build (item-side gather + TF32 product) is timed separately; a call includes the user-side gather
and product.  Models are a few training steps from the seeded init, so the BatchNorm statistics are not identity."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from binrec_b200 import hotpath as H, synth  # noqa: E402
from binrec_b200.NeuMFModel import NeuMFNet  # noqa: E402

SUB = 512


def timed(fn, iters, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def alternated(fa, fb, rounds, iters):
    a, b = [], []
    for _ in range(rounds):
        a.append(timed(fa, iters)); b.append(timed(fb, iters))
    return a, b


def train(net, dev, steps=3, B=4096):
    rng = np.random.default_rng(3)
    for s in range(steps):
        u = torch.from_numpy(rng.integers(0, net.numUser, B).astype(np.int32)).to(dev)
        i = torch.from_numpy(rng.integers(0, net.numItem, B).astype(np.int32)).to(dev)
        y = torch.from_numpy((rng.random(B) < 0.3).astype(np.float32)).to(dev)
        net.train_on_batch(u, i, y, first_index=s * B)
    torch.cuda.synchronize()


def agreement(net, users, iv, ii):
    """Fraction of the index's ids found in score_all's lists of the same users (TF32 first layer in both)."""
    sv, si = net.score_all(users, np.arange(net.numItem), iv.shape[1])
    a, b = ii.cpu().numpy(), si.cpu().numpy()
    return float(np.mean([len(set(a[r]) & set(b[r])) / a.shape[1] for r in range(a.shape[0])]))


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "r06_neumf_topk.json"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown", "torch": torch.__version__, "k": 10, "w1": {}, "w2": {}}
    k = 10

    # ---- W1: ML-1M shape ----
    U, I = 6040, 3706
    users_np, items_np = synth.make_interactions()            # the ML-1M-shaped positives: 1 000 209 pairs
    for name, E, kw in (("class_f32", 32, dict(tensor_cores=True)),
                        ("he_variant", 32, dict(mf_dim=8, mf_mode="hadamard", batch_norm=False, hidden=(32, 16, 8)))):
        net = NeuMFNet(U, I, E, dropout=0.2, seed=42, device=dev, **kw)
        train(net, dev)
        users = np.arange(U, dtype=np.int32)
        t_build = timed(lambda: net.topk_index(), 5)
        index = net.topk_index()
        t_idx, t_all = alternated(lambda: index(users, k), lambda: net.score_all(users, np.arange(I), k), 3, 5)
        iv, ii = index(users, k)
        r = {"index_build_ms": t_build, "index_call_ms": t_idx, "score_all_ms": t_all,
             "speedup_median": float(np.median(t_all) / np.median(t_idx)),
             "pairs_per_s_index": U * I / (np.median(t_idx) * 1e-3),
             "id_agreement_with_score_all": agreement(net, users[:256], iv[:256], ii[:256])}
        csr = H.exclusion_csr(users_np, items_np, U, dev)
        t_xi, t_xa = alternated(lambda: index.query_with_exclusions(users, csr, k),
                                lambda: net.score_all(users, np.arange(I), k, exclude=csr), 3, 5)
        r.update({"excl_pairs": int(len(users_np)), "excl_index_call_ms": t_xi, "excl_score_all_ms": t_xa,
                  "excl_speedup_median": float(np.median(t_xa) / np.median(t_xi))})
        res["w1"][name] = r
        print(name, json.dumps(r), flush=True)
        del net, index
        torch.cuda.empty_cache()

    # ---- W2: one configs[4]-sized item shard, numFactor 64 ----
    U, I = 65536, 250000
    net = NeuMFNet(U, I, 64, dropout=0.2, seed=42, device=dev, tensor_cores=True)
    train(net, dev)
    users = np.arange(U, dtype=np.int32)
    t_build = timed(lambda: net.topk_index(), 3)
    index = net.topk_index()
    t_idx = [timed(lambda: index(users, k), 3, warm=1) for _ in range(3)]
    sub = users[:SUB]
    t_sub = [timed(lambda: net.score_all(sub, np.arange(I), k), 1, warm=1) for _ in range(2)]
    res["w2"] = {"users": U, "items": I, "index_build_ms": t_build, "index_call_ms": t_idx,
                 "pairs_per_s_index": U * I / (np.median(t_idx) * 1e-3),
                 "score_all_subsample_users": SUB, "score_all_subsample_ms": t_sub,
                 "score_all_extrapolated_ms": float(np.median(t_sub) * U / SUB),
                 "note": f"score_all timed on the first {SUB} users only and scaled linearly to {U}"}
    print("w2", json.dumps(res["w2"]), flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
