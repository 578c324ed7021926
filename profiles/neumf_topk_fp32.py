"""Full-catalog top-k of the fp32 NeuMF models: the fused index (NeuMFNet.topk_index_fp32, csrc/neumf_topk_fp32.cu)
against score_all (the forward over every pair + materialised scores + brk_topk_rows), one GPU command, one JSON file
(argv[1], default r07_neumf_topk_fp32.json in the working directory).  The card's name and power limit are read in
the same run.

W1, ML-1M shape: 6040 users x 3706 items, k = 10, for the net NeuMFModel.compileModel builds (numFactor 32, relu,
fp32) and the NFC_plain script net of NCFModel / fit_nfc_plain (numFactor 10, sigmoid, hidden (100, 50, 10)): index
call and score_all on the same model in the same process, alternated; then with the 1 000 209 synthetic interactions
(synth.make_interactions) as exclusions.
W2, 65 536 users x 250 000 items at numFactor 64 fp32, k = 10.  score_all is timed on the first SUB users only (its
cost is linear in the users) and scaled; the output says so.

CUDA events around back-to-back calls after warm-up; L2 warm (the item side stays resident between calls).  A call
includes the user-side gather and fp32 product.  Models are a few training steps from the seeded init, so the
BatchNorm statistics are not the identity.

Per-pair lane instructions are modelled by `pair_instructions` from the kernel's loop structure (two items per step);
the FFMA-issue floor is that count over 148 SMs x 128 FP32 lanes x an assumed 1.9 GHz."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from binrec_b200 import hotpath as H, synth  # noqa: E402
from binrec_b200.NCFModel import SCRIPT_SPEC  # noqa: E402
from binrec_b200.NeuMFModel import NeuMFNet  # noqa: E402

SUB = 512
SMS, LANES, CLOCK = 148, 128, 1.9e9
SIGMOID_INSTR = 20          # 1 / (1 + expf(-x)) with a true division: the expf sequence + MUFU.EX2, the division's
                            # MUFU.RCP + Newton steps + range check (an estimate, not a SASS count)


def pad4(x):
    return (x + 3) // 4 * 4


def pair_instructions(E, hidden, emf, act, hadamard):
    """Lane instructions per (user, item) pair of neumf_topk_fp32_kernel: each step handles two items, so shared
    loads of the weights count half."""
    h1, h2, h3 = hidden
    a = 1 if act == "relu" else SIGMOID_INSTR
    # layers 1 + 2, per feature c of H1 and per item: FADD, act, BN FFMA; per step: 3 loads, 2 loop
    l12 = h1 * ((2 + a) + (3 + 2) / 2 + pad4(h2) + (pad4(h2) // 4) / 2)
    # layer 3, per feature of H2: FADD, act, BN FFMA, pad4(h3) FFMA; per step one LDS.128 of (b2, s, t) + W3 row loads
    l3 = h2 * ((2 + a) + pad4(h3) + (1 + pad4(h3) // 4) / 2)
    head = h3 * (2 + a) + (2 * emf if hadamard else emf) + emf / 2 + 1 + SIGMOID_INSTR + 3
    return {"layer1_2": l12, "layer3": l3, "head": head, "total": l12 + l3 + head,
            "ffma_layer2": h1 * pad4(h2), "sigmoids": (h1 + h2 + h3 + 1) if act == "sigmoid" else 1}


def floor_ms(pairs, instr):
    return pairs * instr / (SMS * LANES * CLOCK) * 1e3


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
    """Fraction of the index's ids found in score_all's lists of the same users."""
    sv, si = net.score_all(users, np.arange(net.numItem), iv.shape[1])
    a, b = ii.cpu().numpy(), si.cpu().numpy()
    return float(np.mean([len(set(a[r]) & set(b[r])) / a.shape[1] for r in range(a.shape[0])]))


def model_entry(net, pairs, t_ms):
    ins = pair_instructions(net.E, net.hidden, net.EMF, net.act, net.mf_mode == "hadamard")
    fl = floor_ms(pairs, ins["total"])
    return {"pair_instructions_model": ins, "issue_floor_ms": fl, "floor_over_measured": fl / t_ms}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else "r07_neumf_topk_fp32.json"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown", "torch": torch.__version__, "k": 10, "l2": "warm", "w1": {}, "w2": {},
           "floor_assumptions": {"sms": SMS, "fp32_lanes_per_sm": LANES, "clock_hz": CLOCK,
                                 "sigmoid_instructions": SIGMOID_INSTR}}
    k = 10

    # ---- W1: ML-1M shape ----
    U, I = 6040, 3706
    users_np, items_np = synth.make_interactions()            # the ML-1M-shaped positives: 1 000 209 pairs
    script = dict(SCRIPT_SPEC)
    for name, E, kw in (("neumfmodel_f32", 32, dict()), ("nfc_plain_script", script.pop("numFactor"), script)):
        net = NeuMFNet(U, I, E, dropout=0.2, seed=42, device=dev, **kw)
        assert not net.tensor_cores
        train(net, dev)
        users = np.arange(U, dtype=np.int32)
        t_build = timed(lambda: net.topk_index_fp32(), 5)
        index = net.topk_index_fp32()
        t_idx, t_all = alternated(lambda: index(users, k), lambda: net.score_all(users, np.arange(I), k), 3, 5)
        iv, ii = index(users, k)
        r = {"index_build_ms": t_build, "index_call_ms": t_idx, "score_all_ms": t_all,
             "speedup_median": float(np.median(t_all) / np.median(t_idx)),
             "pairs_per_s_index": U * I / (np.median(t_idx) * 1e-3),
             "pairs_per_s_score_all": U * I / (np.median(t_all) * 1e-3),
             "id_agreement_with_score_all": agreement(net, users[:256], iv[:256], ii[:256])}
        r.update(model_entry(net, U * I, float(np.median(t_idx))))
        csr = H.exclusion_csr(users_np, items_np, U, dev)
        t_xi, t_xa = alternated(lambda: index.query_with_exclusions(users, csr, k),
                                lambda: net.score_all(users, np.arange(I), k, exclude=csr), 3, 5)
        r.update({"excl_pairs": int(len(users_np)), "excl_index_call_ms": t_xi, "excl_score_all_ms": t_xa,
                  "excl_speedup_median": float(np.median(t_xa) / np.median(t_xi))})
        res["w1"][name] = r
        print(name, json.dumps(r), flush=True)
        del net, index
        torch.cuda.empty_cache()

    # ---- W2: 65 536 users x 250 000 items, numFactor 64 fp32 ----
    U, I = 65536, 250000
    net = NeuMFNet(U, I, 64, dropout=0.2, seed=42, device=dev)
    train(net, dev)
    users = np.arange(U, dtype=np.int32)
    t_build = timed(lambda: net.topk_index_fp32(), 3)
    index = net.topk_index_fp32()
    t_idx = [timed(lambda: index(users, k), 1, warm=1) for _ in range(3)]
    sub = users[:SUB]
    t_sub = [timed(lambda: net.score_all(sub, np.arange(I), k), 1, warm=1) for _ in range(2)]
    res["w2"] = {"users": U, "items": I, "index_build_ms": t_build, "index_call_ms": t_idx,
                 "pairs_per_s_index": U * I / (np.median(t_idx) * 1e-3),
                 "score_all_subsample_users": SUB, "score_all_subsample_ms": t_sub,
                 "score_all_scaled_ms": float(np.median(t_sub) * U / SUB),
                 "note": f"score_all timed on the first {SUB} users only and scaled linearly to {U}"}
    res["w2"].update(model_entry(net, U * I, float(np.median(t_idx))))
    print("w2", json.dumps(res["w2"]), flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
