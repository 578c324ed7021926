"""Cost of tfrs Retrieval's options on the two-tower training step (TwoTowerModel(temperature=..., candidateProbKey=...,
weightKey=..., streamingFrequency=...), brk_twotower_train_step_retrieval), E = S = 128, BASELINE.json configs[2]'s
6040 users x 3706 items, Keras Adagrad, TF32 tensor cores.

For batch 1000 (one cooperative launch) and 8192 (the multi-kernel step), three variants of the same step, each captured
as one CUDA graph and replayed as the bench and TwoTowerModel.fit do:
  plain      no options (the option-free kernels)
  options    temperature 0.5, caller-supplied candidate probabilities and sample weights
  estimator  temperature 0.5, the streaming frequency estimator (alpha 0.01) instead of supplied probabilities
Rounds alternate the variants inside one process (CUDA events around --steps replays per variant and round; the median
over rounds is reported, with the spread).  The estimator on its own: the device time of tt_logq_kernel (the multi-kernel
step's estimator and column terms) from a torch.profiler pass, and estimator minus options in the one-launch step, where
the estimator runs inside the launch.  The card's name and power limit are read in the same run.  Writes --out (JSON)."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from binrec_b200.twoTower import TwoTowerModel  # noqa: E402
from twotower_sharded import card  # noqa: E402

VARIANTS = {"plain": {}, "options": dict(temperature=0.5, candidateProbKey="p", weightKey="w"),
            "estimator": dict(temperature=0.5, streamingFrequency=0.01)}


def make_step(kw, U, I, B, dev):
    m = TwoTowerModel(128, I, U, "u", "i", list(range(U)), list(range(I)), semb=128, device=dev, tensor_cores=True, **kw)
    m.compile("Adagrad", learningRate=0.1)
    g = torch.Generator(device=dev); g.manual_seed(17)
    u = torch.randint(2, U + 2, (B,), generator=g, device=dev, dtype=torch.int32)
    i = (torch.rand(B, generator=g, device=dev) ** 2 * I).to(torch.int32) + 2      # skewed items, SURVEY 8d
    rng = np.random.default_rng(5)
    p = torch.from_numpy((rng.random(B) ** 2).astype(np.float32)).to(dev)
    w = torch.from_numpy(rng.uniform(0.5, 1.5, B).astype(np.float32)).to(dev)
    extras = (p if "candidateProbKey" in kw else None, w if "weightKey" in kw else None)

    def step():
        m._train_ids(u, i, None, extras=extras)

    step()
    side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    gph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gph):
        step()
    return m, gph, step


def timed(gph, K):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        gph.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K


def logq_kernel_ms(step, K):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(K):
            step()
        torch.cuda.synchronize()
    return sum(ev.device_time_total for ev in prof.key_averages() if "tt_logq_kernel" in ev.key) / 1e3 / K


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=6040)
    ap.add_argument("--items", type=int, default=3706)
    ap.add_argument("--batches", default="1000,8192")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plimit = card()
    res = {}
    for B in (int(x) for x in a.batches.split(",")):
        runs = {k: make_step(kw, a.users, a.items, B, dev) for k, kw in VARIANTS.items()}
        for k, (_, gph, _) in runs.items():
            timed(gph, 20)                                             # warm-up of every variant
        t = {k: [] for k in runs}
        for _ in range(a.rounds):
            for k, (_, gph, _) in runs.items():
                t[k].append(timed(gph, a.steps))
        case = {f"{k}_ms_per_step": statistics.median(v) for k, v in t.items()}
        case.update({f"{k}_ms_spread": [min(v), max(v)] for k, v in t.items()})
        case["options_minus_plain_ms"] = case["options_ms_per_step"] - case["plain_ms_per_step"]
        case["estimator_minus_options_ms"] = case["estimator_ms_per_step"] - case["options_ms_per_step"]
        case["tt_logq_kernel_ms_per_step"] = logq_kernel_ms(runs["estimator"][2], 20)
        res[f"b{B}"] = case
        print(B, json.dumps(case), flush=True)
        del runs
        torch.cuda.empty_cache()
    out = {"card": name, "power_limit_w": plimit,
           "config": f"two-tower E=S=128, {a.users} users x {a.items} items, Keras Adagrad, TF32 tensor cores, items drawn "
                     "skewed (floor(I r^2)); b1000 is the one-launch step, b8192 the multi-kernel step",
           "timing": f"CUDA events around {a.steps} CUDA-graph replays per variant and round, variants alternating, median of "
                     f"{a.rounds} rounds; tt_logq_kernel from torch.profiler in a separate eager pass (0 where the step "
                     "is one launch)",
           "results": res}
    print(json.dumps(out), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
