"""Cost of mixed negative sampling on the two-tower training step (TwoTowerModel(sampledNegatives=M),
brk_twotower_train_step_sampled), E = S = 128, BASELINE.json configs[2]'s 6040 users x 3706 items, Keras Adagrad, TF32
tensor cores.

Batch 1000 with M = 0 (the option-free step), 128, 512 and 1000 -- one cooperative launch each (fused_step<false, true,
true> for M > 0: at most 8 x 16 score tiles) -- and batch 8192 with M = 0 and 1024 (the multi-kernel step either way).  Each
variant is captured as one CUDA graph and replayed, as the bench and TwoTowerModel.fit do; rounds alternate the variants
inside one process (CUDA events around --steps replays per variant and round; the median over rounds is reported, with
the spread).  The sampler on its own: the device time of tt_sample_negatives_kernel from a torch.profiler pass.  The
card's name and power limit are read in the same run.  Writes --out (JSON)."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch  # noqa: E402

from binrec_b200.twoTower import TwoTowerModel  # noqa: E402
from twotower_retrieval import timed  # noqa: E402
from twotower_sharded import card  # noqa: E402


def make_step(M, U, I, B, dev):
    m = TwoTowerModel(128, I, U, "u", "i", list(range(U)), list(range(I)), semb=128, device=dev, tensor_cores=True,
                      sampledNegatives=M or None)
    m.compile("Adagrad", learningRate=0.1)
    g = torch.Generator(device=dev); g.manual_seed(17)
    u = torch.randint(2, U + 2, (B,), generator=g, device=dev, dtype=torch.int32)
    i = (torch.rand(B, generator=g, device=dev) ** 2 * I).to(torch.int32) + 2      # skewed items, SURVEY 8d

    def step():
        m._train_ids(u, i, None)

    step()
    side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    gph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gph):
        step()
    return m, gph, step


def sampler_kernel_ms(step, K):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(K):
            step()
        torch.cuda.synchronize()
    return sum(ev.device_time_total for ev in prof.key_averages() if "tt_sample_negatives_kernel" in ev.key) / 1e3 / K


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=6040)
    ap.add_argument("--items", type=int, default=3706)
    ap.add_argument("--cases", default="1000:0,128,512,1000;8192:0,1024")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, plimit = card()
    res = {}
    for case in a.cases.split(";"):
        B, Ms = case.split(":")
        B, Ms = int(B), [int(x) for x in Ms.split(",")]
        runs = {M: make_step(M, a.users, a.items, B, dev) for M in Ms}
        for _, gph, _ in runs.values():
            timed(gph, 20)                                             # warm-up of every variant
        t = {M: [] for M in runs}
        for _ in range(a.rounds):
            for M, (_, gph, _) in runs.items():
                t[M].append(timed(gph, a.steps))
        out = {f"m{M}_us_per_step": 1e3 * statistics.median(v) for M, v in t.items()}
        out.update({f"m{M}_us_spread": [1e3 * min(v), 1e3 * max(v)] for M, v in t.items()})
        out.update({f"m{M}_sampler_kernel_us": 1e3 * sampler_kernel_ms(runs[M][2], 20) for M in Ms if M})
        res[f"b{B}"] = out
        print(B, json.dumps(out), flush=True)
        del runs
        torch.cuda.empty_cache()
    out = {"card": name, "power_limit_w": plimit,
           "config": f"two-tower E=S=128, {a.users} users x {a.items} items, Keras Adagrad, TF32 tensor cores, items drawn "
                     "skewed (floor(I r^2)); b1000: one launch for every M (fused_step<false, true, true> for M > 0), "
                     "b8192: the multi-kernel step",
           "timing": f"CUDA events around {a.steps} CUDA-graph replays per variant and round, variants alternating, median of "
                     f"{a.rounds} rounds with [min, max]; the sampler kernel from torch.profiler in a separate eager pass",
           "results": res}
    print(json.dumps(out), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
