"""Cost of tfrs Retrieval's options on row-sharded two-tower training (ShardedTwoTowerNet(temperature=...,
streamingFrequency=...), brk_tt_estimator_update_sharded + brk_twotower_step_sharded_retrieval) in r05's configuration
(profiles/twotower_sharded.py): 20 M users x 2 M items row-sharded, E = S = 128, Keras Adagrad, TF32 tensor cores.  Run
on one GPU as a plain script, or under torchrun with one rank per GPU.

For local batch 1024 (the one-launch step) and 8192 (the multi-kernel step), with cubic-skew items (id = floor(N r^3)),
three variants of the same whole step (train_on_batch), each its own model:
  plain      no options (fused_step<true> / the option-free multi-kernel step)
  options    temperature 0.5, caller-supplied candidate probabilities and sample weights
  estimator  temperature 0.5 and the streaming frequency estimator (alpha 0.01): update launch, peer barrier (N >= 2), step
Rounds alternate the variants inside one process (CUDA events around --steps steps per variant and round, max over
ranks); the median over rounds is reported with the spread.  Then, per batch: the device time of the update kernel
(tt_estimator_update_sharded_kernel, torch.profiler pass of its own) and, at N >= 2, the extra peer barrier (CUDA events
around the barrier calls of an eager pass).  The card's name and power limit are read in the same run.  Rank 0 writes
--out (JSON)."""
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
import torch.distributed as dist  # noqa: E402

from binrec_b200 import distributed as D  # noqa: E402
from binrec_b200.sharded import ShardedTwoTowerNet  # noqa: E402
from twotower_sharded import card, ids, max_over_ranks  # noqa: E402

VARIANTS = {"plain": {}, "options": dict(temperature=0.5), "estimator": dict(temperature=0.5, streamingFrequency=0.01)}


def run(net, batch):
    u, i, p, w = batch
    if net._est is not None:
        net.train_on_batch(u, i)
    elif net.temperature is not None:
        net.train_on_batch(u, i, cand_prob=p, weights=w)
    else:
        net.train_on_batch(u, i)


def timed(net, batches, K, dev):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    e0.record()
    for k in range(K):
        run(net, batches[k % len(batches)])
    e1.record(); torch.cuda.synchronize()
    return max_over_ranks(e0.elapsed_time(e1) / K, dev)


def update_kernel_ms(net, batches, K):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(K):
            net._est.update(batches[k % len(batches)][1])
        torch.cuda.synchronize()
    return sum(ev.device_time_total for ev in prof.key_averages() if "tt_estimator_update_sharded" in ev.key) / 1e3 / K


def barrier_ms(net, batches, K):
    """The estimator's extra barrier as it runs in the step: CUDA events around it, after each rank's update."""
    if net.barrier is None:
        return "n/a (one rank: the update and the step are ordered by the stream)"
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    tot = 0.0
    for k in range(K):
        u, i, _, _ = batches[k % len(batches)]
        net._est.update(i)
        e[0].record()
        net.barrier()
        e[1].record()
        net.forward_backward(u, i)                        # the rest of the step, so the ranks stay in lockstep
        net.apply_gradients()
        torch.cuda.synchronize()
        tot += e[0].elapsed_time(e[1])
    net.check()
    return tot / K


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=20_000_000)
    ap.add_argument("--items", type=int, default=2_000_000)
    ap.add_argument("--batches", default="1024,8192")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    D.init_from_env()
    G, rank = D.world_size(), D.rank()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    name, plimit = card()
    nets = {k: ShardedTwoTowerNet(a.users, a.items, 128, 128, device=dev, seed=7, **kw) for k, kw in VARIANTS.items()}
    res = {}
    for B in (int(x) for x in a.batches.split(",")):
        g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
        rng = np.random.default_rng(5 + rank)
        batches = []
        for _ in range(8):
            u, i = ids(g, a.users, (B,), True, dev), ids(g, a.items, (B,), True, dev)
            p = torch.from_numpy((rng.random(B) ** 2).astype(np.float32)).to(dev)
            w = torch.from_numpy(rng.uniform(0.5, 1.5, B).astype(np.float32)).to(dev)
            batches.append((u, i, p, w))
        for net in nets.values():
            timed(net, batches, 5, dev)                    # warm-up of every variant
        t = {k: [] for k in nets}
        for _ in range(a.rounds):
            for k, net in nets.items():
                t[k].append(timed(net, batches, a.steps, dev))
        for net in nets.values():
            net.check()
        case = {"path": "one launch (fused_step<true>, fused_step<true, true>)" if B <= 1536 else
                "multi-kernel (tt_logq_sharded_kernel + inbatch_softmax_kernel<true> with the options)"}
        case.update({f"{k}_ms_per_step": statistics.median(v) for k, v in t.items()})
        case.update({f"{k}_ms_spread": [min(v), max(v)] for k, v in t.items()})
        case["options_minus_plain_ms"] = case["options_ms_per_step"] - case["plain_ms_per_step"]
        case["estimator_minus_options_ms"] = case["estimator_ms_per_step"] - case["options_ms_per_step"]
        case["update_kernel_ms"] = update_kernel_ms(nets["estimator"], batches, 20)
        case["extra_barrier_ms"] = barrier_ms(nets["estimator"], batches, 20)
        res[f"b{B}"] = case
        if rank == 0:
            print(f"b{B}", json.dumps(case), flush=True)
        del batches
    out = {"card": name, "power_limit_w": plimit, "world": G,
           "config": f"two-tower E=S=128, {a.users} users x {a.items} items row-sharded x{G}, Keras Adagrad, TF32 tensor "
                     "cores, items and users drawn cubic-skewed (floor(N r^3)); options: temperature 0.5 with supplied "
                     "probabilities and weights; estimator: temperature 0.5, alpha 0.01",
           "timing": f"CUDA events around {a.steps} eager whole steps per variant and round, variants alternating, median "
                     f"of {a.rounds} rounds, max over ranks; update kernel from torch.profiler in a separate pass; extra "
                     "barrier from CUDA events around it in a separate eager pass",
           "results": res,
           "not_measured": "world sizes above the one of this run" if G > 1 else
                           "N >= 2: the extra barrier and every multi-GPU step time (this run had one GPU)"}
    if rank == 0:
        print(json.dumps(out), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(out, f, indent=1)
    if G > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
