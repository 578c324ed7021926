"""Global in-batch negatives (ShardedTwoTowerNet(global_negatives=True), brk_twotower_step_global) against the per-replica
loss, E = S = 128, Keras Adagrad, TF32 tensor cores, 1 M users x 200 k items row-sharded.  Run on one GPU as a plain
script (emulate = 1, 2, 8: one process issues the phases of every emulated rank), or under torchrun with one rank per
GPU (real peer memory and barriers).

For global batch 1000 and 8192 (uniform ids): device-timed whole steps after warm-up (CUDA events, max over ranks) with
per-replica and with global negatives, and, from a separate torch.profiler pass over the global-negatives steps, the
device time per step of the added kernels: the peer gather, the two phase barriers (real ranks only), the rectangular
softmax and the owner reduce.  Under emulation the per-replica step trains the whole batch as one replica (the one-GPU
step) and the global step runs every emulated rank's phases in turn, so the difference there is the cost of the split,
not of the network.  The card's name and power limit are read in the same run.  Rank 0 writes --out (JSON)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from binrec_b200 import distributed as D  # noqa: E402
from binrec_b200.sharded import ShardedTwoTowerNet  # noqa: E402
from twotower_sharded import card, ids, max_over_ranks  # noqa: E402

ADDED = {"gather": "gather_blocks_kernel", "barrier": "peer_barrier_kernel", "softmax": "global_softmax_kernel",
         "owner_reduce": "owner_reduce_kernel"}


def step_fn(net, us, its, B, G, real):
    """Step k on this rank's slice of global batch k (every emulated rank's slice under emulation)."""
    def run(k):
        u, i = us[k % len(us)], its[k % len(its)]
        if real:
            lo, hi = D.local_slice(B)
            split = [D.local_slice(B, r, G)[1] - D.local_slice(B, r, G)[0] for r in range(G)]
            net.train_on_batch(u[lo:hi], i[lo:hi], split=split if net.global_negatives else None)
        else:
            net.train_on_batch(u, i)
    return run


def time_steps(run, net, K, W, dev):
    for k in range(W):
        run(k)
    torch.cuda.synchronize(); D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        run(k)
    e1.record(); torch.cuda.synchronize()
    net.check()
    return max_over_ranks(e0.elapsed_time(e1) / K, dev)


def added_kernels(run, K):
    """Device time per step (ms) of the kernels the global mode adds, summed over the launches of a step."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(K):
            run(k)
        torch.cuda.synchronize()
    tot = {key: 0.0 for key in ADDED}
    for ev in prof.key_averages():
        for key, name in ADDED.items():
            if name in ev.key:
                tot[key] += ev.device_time_total / 1e3 / K          # us -> ms, per step
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=1_000_000)
    ap.add_argument("--items", type=int, default=200_000)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--semb", type=int, default=128)
    ap.add_argument("--batches", default="1000,8192")
    ap.add_argument("--emulate", default="1,2,8")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    D.init_from_env()
    world, rank = D.world_size(), D.rank()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    name, plimit = card()
    E, S, U, I = a.dim, a.semb, a.users, a.items
    real = world > 1
    gs = [world] if real else [int(x) for x in a.emulate.split(",")]
    res = {}
    for B in (int(x) for x in a.batches.split(",")):
        g = torch.Generator(device=dev); g.manual_seed(4321)                    # the same global batches on every rank
        us, its = ids(g, U, (8, B), False, dev), ids(g, I, (8, B), False, dev)
        for G in gs:
            case = {}
            for mode in ("per_replica", "global"):
                net = ShardedTwoTowerNet(U, I, E, S, device=dev, seed=7, emulate=0 if real else G,
                                         global_negatives=mode == "global")
                run = step_fn(net, us, its, B, G, real)
                case[mode + "_ms_per_step"] = time_steps(run, net, a.steps, a.warmup, dev)
                if mode == "global":
                    case["global_added_kernels_ms_per_step_rank0"] = added_kernels(run, min(a.steps, 10))
                del net
                torch.cuda.empty_cache()
            case["global_minus_per_replica_ms"] = case["global_ms_per_step"] - case["per_replica_ms_per_step"]
            key = f"b{B}/{'N' if real else 'emulate'}{G}"
            res[key] = case
            if rank == 0:
                print(key, json.dumps(case), flush=True)
    out = {"card": name, "power_limit_w": plimit, "world": world,
           "config": f"two-tower E={E} S={S}, {U} users x {I} items row-sharded, Keras Adagrad, TF32 tensor cores, "
                     "uniform ids, global batch as in the key",
           "timing": f"CUDA events around {a.steps} whole steps after {a.warmup} warm-up steps, max over ranks; added kernels "
                     "from torch.profiler device times in a separate pass (summed over the emulated ranks' launches)",
           "results": res}
    if not real:
        out["torchrun"] = "not measured here: N = 2 / 4 / 8 need that many GPUs (run under torchrun)"
    if rank == 0:
        print(json.dumps(out), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(out, f, indent=1)
    if real:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
