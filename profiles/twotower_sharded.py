"""Row-sharded two-tower training (sharded.ShardedTwoTowerNet) at BASELINE.json configs[3] row counts with the two-tower
width of configs[2]: 20 M users x 2 M items, E = S = 128, Keras Adagrad.  Run on one GPU as a plain script, or under
torchrun with one rank per GPU.

For local batch 1024 (the one-launch step) and 8192 (the multi-kernel step), uniform and cubic-skew ids (id =
floor(N r^3)): device-timed whole steps after warm-up (CUDA events, max over ranks), global interactions/s, the per-step
split on rank 0 (step kernel(s), peer barrier, row Adagrad, Dense all-reduce + Adagrad, each bracketed by events in a
separate pass), and a roofline: HBM bytes at the owners against the copy peak measured in the same run, NVLink bytes
(G - 1)/G * (row gathers + row-gradient REDs) against 770 GB/s.  At world size 2 it also times the ML-1M shape (6040 x
3706, E = S = 128, local batch 1000) sharded against the mirrored TwoTowerModel on the same global batches.
The card's name and power limit are read in the same run.  Rank 0 writes --out (JSON)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from binrec_b200 import _native as N  # noqa: E402
from binrec_b200 import distributed as D  # noqa: E402
from binrec_b200 import hotpath as H  # noqa: E402
from binrec_b200.sharded import ShardedTwoTowerNet  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        pl = float(pl)
    except Exception as e:                                       # noqa: BLE001 - reported, not hidden
        pl = f"not read ({e!r})"
    return name, pl


def copy_peak_gbs(dev):
    """Device-to-device copy of 2 GiB (read + write bytes over time): the HBM peak the roofline uses."""
    n = 1 << 29
    a = torch.empty(n, dtype=torch.float32, device=dev); b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record(); torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / 10
    del a, b
    torch.cuda.empty_cache()
    return 2 * n * 4 / s / 1e9


def max_over_ranks(x, dev):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    if D.world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def ids(g, N_, shape, skew, dev):
    r = torch.rand(shape, generator=g, device=dev)
    return (2 + N_ * (r ** 3 if skew else r)).to(torch.int32).clamp_(max=N_ + 1)


def time_steps(net, us, its, K, W, dev):
    for k in range(W):
        net.train_on_batch(us[k % len(us)], its[k % len(its)])
    torch.cuda.synchronize(); D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        net.train_on_batch(us[k % len(us)], its[k % len(its)])
    e1.record(); torch.cuda.synchronize()
    net.check()
    return max_over_ranks(e0.elapsed_time(e1) / K, dev)


def split_steps(net, us, its, K, dev):
    """Rank 0's per-step split, each piece bracketed by events (this pass is not the one the step time comes from)."""
    lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()
    opt = net.optimizer
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    acc = [0.0] * 4
    for k in range(K):
        ev[0].record()
        net.forward_backward(us[k % len(us)], its[k % len(its)])
        ev[1].record()
        if net.barrier is not None:
            net.barrier()
        ev[2].record()
        tabs = [net.user.local, net.item.local] if net.barrier is not None else \
            [t.tables[r] for t in (net.user, net.item) for r in range(net.G)]
        N.check(lib.brk_adagrad_rows(ctx, H._pack(tabs), len(tabs), opt.lr, opt.eps, st), "brk_adagrad_rows")
        ev[3].record()
        if net.barrier is not None:
            D.all_reduce_sum_(net.grad_arena, net._reducer)
        N.check(lib.brk_adagrad_dense(ctx, H._pack(net.dense), 2, opt.lr, opt.eps, st), "brk_adagrad_dense")
        ev[4].record()
        torch.cuda.synchronize()
        for j in range(4):
            acc[j] += ev[j].elapsed_time(ev[j + 1])
    net.check()
    out = dict(zip(("step_kernels_ms", "peer_barrier_ms", "row_adagrad_ms", "dense_allreduce_adagrad_ms"), [a / K for a in acc]))
    if net.barrier is None:                                    # one process holds every shard: no barrier, no all-reduce
        out["peer_barrier_ms"] = "n/a (one rank)"
        out["dense_adagrad_ms"] = out.pop("dense_allreduce_adagrad_ms")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=20_000_000)
    ap.add_argument("--items", type=int, default=2_000_000)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--semb", type=int, default=128)
    ap.add_argument("--batches", default="1024,8192")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    D.init_from_env()
    G, rank = D.world_size(), D.rank()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    name, plimit = card()
    peak = copy_peak_gbs(dev)
    E, S, U, I = a.dim, a.semb, a.users, a.items
    res = {}
    net = ShardedTwoTowerNet(U, I, E, S, device=dev, seed=7)
    for B in (int(x) for x in a.batches.split(",")):
        for dist_name in ("uniform", "cubic"):
            g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
            nb = 8
            us, its = ids(g, U, (nb, B), dist_name == "cubic", dev), ids(g, I, (nb, B), dist_name == "cubic", dev)
            ms = time_steps(net, us, its, a.steps, a.warmup, dev)
            split = split_steps(net, us, its, min(a.steps, 20), dev)
            # bytes per step at the owners (per rank, averaged over the 8 batches): the one-launch step gathers each row
            # twice (phase F and the re-gather of phase G), the multi-kernel step once; each row gradient is a RED (read +
            # write at the owner); the row pass reads and writes w, m, g of every distinct touched row
            passes = 2 if B <= 1536 else 1
            distinct = sum(int(torch.unique(x[k]).numel()) for x in (us, its) for k in range(nb)) / nb
            row = 4 * E
            hbm = B * 2 * row * passes + B * 2 * row * 2 + distinct * 6 * row
            link = (G - 1) / G * B * 2 * row * (passes + 1)
            s = ms * 1e-3
            res[f"b{B}/{dist_name}"] = {
                "path": "one-launch (fused_step<true>)" if passes == 2 else "multi-kernel (gather/scatter sharded)",
                "ms_per_step": ms, "global_interactions_per_s": G * B / s, "split_rank0": split,
                "roofline": {"hbm_bytes_per_step_per_gpu": int(hbm), "hbm_achieved_gbs": hbm / s / 1e9, "hbm_peak_gbs": peak,
                             "hbm_frac": hbm / s / 1e9 / peak, "nvlink_bytes_per_step_per_gpu": int(link),
                             "nvlink_achieved_gbs": link / s / 1e9, "nvlink_peak_gbs": 770.0,
                             "nvlink_frac": link / s / 1e9 / 770.0,
                             "target_ms": max(hbm / (peak * 1e9), link / 770e9) * 1e3}}
            if rank == 0:
                print(f"b{B}/{dist_name}", json.dumps(res[f"b{B}/{dist_name}"]), flush=True)
            del us, its
    del net
    torch.cuda.empty_cache()
    ml1m = "not measured (needs world size 2)"
    if G == 2:
        from binrec_b200.twoTower import TwoTowerModel
        Um, Im, Bm = 6040, 3706, 1000
        g = torch.Generator(device=dev); g.manual_seed(99)                      # same global batches on both ranks
        gu, gi = ids(g, Um, (8, G * Bm), False, dev), ids(g, Im, (8, G * Bm), False, dev)
        lo, hi = D.local_slice(G * Bm)
        us, its = gu[:, lo:hi].contiguous(), gi[:, lo:hi].contiguous()
        sh = ShardedTwoTowerNet(Um, Im, 128, 128, device=dev)
        t_sh = time_steps(sh, us, its, a.steps, a.warmup, dev)
        mm = TwoTowerModel(128, Im, Um, "u", "i", list(range(Um)), list(range(Im)), semb=128, device=dev, tensor_cores=True)
        mm.compile("Adagrad", learningRate=0.1)

        class _M:                                                              # the mirrored model under the same timer
            def train_on_batch(self, u, i):
                mm._train_ids(u, i, None)

            def check(self):
                if mm._reducer is not None:
                    mm._reducer.check()
        t_mm = time_steps(_M(), us, its, a.steps, a.warmup, dev)
        ml1m = {"sharded_ms_per_step": t_sh, "mirrored_ms_per_step": t_mm, "local_batch": Bm,
                "sharded_global_interactions_per_s": G * Bm / (t_sh * 1e-3),
                "mirrored_global_interactions_per_s": G * Bm / (t_mm * 1e-3)}
    out = {"card": name, "power_limit_w": plimit, "world": G, "copy_peak_gbs": peak,
           "config": f"two-tower E={E} S={S}, {U} users x {I} items row-sharded x{G}, Keras Adagrad, TF32 tensor cores",
           "timing": f"CUDA events around {a.steps} whole steps after {a.warmup} warm-up steps, max over ranks",
           "results": res, "ml1m_n2_sharded_vs_mirrored": ml1m}
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
