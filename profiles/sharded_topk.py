"""Full-catalog top-k of the row-sharded models over item ranges (sharded.ShardedTopKIndex) at BASELINE.json configs[3]
row counts: 20 M users x 2 M items, 64 wide.  Run on one GPU as a plain script, or under torchrun with one rank per GPU
(world sizes 2, 4, 8).

Per world size: the index build and users/s at k = 10 for a tensor-core ShardedNeuMFNet (E 64) and a ShardedBPRNet
(d 64), host clock around work that ends in a device synchronise, max over ranks; and the exchange step alone on
[U, 10] lists: the peer merge (publish + barrier + brk_topk_merge_peer) against the NCCL all-gather + brk_topk_merge.
On one GPU there is no exchange between devices; the script then times the merge of 8 local lists (emulate=8), the
kernel's cost without NVLink.  The card's name and power limit are read in the same run.  Rank 0 prints the results as
JSON and writes them to --out when it is given."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from binrec_b200 import distributed as D  # noqa: E402
from binrec_b200 import hotpath as H  # noqa: E402
from binrec_b200.sharded import ShardedBPRNet, ShardedNeuMFNet  # noqa: E402

NU, NI, E = 20_000_000, 2_000_000, 64


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = float(subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                                   str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout)
    except Exception as e:                                       # noqa: BLE001 - reported, not hidden
        pl = f"not read ({e!r})"
    return name, pl


def timed(fn, reps):
    """Seconds per call (max over ranks) after one warm-up call."""
    fn()
    torch.cuda.synchronize(); D.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    t = torch.tensor([(time.perf_counter() - t0) / reps], dtype=torch.float64, device="cuda")
    if D.world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def bench_index(name, make, U, reps):
    net = make()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    idx = net.topk_index()
    torch.cuda.synchronize()
    build = time.perf_counter() - t0
    users = torch.from_numpy(np.random.default_rng(1).integers(0, NU, U).astype(np.int32)).cuda()
    q = timed(lambda: idx(users, 10), reps)
    del idx, net
    torch.cuda.empty_cache()
    return {"model": name, "build_s": build, "users": U, "query_s": q, "users_per_s": U / q,
            "pairs_per_s": U * NI / q}


def bench_exchange(U, reps):
    G = D.world_size()
    k = 10
    dev = torch.device("cuda", torch.cuda.current_device())
    net = ShardedBPRNet(1024, 1024, 64, device=dev, emulate=8 if G == 1 else 0)
    v = torch.sort(torch.randn(U, k, device=dev), dim=1, descending=True).values
    i = torch.randint(0, 1 << 30, (U, k), dtype=torch.int32, device=dev)
    out_v, out_i = torch.empty_like(v), torch.empty_like(i)
    real = net.topk_index(None, k)
    lists = {r: (v, i) for r in real.parts}
    res = {"U": U, "k": k, "parts": real.G}
    # the publish (padding copy + header) and the merge of one chunk; the same lists on every rank
    res["peer_merge_ms"] = 1e3 * timed(lambda: real._exchange(lists, U, k, out_v, out_i), reps)
    if G > 1:
        res["nccl_allgather_merge_ms"] = 1e3 * timed(lambda: H.topk_merge(*D.gather_topk_parts(v, i)), reps)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the results (they are printed either way)")
    ap.add_argument("--neumf-users", type=int, default=16384)
    ap.add_argument("--bpr-users", type=int, default=65536)
    ap.add_argument("--exchange-users", type=int, default=131072)
    a = ap.parse_args()
    D.init_from_env()
    dev = torch.device("cuda", torch.cuda.current_device())
    G = D.world_size()
    name, pl = card()
    res = {"gpu": name, "power_limit_w": pl, "world": G, "shape": {"users": NU, "items": NI, "width": E, "k": 10},
           "runs": []}
    res["runs"].append(bench_index("ShardedNeuMFNet tc E64", lambda: ShardedNeuMFNet(
        NU, NI, E, dropout=0.0, device=dev, tensor_cores=True), a.neumf_users, 2))
    res["runs"].append(bench_index("ShardedBPRNet d64", lambda: ShardedBPRNet(NU, NI, E, device=dev), a.bpr_users, 3))
    res["exchange"] = bench_exchange(a.exchange_users, 20)
    if D.rank() == 0:
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(res, f, indent=1)
        print(json.dumps(res, indent=1))
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
