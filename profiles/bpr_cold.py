"""BPR step (headline workload: ML-1M shape, d = 64, batch 16 384) timed the way bench.py's `value` is: L2 flushed before
every step (256 MiB written and read back), CUDA events around the step's one launch -- and back to back (hot L2)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import torch
from binrec_b200 import synth
from binrec_b200.BPRModel import BPRNet
dev = torch.device("cuda:0")
users, items = synth.make_interactions()
net = BPRNet(6040, 3706, 64, device=dev)
net.set_training_pairs(users, items); net.sample_negatives(7, 0)
B, K = 16384, 50
flush = torch.empty(64 << 20, dtype=torch.float32, device=dev); sink = torch.empty((), dtype=torch.float32, device=dev)
for k in range(5):
    net.train_steps([k], B)
ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
for k in range(K):
    flush.zero_(); torch.sum(flush, dim=0, out=sink)
    ev[k][0].record(); net.train_steps([5 + k], B); ev[k][1].record()
torch.cuda.synchronize()
ts = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
print(f"flushed L2: median {ts[K // 2]:.2f} us/step  mean {sum(ts) / K:.2f}  min {ts[0]:.2f}")
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
order = list(range(40))
net.train_steps(order, B); torch.cuda.synchronize()
e0.record(); net.train_steps(order, B); e1.record(); torch.cuda.synchronize()
print(f"hot L2, 40 steps in one launch: {e0.elapsed_time(e1) * 1e3 / len(order):.2f} us/step")
