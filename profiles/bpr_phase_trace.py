"""Where one BPR training step of `bpr_steps_coop` goes, phase by phase (globaltimer stamps of block 0, BRK_COOP_TRACE).

  python profiles/bpr_phase_trace.py [--launches 200] [--json OUT]

Two settings at the bench.py headline shape (ML-1M tables, d = 64, batch 16 384):
  flushed  single-step launches with L2 flushed before each one, as bench.py's `value` times them;
  hot      one 40-step launch with L2 hot (medians over its steps; the launch's last step is reported on its own).
Each setting alternates the global-memory Adam of BRK_BPR_NO_SMEM_ADAM=1 ("global": Adam operands loaded from L2 after the
gradient barrier, grid barrier after every step) with the default path ("smem": w / m / v bulk-copied into shared memory at
kernel entry, no grid barrier after a launch's last step), launch by launch, in one process.

Phases (medians, us): startup = kernel entry of block 0 -> step start; phase1 = gather + loss + gradient REDs of block 0;
barrier_a = block 0 done -> gradient barrier passed; adam = Adam of block 0's slices; barrier_b = the trailing grid barrier
(zero when the launch ends without it); step_event = CUDA events around the launch (flushed setting only)."""
import argparse, ctypes, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
os.environ["BRK_COOP_TRACE"] = "1"
import numpy as np, torch
from binrec_b200 import synth, _native as N
from binrec_b200.BPRModel import BPRNet

B, D, HOT_STEPS = 16384, 64, 40
MODES = {"global": "1", "smem": None}


def set_mode(m):
    if MODES[m]: os.environ["BRK_BPR_NO_SMEM_ADAM"] = MODES[m]
    else: os.environ.pop("BRK_BPR_NO_SMEM_ADAM", None)


def read_trace(n_steps):
    buf = (ctypes.c_uint64 * (n_steps * 8))()
    assert N.lib().brk_coop_trace_read(buf, n_steps * 8) == 0
    return np.frombuffer(buf, dtype=np.uint64).reshape(n_steps, 8).astype(np.int64)


def phases(a):
    """a: [steps, 8] stamps -> dict of per-step phase durations (us)."""
    return {"phase1": (a[:, 2] - a[:, 0]) / 1e3, "barrier_a": (a[:, 1] - a[:, 2]) / 1e3,
            "adam": (a[:, 3] - a[:, 1]) / 1e3, "barrier_b": (a[:, 6] - a[:, 3]) / 1e3}


def med(d):
    return {k: round(float(np.median(v)), 3) for k, v in d.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    lib = N.lib(); lib.brk_coop_trace_read.argtypes = [ctypes.c_void_p, ctypes.c_int32]
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        gpu = torch.cuda.get_device_name(0)
    users, items = synth.make_interactions()
    net = BPRNet(synth.ML1M_USERS, synth.ML1M_ITEMS, D, seed=42, device=dev)
    net.set_training_pairs(users, items); net.sample_negatives(7, 0)
    nb = len(users) // B
    flush = torch.empty((256 << 20) // 4, dtype=torch.float32, device=dev)
    out = {"gpu": gpu, "shape": {"users": synth.ML1M_USERS, "items": synth.ML1M_ITEMS, "d": D, "batch": B}}

    # ---- flushed: single-step launches --------------------------------------------------------------------------
    for m in MODES:                                        # warm both paths
        set_mode(m); net.train_steps(list(range(3)), B)
    torch.cuda.synchronize()
    rows = {m: [] for m in MODES}; ev_us = {m: [] for m in MODES}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for k in range(2 * args.launches):
        m = list(MODES)[k % 2]
        set_mode(m)
        flush.zero_(); torch.sum(flush, dim=0)
        e0.record(); net.train_steps([k % nb], B); e1.record()
        torch.cuda.synchronize()
        a = read_trace(1)
        rows[m].append(a[0]); ev_us[m].append(1e3 * e0.elapsed_time(e1))
    out["flushed"] = {}
    for m in MODES:
        a = np.stack(rows[m])
        r = med(phases(a))
        r["startup"] = round(float(np.median((a[:, 0] - a[:, 7]) / 1e3)), 3)
        r["entry_to_end"] = round(float(np.median((a[:, 6] - a[:, 7]) / 1e3)), 3)
        r["step_event"] = round(float(np.median(ev_us[m])), 3)
        r["launches_on_smem_adam"] = int((a[:, 4] == 1).sum())     # word 4 of step 0: which Adam the launch ran
        out["flushed"][m] = r

    # ---- hot: one 40-step launch ---------------------------------------------------------------------------------
    out["hot"] = {}
    order = [k % nb for k in range(HOT_STEPS)]
    samples = {m: [] for m in MODES}
    for rep in range(10):
        for m in MODES:
            set_mode(m)
            net.train_steps(order, B); torch.cuda.synchronize()
            samples[m].append(read_trace(HOT_STEPS))
    for m in MODES:
        a = np.stack(samples[m][1:])                       # [reps, steps, 8]; first repetition is warm-up
        inner = a[:, :-1].reshape(-1, 8)
        r = {"steps_but_last": med(phases(inner)), "last_step": med(phases(a[:, -1])),
             "step_period": round(float(np.median(np.diff(a[:, :, 0], axis=1)) / 1e3), 3)}
        out["hot"][m] = r
    set_mode("smem")
    print(json.dumps(out, indent=1))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
