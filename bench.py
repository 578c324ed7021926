#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native recommender hot path.

Workload (BASELINE.json configs[1]): BPR matrix factorisation, d = 64, on synthetic binary implicit
feedback of MovieLens-1M shape (6040 users x 3706 items, 1 000 209 positives), one Philox negative
per positive, loss 1 - sigmoid (reference BPRModel.py:144), exact Keras Adam(1e-3), batch 16 384.
A "step" is one batch: fused gather + loss + scatter-add kernel, then the fused Adam pass.
Metric: training interactions (triplets) per second.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how each field is produced.
--dump-outputs DIR writes what the last timed step returned (its mean loss and the user / item tables it updated) as
DIR/<name>.npy, float32; the inputs are seeded, so two builds run with the same arguments can be compared array by array.

Beside the headline the line carries, each with its own `roofline` block:
  neumf            BASELINE.json configs[0] (NeuMF, ML-1M shape, batch 16 384): the reference class graph (numFactor 32,
                   BatchNorm, dropout) as ONE cooperative tcgen05 launch per step, device value / hot / host-fed e2e;
  neumf_he         the He et al. variant configs[0] names (8-dim Hadamard GMF + MLP 64-32-16-8);
  extras           (N = 1) two-tower, full-catalog top-K, NeuMF at configs[3] table sizes on one GPU, biased SVD;
  c4_neumf_sharded (N > 1) BASELINE.json configs[3]: 20 M x 2 M x 64 tables row-sharded over the ranks, rows and row
                   gradients exchanged inside the fused kernels over NVLink peer memory, local batch 65 536;
  c5_topk_sharded  (N > 1) BASELINE.json configs[4]: 1 M users x 2 M items, items range-sharded, lists merged;
  parity_multi     (N > 1) the data-parallel and row-sharded paths against a single-GPU run of the same global batches,
                   computed inside this very run (the driver's GPU test lease has one GPU);
  parity_check     (N = 1) per-step losses of the product against the CPU oracle's on the same seeds.
The oracle never runs in this process: every CPU leg is a subprocess (`--impl cpu_legs`), so the product process maps
nothing under oracle/.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = "train interactions/sec (BPR, d=64, ML-1M shape)"
UNIT = "interactions/s"
BATCH = 16384
DIM = 64
BYTES_PER_TRIPLET = 3 * 4 * DIM * 2          # 3 rows gathered + 3 row gradients reduced (SURVEY 8d): 1536 B
L2_FLUSH_BYTES = 256 << 20


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def traffic_bytes(world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/r02_traffic.json); N=1 only (ncu is never run on a multi-rank command)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if world != 1 or not os.path.exists(p):
        return None
    with open(p) as f:
        t = json.load(f)
    return t["dram_bytes_read_per_launch"] + t["dram_bytes_write_per_launch"]


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


def make_workload():
    from binrec_b200 import synth
    users, items = synth.make_interactions()           # ML-1M shape, skewed
    return users, items, synth.ML1M_USERS, synth.ML1M_ITEMS


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's torch-CPU BPR loop on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_loop(users, items, U, I, steps, warmup, time_budget_s=None):
    """Returns (interactions/s, steps timed, threads)."""
    from oracle import bpr as OB, bpr_torch as OT, philox as OP
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    orc = OB.BPROracle(U, I, DIM, seed=42)
    model = OT.BPRTorchCPU(orc.user, orc.item)
    n_batches = len(users) // BATCH
    need = min(n_batches, steps + warmup)
    indptr, sitems = OP.build_csr(users, items, U)
    neg = OP.bpr_negatives(users[:need * BATCH], 7, 0, I, indptr, sitems)

    def run(k):
        b = k % need
        sl = slice(b * BATCH, (b + 1) * BATCH)
        return model.step(users[sl], items[sl], neg[sl])

    for k in range(warmup):
        run(k)
    t0 = time.perf_counter()
    done = 0
    for k in range(steps):
        run(warmup + k)
        done += 1
        if time_budget_s is not None and time.perf_counter() - t0 > time_budget_s:
            break
    dt = time.perf_counter() - t0
    return done * BATCH / dt, done, threads, dt


PARITY_STEPS = 20


def cpu_parity_losses(users, items, U, I):
    """Per-step losses of the oracle port on batches 0..19 of the bench frame from the seeded initial weights: the
    product arm runs the same 20 steps (same Philox negatives, seed 7 epoch 0) and reports the largest difference."""
    from oracle import bpr as OB, bpr_torch as OT, philox as OP
    orc = OB.BPROracle(U, I, DIM, seed=42)
    model = OT.BPRTorchCPU(orc.user, orc.item)
    indptr, sitems = OP.build_csr(users, items, U)
    neg = OP.bpr_negatives(users[:PARITY_STEPS * BATCH], 7, 0, I, indptr, sitems)
    out = []
    for b in range(PARITY_STEPS):
        sl = slice(b * BATCH, (b + 1) * BATCH)
        out.append(float(model.step(users[sl], items[sl], neg[sl])))
    return out


def cpu_legs_main(args):
    """`--impl cpu_legs` (a subprocess of the product arm, rank 0, N = 1): every oracle CPU leg of the line, as one JSON
    object on stdout.  Bounded samples (about 25 s in all) of the same workloads, all host threads."""
    users, items, U, I = make_workload()
    out = {}
    val, done, threads, dt = cpu_loop(users, items, U, I, steps=100000, warmup=3, time_budget_s=10.0)
    out["bpr"] = {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                  "sample": f"{done} full batches of {BATCH} triplets in {dt:.1f} s, torch-CPU oracle port of the reference "
                            f"loop (not TensorFlow)"}
    out["bpr_parity_losses"] = cpu_parity_losses(users, items, U, I)
    out.update(extras_cpu_baselines())
    out["svd_fit"] = svd_cpu_baseline()
    print(json.dumps(out), flush=True)


def run_cpu_legs():
    """Runs the CPU legs in a child process and returns its JSON (None when it fails: the line then says so)."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu_legs"], capture_output=True, text=True,
                           timeout=600, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": (r.stderr or r.stdout)[-400:]}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    users, items, U, I = make_workload()
    val, done, threads, dt = cpu_loop(users, items, U, I, args.steps, args.warmup)
    sample = f"{done} steps x {BATCH} triplets (full batches of the same workload), torch-CPU oracle port, fp32"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": done, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(done, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[1]: BPR MF d=64, ML-1M shape, batch 16384, Keras Adam",
                   "note": "oracle port of the reference loop (TensorFlow/Keras cannot be installed here); not TensorFlow"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------
def product_arm(args):
    import torch.distributed as dist
    from binrec_b200 import hotpath as H
    from binrec_b200.BPRModel import BPRNet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    users, items, U, I = make_workload()
    n_batches = len(users) // BATCH                        # 61 full batches per epoch
    # weak scaling, mirrored synchronous data parallelism (the reference's MultiWorkerMirroredStrategy,
    # RModel.py:119-121): every rank holds the tables, trains its own 16 384-triplet batch of the global
    # batch (world x 16 384), gradients are summed by ONE NCCL all-reduce per step, identical Adam step.
    net = BPRNet(U, I, DIM, seed=42, learning_rate=1e-3, sparse_adam="keras", device=dev)
    net.set_training_pairs(users, items)
    net.sample_negatives(7, 0)
    pr = net._pairs
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=dev)
    K, W = args.steps, args.warmup

    from binrec_b200 import distributed as D
    loss_buf = torch.empty(1, dtype=torch.float32, device=dev)

    def one_step(k, ev=None):
        b = (k * world + rank) % n_batches
        sl = slice(b * BATCH, (b + 1) * BATCH)
        if ev is not None:
            ev[0].record()
        if world == 1 or net.peer is not None:
            # ONE cooperative kernel per step: fused gather+loss+scatter -> grid.sync -> exact Keras Adam (N=1), or
            # -> cross-GPU barrier -> reduce-scatter + Adam + all-gather over NVLink peer memory -> barrier (N>1)
            net.train_steps([b], BATCH, losses=loss_buf)
            if ev is not None:
                ev[1].record(); ev[2].record()
            return loss_buf
        loss = H.bpr_fwd_bwd(net.user, net.item, pr["u"][sl], pr["p"][sl], pr["n"][sl], loss_out=loss_buf,
                             global_batch=world * BATCH if world > 1 else 0)
        if ev is not None:
            ev[1].record()
        net.apply_gradients()      # N=1: fused Adam; N>1: fused reduce-scatter + Adam + all-gather over NVLink peers
        if ev is not None:
            ev[2].record()
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def flush_l2():
        # write a buffer larger than L2, then read it back: evicts everything and leaves the lines clean,
        # so the timed kernels' cold misses are not also charged the write-back of the flush's own data
        flush.zero_()
        flush_sink.copy_(flush[:flush_sink.numel()] + flush[-flush_sink.numel():])
        torch.sum(flush, dim=0, out=flush_sum)

    flush_sink = torch.empty(1024, dtype=torch.float32, device=dev)
    flush_sum = torch.empty((), dtype=torch.float32, device=dev)

    # ---- (1) device-resident value: K steps, L2 flushed between steps, CUDA events per step ------
    for k in range(W):
        flush_l2(); one_step(k)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    sampler = ClockSampler(physical_gpu_index(local)); sampler.start()
    barrier()
    wall0 = time.perf_counter()
    for k in range(K):
        flush_l2()
        one_step(W + k, evs[k])
    barrier()
    wall = time.perf_counter() - wall0
    step_ms = np.array([e[0].elapsed_time(e[2]) for e in evs])
    fb_ms = np.array([e[0].elapsed_time(e[1]) for e in evs])
    total_ms = float(step_ms.sum())
    if args.dump_outputs and rank == 0:
        # taken here: the legs below keep training the same tables
        dump_outputs(args.dump_outputs, {"loss": loss_buf, "user_embedding": net.user.w, "item_embedding": net.item.w})

    # ---- (2) same steps back to back (tables stay in L2, as in the real training loop) -----------
    order = [(k * world + rank) % n_batches for k in range(K)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    mapped_ms = None
    if world == 1 or net.peer is not None:
        net.train_steps(order[:max(W, 3)], BATCH)
        barrier()
        e0.record(); net.train_steps(order, BATCH); e1.record()
    else:
        for k in range(max(W, 3)):
            one_step(k)
        barrier()
        e0.record()
        for k in range(K):
            one_step(W + k)
        e1.record()
    barrier()
    hot_ms = e0.elapsed_time(e1)

    # ---- (3) end to end through the public API with HOST buffers --------------------------------
    hu = torch.from_numpy(users[:n_batches * BATCH].copy()).pin_memory()
    hp = torch.from_numpy(items[:n_batches * BATCH].copy()).pin_memory()
    du = torch.empty(BATCH, dtype=torch.int32, device=dev); dp = torch.empty_like(du); dn = torch.empty_like(du)
    hloss = torch.empty(K + W, dtype=torch.float32).pin_memory()

    def e2e_step(k):
        b = (k * world + rank) % n_batches
        sl = slice(b * BATCH, (b + 1) * BATCH)
        du.copy_(hu[sl], non_blocking=True); dp.copy_(hp[sl], non_blocking=True)
        H.philox_bpr_negatives(du, 7, 1, I, pr["indptr"], pr["sitems"], b * BATCH, out=dn)
        loss = net.train_on_batch(du, dp, dn)
        hloss[k:k + 1].copy_(loss, non_blocking=True)

    if world == 1 or net.peer is not None:
        # one C call enqueues K x (H2D ids, sampler, fused step, Adam, loss D2H): BPRNet.train_steps_from_host
        # host input in the loader's batch-major layout [n_batches, 2, BATCH] (pinned): one H2D per step
        packed = BPRNet.pack_host_batches(users[:n_batches * BATCH], items[:n_batches * BATCH], BATCH)
        # warm-up = one untimed pass over the SAME K host batches (what every epoch after the first sees): the first DMA out of a
        # page-locked host page pays its address translation (a first 20-step call measured 513 us, every later one 380-396:
        # profiles/e2e_k20.py), and all launch shapes of the chunk plan have run once
        # -- two passes when the call is short: the second 20-step call still measured 440 us against 380-395 from the third on
        hwarm = torch.empty(K, dtype=torch.float32).pin_memory()
        for _ in range(2 if K <= 64 else 1):
            net.train_steps_from_host(packed, None, order, BATCH, 7, 1, hwarm)
        barrier()
        # host clock from before the call to after the synchronize that follows it (no CUDA events inside: two event records are
        # 25 us of a 400 us region, and the host clock is the more inclusive measure anyway)
        t0 = time.perf_counter()
        net.train_steps_from_host(packed, None, order, BATCH, 7, 1, hloss[W:W + K])
        barrier()
        e2e_wall = time.perf_counter() - t0
        e2e_events_ms = 0.0
        if os.environ.get("BRK_BENCH_E2E_DEBUG"):
            ws = []
            for _ in range(6):
                barrier(); _t = time.perf_counter()
                net.train_steps_from_host(packed, None, order, BATCH, 7, 1, hloss[W:W + K])
                barrier(); ws.append(round(1e6 * (time.perf_counter() - _t)))
            print(f"[e2e debug] timed shot {1e6 * e2e_wall:.0f} us; repeats {ws}", file=sys.stderr)
        e2e_launches, _k, _c = 0, 0, 2                     # one cooperative launch per chunk: 2, 4, 8, then 16 steps each
        while _k < K:
            e2e_launches += 1; _k += _c; _c = min(2 * _c, 16)
        if world == 1:
            # zero-copy variant: ids stay in pinned host memory, ONE launch, the kernel pulls them over PCIe itself
            for _ in range(2 if K <= 64 else 1):
                net.train_steps_mapped(hu, hp, order, BATCH, 7, 1, hwarm)
            barrier()
            _t = time.perf_counter()
            net.train_steps_mapped(hu, hp, order, BATCH, 7, 1, hloss[W:W + K])
            barrier()
            mapped_ms = 1e3 * (time.perf_counter() - _t)          # host clock, as for the copy leg
    else:
        for k in range(W):
            e2e_step(k)
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for k in range(K):
            e2e_step(W + k)
        e1.record()
        barrier()
        e2e_launches = 3 * K
        e2e_wall = time.perf_counter() - t0
        e2e_events_ms = e0.elapsed_time(e1)
    e2e_ms = max(e2e_events_ms, 1e3 * e2e_wall)
    clocks = sampler.stop()
    assert np.isfinite(hloss[W:W + K].numpy()).all()
    peaks, peak_src = load_peaks()
    # ---- (4) parity: the first 20 steps of the workload from the seeded initial weights, product vs CPU oracle -----------
    parity_losses = None
    if world == 1:
        pnet = BPRNet(U, I, DIM, seed=42, learning_rate=1e-3, sparse_adam="keras", device=dev)
        pnet.set_training_pairs(users, items)
        pnet.sample_negatives(7, 0)
        parity_losses = pnet.train_steps(list(range(PARITY_STEPS)), BATCH).cpu().numpy().astype(np.float64)
        del pnet
    # ---- (5) the other BASELINE.json configs ------------------------------------------------------------------------
    blocks = {}
    if not args.no_extras:
        if world == 1:
            blocks["neumf"] = neumf_block(dev, peaks, "class")
            blocks["neumf_he"] = neumf_block(dev, peaks, "he")
            blocks["extras"] = secondary_measurements(dev, peaks)
            blocks["extras"]["svd_fit"] = svd_measurement(dev)
        else:
            blocks["parity_multi"] = parity_multi_block(dev, world, rank)
            blocks["c4_neumf_sharded"] = c4_sharded_block(dev, world, rank, peaks)
            blocks["c5_topk_sharded"] = c5_topk_block(dev, world, rank, peaks)
    cpu = run_cpu_legs() if (world == 1 and rank == 0 and not args.no_cpu_baseline) else None

    # ---- max over ranks ---------------------------------------------------------------------------
    t = torch.tensor([total_ms, hot_ms, e2e_ms, float(fb_ms.mean())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, hot_ms, e2e_ms, fb_mean_ms = (float(x) for x in t.tolist())

    if rank == 0:
        value = world * K * BATCH / (total_ms * 1e-3)
        adam_bytes = 32 * (U + I) * DIM                     # w,m,v read+write, g read, g zeroed: 32 B per element
        launch_bytes = BYTES_PER_TRIPLET * BATCH + (adam_bytes // world if (world == 1 or net.peer is not None) else 0)
        achieved = launch_bytes / (fb_mean_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE.json configs[1]: BPR MF d=64, ML-1M shape (6040x3706, 1000209 positives), "
                                   "1 Philox negative/positive, loss 1-sigmoid, exact Keras Adam(1e-3)",
                       "batch": BATCH, "l2": "flushed between timed steps (256 MiB written, then read back so the lines "
                                             "are clean); step time = CUDA events around the step's kernels, flush excluded",
                       "parallelism": (f"mirrored data parallel x{world}: local batch {BATCH}; per step ONE cooperative kernel "
                                       f"per rank: fused fwd/bwd, cross-GPU barrier, reduce-scatter + Adam + all-gather over "
                                       f"NVLink peer memory (2.5 MB arenas, sharded Adam moments), barrier"
                                       if net.peer is not None else
                                       f"mirrored data parallel x{world}: local batch {BATCH}, one NCCL all-reduce of the "
                                       f"2.5 MB gradient arena per step") if world > 1 else "single GPU",
                       "wall_s_timed_region": wall},
            "value_hot_l2": world * K * BATCH / (hot_ms * 1e-3),
            "roofline": {"bound": "hbm",
                         "kernel": ("bpr_steps_coop<16,1> (whole step: fused gather+loss+scatter-add, grid.sync, Keras Adam)"
                                    if world == 1 else
                                    "bpr_steps_coop<16,1> (whole step incl. cross-GPU barriers and the peer-memory optimizer)"
                                    if net.peer is not None else "bpr_vec<16,1,true> (fused gather+loss+scatter-add)"),
                         "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"], "traffic": traffic_bytes(world), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": launch_bytes,
                         "avg_launch_ms": fb_mean_ms,
                         "note": "1536 B/triplet x 16384 (+ 32 B x 623744 table elements for the Adam phase at N=1); the "
                                 "10 MB of table state is cold in L2 at launch (flush) but rows are re-read ~4x from L2 "
                                 "within the launch and REDs resolve in L2: latency/L2-bound by construction at this "
                                 "table size -- see DESIGN.md section 4 for the same kernels on 20M-row tables"},
            "e2e": {"value": world * K * BATCH / (e2e_ms * 1e-3), "unit": UNIT, "path": "copy",
                    "h2d_bytes_per_step": 2 * BATCH * 4, "d2h_bytes_per_step": 4,
                    "gpu_launches": e2e_launches,
                    "note": ("BPRNet.train_steps_from_host: per step one cudaMemcpyAsync H2D of the step's user + positive "
                             "ids (128 KiB block of the pinned batch-major host array; copy stream, ring of staging "
                             "slots); steps run in cooperative launches of 2, 4, 8, then 16 steps (Philox negatives drawn "
                             "in-kernel, fused step, Adam); the step losses of a launch return in one cudaMemcpyAsync D2H; one host "
                             "sync per K steps" + ("" if world == 1 else "; every rank feeds its own batches, the launches are the "
                                                   "data-parallel cooperative kernel")) if (world == 1 or net.peer is not None) else
                            "per step: H2D ids, Philox negatives, fused fwd/bwd, NCCL all-reduce, Adam, loss D2H"},
            "gpu_launches": (1 if (world == 1 or net.peer is not None) else 2) * K,   # one cooperative step kernel per step
            "clocks": clocks,
        }
        if mapped_ms is not None:
            zc = {"value": K * BATCH / (mapped_ms * 1e-3), "unit": UNIT, "path": "zero_copy",
                  "h2d_bytes_per_step": 2 * BATCH * 4, "d2h_bytes_per_step": 4, "gpu_launches": 1,
                  "note": "BPRNet.train_steps_mapped: the host id arrays stay in pinned (mapped) host memory; ONE "
                          "cooperative launch runs all K steps; every step the kernel itself pulls that step's 128 KiB "
                          "of ids over PCIe (host->device) and stores the step's loss into pinned host memory "
                          "(device->host); no copy engine, no per-step driver call"}
            # both host-fed entry points are public API; the headline e2e is the faster one on this box (DMA latency of
            # the copy engines varies 3x between the pool's virtualised hosts), the other stays beside it
            if zc["value"] > line["e2e"]["value"]:
                line["e2e_copy"], line["e2e"] = line["e2e"], zc
            else:
                line["e2e_zero_copy"] = zc
        line.update(blocks)
        if cpu is not None:
            if "error" in cpu:
                line["cpu_baseline"] = {"error": cpu["error"]}
            else:
                line["cpu_baseline"] = cpu["bpr"]
                ref = np.asarray(cpu["bpr_parity_losses"], dtype=np.float64)
                line["parity_check"] = {
                    "what": f"per-step loss of the first {PARITY_STEPS} steps of this workload from the seeded initial weights "
                            f"(same frame, same Philox negatives): product (bpr_steps_coop on the GPU) vs the CPU oracle "
                            f"(subprocess)",
                    "max_abs_loss_diff": float(np.abs(parity_losses - ref).max()),
                    "max_rel_loss_diff": float((np.abs(parity_losses - ref) / np.abs(ref)).max()),
                    "loss_first": float(parity_losses[0]), "loss_last": float(parity_losses[-1]),
                    "tolerance": "fp32: 1e-5 relative per step (tests/test_gpu_fullsize.py holds the same run to it)"}
                for key, blk in (("neumf", line.get("neumf")), ("neumf_he", line.get("neumf_he"))):
                    if blk is not None and key + "_train" in cpu:
                        blk["cpu_baseline"] = cpu[key + "_train"]
                ex = line.get("extras") or {}
                for key in ("neumf_train_reference_batch", "twotower_train", "topk_ml1m", "svd_fit"):
                    if key in cpu:
                        ex.setdefault(key, {"config": "CPU leg only"})["cpu_baseline"] = cpu[key]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """Writes every tensor as out_dir/<name>.npy in float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def extras_cpu_baselines(budget_s=2.5):
    """The oracle (torch-CPU restatement of the reference, all host threads; NOT TensorFlow) timed on bounded samples
    of the other BASELINE.json configs: NeuMF (class graph and He et al. variant) at the bench batch and the class graph
    at the reference's own batch of 128 (NeuMFModel.py:102), the two-tower step at its batch of 1000 (twoTower.py:292),
    full-catalog top-K as the reference evaluates it (matmul + top_k in 5000-user batches, twoTower.py:293)."""
    from oracle import neumf as ON, twotower as OTT
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    rng = np.random.default_rng(0)
    U, I = 6040, 3706
    out = {}

    def timed(fn, units):
        fn()                                                            # warm-up
        t0 = time.perf_counter(); n = 0
        while time.perf_counter() - t0 < budget_s:
            fn(); n += 1
        dt = time.perf_counter() - t0
        return units * n / dt, n, dt

    for B, key, kw, what in ((BATCH, "neumf_train", {}, "NeuMF F=32 class graph"),
                             (BATCH, "neumf_he_train", dict(mf_dim=8, mf_mode="hadamard", batch_norm=False), "He et al. variant"),
                             (128, "neumf_train_reference_batch", {}, "NeuMF F=32 class graph")):
        orc = ON.NeuMFOracle(U, I, emb=32, dropout=0.0, **kw)            # no dropout: the oracle's NumPy Philox masks would dominate
        u = rng.integers(0, U, B); i = rng.integers(0, I, B); y = (rng.random(B) < 0.2).astype(np.float32)
        v, n, dt = timed(lambda: orc.step(u, i, y), B)
        out[key] = {"value": v, "unit": "interactions/s", "cores": threads, "kind": "port",
                    "sample": f"{n} steps of batch {B} in {dt:.1f} s, {what} oracle (autograd + exact Keras Adam, dropout off), fp32"}
    tt = OTT.TwoTowerOracle(U, I, 128, 128)
    u = rng.integers(2, U + 2, 1000); i = rng.integers(2, I + 2, 1000)
    v, n, dt = timed(lambda: tt.step(u, i, cand_ids=i), 1000)
    out["twotower_train"] = {"value": v, "unit": "interactions/s", "cores": threads, "kind": "port",
                             "sample": f"{n} steps of batch 1000 in {dt:.1f} s, two-tower E=S=128 oracle (in-batch softmax, Adagrad), fp32"}
    Q = torch.randn(U, 128); Cm = torch.randn(I, 128)

    def topk():
        for a in range(0, U, 5000):
            torch.topk(Q[a:a + 5000] @ Cm.T, 10)
    v, n, dt = timed(topk, U)
    out["topk_ml1m"] = {"value": v, "unit": "users/s", "cores": threads, "kind": "port",
                        "sample": f"{n} passes of 6040 users x 3706 items, d=128, k=10 in {dt:.1f} s (fp32 matmul + top_k, 5000-user batches)"}
    return out


def svd_cpu_baseline():
    """The sequential C loop of the oracle on the same rating file as svd_measurement (1 core: the algorithm is sequential)."""
    from binrec_b200 import synth
    from oracle import svd as OS
    u, i = synth.make_interactions()
    r = np.random.default_rng(5).integers(1, 6, len(u)).astype(np.float64)
    U, I, d = synth.ML1M_USERS, synth.ML1M_ITEMS, 50
    rng = np.random.default_rng(0)
    Pc, Qc = rng.normal(0, 0.1, (U, d)), rng.normal(0, 0.1, (I, d))
    buc, bic = np.zeros(U), np.zeros(I)
    mu = float(r.mean())
    OS.build_c()
    OS.fit_epoch_c(u[:1000], i[:1000], r[:1000], Pc, Qc, buc, bic, mu, 0.01, 0.0, 0.01)
    t0 = time.perf_counter()
    OS.fit_epoch_c(u, i, r, Pc, Qc, buc, bic, mu, 0.01, 0.0, 0.01)
    t = time.perf_counter() - t0
    return {"value": len(u) / t, "unit": "ratings/s", "cores": 1, "kind": "port",
            "sample": "one full epoch of the same file, sequential C loop (oracle/svd_c.c, gcc -O2)"}


def svd_measurement(dev):
    """Biased-SVD epoch (SURVEY.md section 8 row f4) on the ML-1M-shaped file, the reference's d = 50, float64, exact
    sequential semantics.  Bound: the longest dependency chain x one L2 hand-over (DESIGN.md section 4.5)."""
    from binrec_b200 import SVD as S
    from binrec_b200 import synth
    u, i = synth.make_interactions()
    r = np.random.default_rng(5).integers(1, 6, len(u)).astype(np.float64)
    U, I, d = synth.ML1M_USERS, synth.ML1M_ITEMS, S.NUMBER_OF_EMBEDDINGS
    frame = S.Ratings(u, i, r, num_users=U, num_items=I, device=dev)
    P, Q, bu, bi = S.init_parameters(U, I, d, seed=0, device=dev)
    mu = float(r.mean())
    for _ in range(2):
        S.fit_model(frame, P, Q, bu, bi, mu)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 5
    e0.record()
    for _ in range(iters):
        S.fit_model(frame, P, Q, bu, bi, mu)
    e1.record(); torch.cuda.synchronize()
    S.check_fit(frame)
    s = e0.elapsed_time(e1) * 1e-3 / iters
    chain = frame.critical_path()
    return {"value": len(u) / s, "unit": "ratings/s", "ms_per_epoch": s * 1e3, "critical_path": chain,
            "ns_per_chain_link": s * 1e9 / chain,
            "roofline": {"bound": "latency", "kernel": "svd_epoch_kernel", "achieved": s * 1e9 / chain, "unit": "ns per chain link",
                         "note": "neither HBM nor tensor: longest per-row dependency chain x one L2 hand-over (~1 us)"},
            "config": f"biased SVD (SVD.py:187-221), {len(u)} ratings in file order, {U} x {I}, d={d}, float64, "
                      f"sequential semantics kept exactly (ticketed rows, one cooperative launch per epoch)"}


def _timed(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / iters


def _hbm_roofline(kernel, bytes_per_launch, seconds, peaks, note):
    a = bytes_per_launch / seconds / 1e9
    return {"bound": "hbm", "kernel": kernel, "achieved": a, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": a / peaks["hbm_gbs"], "algorithmic_bytes_per_launch": int(bytes_per_launch), "avg_launch_ms": seconds * 1e3,
            "traffic": None, "note": note}


def _tensor_roofline(kernel, flops, seconds, peaks, note):
    a = flops / seconds / 1e12
    pk = peaks.get("bf16_tflops", 1590.0)
    return {"bound": "tensor", "kernel": kernel, "achieved": a, "peak": pk, "unit": "TFLOP/s", "frac": a / pk,
            "flops_per_launch": float(flops), "avg_launch_ms": seconds * 1e3, "traffic": None, "note": note}


def neumf_block(dev, peaks, which):
    """BASELINE.json configs[0]: NeuMF on the ML-1M-shaped frame (1 000 209 positives + 4 Philox negatives each, labels
    1 / 0, one seeded row shuffle: NeuMFModel.bootstrapDataset), batch 16 384, exact Keras Adam.  which = "class": the
    reference's graph (numFactor 32: MLP 64-32-16-8, BatchNorm after the activations, dropout 0.2, scalar Dot, MSE;
    NeuMFModel.py:53-100); "he": the He et al. variant the config line names (8-dim Hadamard GMF, no BatchNorm / dropout).
    One cooperative tcgen05 launch per step (csrc/neumf_fused.cu): gather, three Dense layers forward and backward on the
    tensor cores (TF32 operands), loss, row-gradient REDs, Adam over every parameter."""
    from binrec_b200 import synth
    from binrec_b200.NeuMFModel import NeuMFNet, NeuMFDataset
    U, I, B = synth.ML1M_USERS, synth.ML1M_ITEMS, BATCH
    users, items = synth.make_interactions()
    ds = NeuMFDataset(users, items, 4.0, B, True, dev, seed=7)
    nb = ds.n // B
    if which == "class":
        net = NeuMFNet(U, I, 32, dropout=0.2, device=dev, tensor_cores=True)
        emf, per_fwd = 32, 528                                   # SURVEY 8d: 4 rows x 128 B + ids/label 12 B + prediction 4 B
        kernel = "nfz::fused_step<Spec<32,32,32,16,8,relu,BN,dot>> (whole step incl. Adam)"
    else:
        net = NeuMFNet(U, I, 32, dropout=0.0, device=dev, mf_dim=8, mf_mode="hadamard", batch_norm=False)
        emf, per_fwd = 8, 336
        kernel = "nfz::fused_step<Spec<32,8,32,16,8,relu,noBN,hadamard>> (whole step incl. Adam)"
    o = torch.empty(B, device=dev); l = torch.empty(1, device=dev)
    K, W = 200, 5
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=dev)
    sink = torch.empty((), dtype=torch.float32, device=dev)

    def step(k):
        b = k % nb
        sl = slice(b * B, (b + 1) * B)
        net.train_on_batch(ds.u[sl], ds.i[sl], ds.y[sl], first_index=b * B, epoch=0, out=o, loss_out=l)

    for k in range(W):
        step(k)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    torch.cuda.synchronize()
    for k in range(K):                                          # L2 flushed between steps, events around the step's one kernel
        flush.zero_(); torch.sum(flush, dim=0, out=sink)
        evs[k][0].record(); step(W + k); evs[k][1].record()
    torch.cuda.synchronize()
    cold = float(np.mean([a.elapsed_time(b) for a, b in evs])) * 1e-3
    hot = _timed(lambda: step(0), 200)
    # end to end: the frame in pinned HOST memory, one H2D copy of 12 B x batch per step, losses back in one D2H copy
    nh = min(nb, 64)
    packed = NeuMFNet.pack_host_batches(ds.u[:nh * B].cpu().numpy(), ds.i[:nh * B].cpu().numpy(), ds.y[:nh * B].cpu().numpy(), B)
    order = np.arange(K) % nh
    for _ in range(2 if K <= 64 else 1):                        # warm-up: untimed passes over the same host batches (see the BPR e2e leg)
        net.train_steps_from_host(packed, order)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    hl = net.train_steps_from_host(packed, order)
    torch.cuda.synchronize()
    e2e = (time.perf_counter() - t0) / K                        # host clock around the call and the synchronize after it
    assert np.isfinite(hl.numpy()).all()
    n_tab = (U + I) * (32 + emf)
    n_dense = net.dense.w.numel()
    bytes_step = B * (per_fwd + 4 * 4 * (32 + emf) // 2 * 2) + 32 * (n_tab + n_dense)
    # row gradients: the same sum 4 d_t bytes as the gather (SURVEY 8d), REDs resolved in L2
    out = {"metric": "train interactions/sec (NeuMF, ML-1M shape, batch 16384)", "value": B / cold, "unit": "interactions/s",
           "ms_per_step": cold * 1e3, "value_hot_l2": B / hot, "steps": K, "gpu_launches": K,
           "e2e": {"value": B / e2e, "unit": "interactions/s", "h2d_bytes_per_step": 12 * B, "d2h_bytes_per_step": 4,
                   "note": "NeuMFNet.train_steps_from_host (brk_neumf_train_steps_host): pinned batch-major host frame, one "
                           "cudaMemcpyAsync per step on a copy stream (4 staging slots), the fused step, one D2H copy of the K losses"},
           "roofline": _hbm_roofline(kernel, bytes_step, cold, peaks,
                                     "per step: B x (gather + ids/label/prediction + row gradients) + 32 B x every parameter "
                                     "for the exact Keras Adam pass; the 2.5 MB of tables (10 MB with m, v, g) are L2-resident, "
                                     "the step is bound by its grid barriers and L2 round trips (profiles/r02_neumf_fused_trace.txt), "
                                     "not by HBM; tensor pipe < 1 % busy by construction (16 kFLOP per interaction)"),
           "config": {"workload": "BASELINE.json configs[0]: " + ("NeuMF class graph numFactor 32 (MLP 64-32-16-8, BN, dropout 0.2, "
                                                                   "scalar Dot, MSE)" if which == "class" else
                                                                   "He et al. NeuMF (MLP 64-32-16-8 on 32-dim tables + 8-dim Hadamard GMF, "
                                                                   "head 16->1, MSE)") +
                                  ", ML-1M shape, 4 negatives / positive, Keras Adam(1e-3)", "batch": B,
                      "l2": "flushed between timed steps (value); back to back (value_hot_l2)",
                      "dtype": "tf32 operands, fp32 accumulation / parameters"}}
    if which == "class":
        tp = os.path.join(ROOT, "profiles", "r02_neumf_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            out["roofline"]["traffic"] = tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"]
    del net, ds
    torch.cuda.empty_cache()
    return out


def secondary_measurements(dev, peaks):
    """Other BASELINE.json configs on one GPU, short runs (CUDA events, back-to-back steps), each with its roofline."""
    from binrec_b200 import hotpath as H
    from binrec_b200.NeuMFModel import NeuMFNet
    from binrec_b200.twoTower import TwoTowerModel
    out = {}
    g = torch.Generator(device=dev); g.manual_seed(0)
    U, I, B = 6040, 3706, BATCH
    # the reference's own batch size (bootstrapDataset default 128, NeuMFModel.py:102): fit's inner loop over a resident frame
    net = NeuMFNet(U, I, 32, dropout=0.2, device=dev, tensor_cores=True)
    Br, steps_r = 128, 400
    ur = torch.randint(0, U, (Br * steps_r,), generator=g, device=dev, dtype=torch.int32)
    ir = torch.randint(0, I, (Br * steps_r,), generator=g, device=dev, dtype=torch.int32)
    yr = (torch.rand(Br * steps_r, generator=g, device=dev) < 0.2).float()
    order_r = np.arange(steps_r)
    s = _timed(lambda: net.train_steps(ur, ir, yr, Br, order_r), 3, warm=1) / steps_r
    out["neumf_train_reference_batch"] = {"value": Br / s, "unit": "interactions/s", "ms_per_step": s * 1e3,
                                          "roofline": {"bound": "latency", "note": "one 128-sample tile: a single CTA's chain of "
                                                       "phases plus the dense Adam pass; launch- and latency-bound"},
                                          "config": "NeuMF F=32 class graph at the reference's batch of 128, one launch per step"}
    del net
    # fp32 CUDA-core path of the same step (neumf2.cu + Adam) for comparison
    net = NeuMFNet(U, I, 32, dropout=0.2, device=dev)
    u = torch.randint(0, U, (B,), generator=g, device=dev, dtype=torch.int32)
    i = torch.randint(0, I, (B,), generator=g, device=dev, dtype=torch.int32)
    y = (torch.rand(B, generator=g, device=dev) < 0.2).float()
    o = torch.empty(B, device=dev); l = torch.empty(1, device=dev)
    s = _timed(lambda: net.train_on_batch(u, i, y, out=o, loss_out=l), 50)
    out["neumf_train_fp32"] = {"value": B / s, "unit": "interactions/s", "ms_per_step": s * 1e3,
                               "config": "NeuMF F=32 class graph, batch 16384, fp32 on the CUDA cores (csrc/neumf2.cu, five kernels + Adam)"}
    del net
    # NeuMF at BASELINE.json configs[3] table sizes on ONE GPU (20 M x 2 M x 64, lazy Adam, batch 65 536): the five-kernel
    # tensor-core path (the batch does not fit on chip) -- the per-rank work of the row-sharded run
    try:
        from binrec_b200.sharded import ShardedNeuMFNet
        Uc, Ic, Bc = 20_000_000, 2_000_000, 65536
        netc = ShardedNeuMFNet(Uc, Ic, 64, dropout=0.2, device=dev, mode="peer", tensor_cores=True)
        us = torch.randint(0, Uc, (4, Bc), generator=g, device=dev, dtype=torch.int32)
        its = torch.randint(0, Ic, (4, Bc), generator=g, device=dev, dtype=torch.int32)
        yc = (torch.rand((4, Bc), generator=g, device=dev) < 0.2).float()
        oc = torch.empty(Bc, device=dev); lc = torch.empty(1, device=dev)
        kk = [0]

        def cstep():
            k = kk[0]; kk[0] += 1
            netc.train_on_batch(us[k % 4], its[k % 4], yc[k % 4], first_index=k * Bc, epoch=0, out=oc, loss_out=lc)

        s = _timed(cstep, 20)
        per = 1040 + 1024 + 1024 + 4 * 1792                       # fwd + re-gather + row gradients + lazy Adam on ~4 unique rows
        out["neumf_c4_one_gpu"] = {"value": Bc / s, "unit": "interactions/s", "ms_per_step": s * 1e3,
                                   "roofline": _hbm_roofline("ntc::tc_fwd1/fwd2/head/bwd2/bwd1 + adam_rows_kernel (whole step)", Bc * per, s, peaks,
                                                             "per interaction: 1040 B forward + 1024 B re-gather + 1024 B row gradients "
                                                             "+ 4 x 1792 B lazy Adam (SURVEY 8d); tables 33.8 GB, HBM-resident"),
                                   "config": "NeuMF E=64 (MLP 128-64-32-16), 20M x 2M tables on ONE GPU, batch 65536, lazy Adam, TF32 tensor cores"}
        del netc, us, its, yc
        torch.cuda.empty_cache()
    except Exception as e:  # pragma: no cover - memory pressure on a shared box
        out["neumf_c4_one_gpu"] = {"error": repr(e)[:200]}
    users = list(range(U)); items = list(range(I))
    for Bt2, tag in ((1000, "twotower_train"), (8192, "twotower_train_b8192")):
        tt2 = TwoTowerModel(128, I, U, "u", "i", users, items, semb=128, device=dev, tensor_cores=True)
        tt2.compile("Adagrad", learningRate=0.1)
        uid2 = torch.randint(2, U + 2, (Bt2,), generator=g, device=dev, dtype=torch.int32)
        iid2 = torch.randint(2, I + 2, (Bt2,), generator=g, device=dev, dtype=torch.int32)

        def tt2_step():
            tt2._train_ids(uid2, iid2, None)               # step + Adagrad: brk_twotower_train_step

        tt2_step()
        # the step as TwoTowerModel.fit runs it: one CUDA-graph replay per batch
        side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            tt2_step()
        torch.cuda.current_stream().wait_stream(side)
        gph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gph):
            tt2_step()
        s = _timed(gph.replay, 30)
        flops = 2.0 * Bt2 * 128 * 128 * 2 * 3 + 2.0 * Bt2 * Bt2 * 128 * 3   # two tower Dense layers and the B x B scores, fwd + 2 bwd products each
        out[tag] = {"value": Bt2 / s, "unit": "interactions/s", "ms_per_step": s * 1e3,
                    "roofline": _tensor_roofline("ttf::fused_step (one cooperative launch: towers, on-chip score tiles, gradients, Adagrad)"
                                                 if Bt2 <= 1536 else "gemm_tf32_kernel x 9 + inbatch_softmax_kernel + adagrad (graph of one step)",
                                                 flops, s, peaks,
                                                 "TF32 products against the bf16 peak (TF32 dense peak is half of it); at batch 1000 the "
                                                 "step is latency: five phases of ~5 us separated by four grid barriers of ~1.4 us "
                                                 "(profiles/r02_twotower_fused_trace.txt); at 8192 the batch does not fit on chip and the "
                                                 "multi-kernel step is bound by the B x B score matrix"),
                    "config": f"two-tower E=S=128 (twoTower.py:40-41 shape), in-batch softmax batch {Bt2}, Adagrad 0.1, all products on tcgen05 "
                              f"(TF32), replayed as one CUDA graph per step (what TwoTowerModel.fit does)"}
        del tt2, gph
    Q = torch.randn(U, 128, generator=g, device=dev); Cm = torch.randn(I, 128, generator=g, device=dev)
    idx = H.BruteForceIndex(10).index(Cm)
    s = _timed(lambda: idx(Q), 50)
    out["topk_ml1m"] = {"value": U / s, "unit": "users/s", "ms": s * 1e3,
                        "roofline": _tensor_roofline("score_topk_kernel", 2.0 * U * I * 128, s, peaks,
                                                     "48 user tiles x 7 item splits on 296 CTA slots: launch / latency bound at this size"),
                        "config": "6040 users x 3706 items, d=128, k=10, bf16 tcgen05 scoring + fused top-K (incl. query bf16 conversion)"}
    Ub, Ib = 65536, 250000
    for d in (64, 128):
        Q = torch.randn(Ub, d, generator=g, device=dev); Cm = torch.randn(Ib, d, generator=g, device=dev)
        idx = H.BruteForceIndex(10).index(Cm)
        s = _timed(lambda: idx(Q), 5, warm=1)
        out[f"topk_shard_d{d}"] = {"value": Ub / s, "unit": "users/s", "ms": s * 1e3,
                                   "roofline": _tensor_roofline("score_topk_kernel", 2.0 * Ub * Ib * d, s, peaks,
                                                                "two CTAs per SM, branch-free chunk flags; with warm thresholds the epilogue runs at the TMEM drain rate "
                                                                "(31 scores/clk/SM), what is left on random data is the second look at flagged chunks while the "
                                                                "k-th-best thresholds warm up on a short shard (DESIGN.md section 4.1, profiles/r02_topk_probe.txt)"),
                                   "config": f"65536 users x 250000 items (one 8-way item shard of BASELINE.json configs[4]), d={d}, k=10"}
        del Q, Cm, idx
    return out


# ------------------------------------------------------------------------------------------------
# N > 1: the partitioning BASELINE.json north_star asks for, and parity inside the same run
# ------------------------------------------------------------------------------------------------
def c4_sharded_block(dev, world, rank, peaks):
    """BASELINE.json configs[3]: NeuMF E=64 with 20 M x 2 M x 64 tables ROW-SHARDED over the ranks (row r on rank r % G);
    local batch 65 536 per GPU (weak scaling).  The fused kernels gather peer rows with plain loads and send row
    gradients as 16-byte REDs into the owner's accumulator over NVLink: the all-to-all of rows and of row gradients
    happens inside the gather / scatter instructions; then a peer barrier, lazy Adam on the owned shards and the fused
    reduce-scatter + Adam + all-gather of the mirrored dense block (csrc/dp_peer.cu)."""
    import torch.distributed as dist
    from binrec_b200.sharded import ShardedNeuMFNet
    U, I, E, B, K = 20_000_000, 2_000_000, 64, 65536, 20
    net = ShardedNeuMFNet(U, I, E, dropout=0.2, device=dev, mode="peer", tensor_cores=True)
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    nb = 8
    us = torch.randint(0, U, (nb, B), generator=g, device=dev, dtype=torch.int32)
    its = torch.randint(0, I, (nb, B), generator=g, device=dev, dtype=torch.int32)
    y = (torch.rand((nb, B), generator=g, device=dev) < 0.2).float()
    o = torch.empty(B, device=dev); l = torch.empty(1, device=dev)

    def step(k):
        net.train_on_batch(us[k % nb], its[k % nb], y[k % nb], first_index=k * B * world, epoch=0, out=o, loss_out=l)

    for k in range(3):
        step(k)
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        step(3 + k)
    e1.record(); torch.cuda.synchronize()
    net.check()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    s = float(t.item()) * 1e-3 / K
    loss = float(l.item())
    del net, us, its, y
    torch.cuda.empty_cache()
    per_hbm = 1040 + 1024 + 1024 + 4 * 1792                        # as on one GPU (SURVEY 8d)
    per_link = (world - 1) / world * (4 * 4 * E + 16) * 3          # rows out (fwd + re-gather) and row gradients back
    t_hbm = B * per_hbm / (peaks["hbm_gbs"] * 1e9)
    t_link = B * per_link / 770e9
    return {"metric": "train interactions/sec (NeuMF E=64, 20M x 2M tables row-sharded)", "value": world * B / s,
            "unit": "interactions/s", "n_gpus": world, "ms_per_step": s * 1e3, "steps": K, "scaling": "weak", "loss": loss,
            "roofline": {"bound": "hbm+nvlink", "kernel": "ntc::tc_* on peer-mapped shards + adam_rows_kernel + dp_adam_peer_kernel (whole step, per rank)",
                         "achieved": B * per_hbm / s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": B * per_hbm / s / 1e9 / peaks["hbm_gbs"],
                         "nvlink_bytes_per_step_per_gpu": int(B * per_link), "nvlink_achieved_gbs": B * per_link / s / 1e9,
                         "nvlink_peak_gbs": 770.0, "nvlink_frac": B * per_link / s / 1e9 / 770.0,
                         "target_ms": max(t_hbm, t_link) * 1e3, "frac_of_target": max(t_hbm, t_link) / s, "traffic": None,
                         "note": "per interaction: HBM 1040 + 1024 + 1024 + 4 x 1792 B at the owners; NVLink (G-1)/G x (sum 4 d_t + 16) B "
                                 "each for the forward rows, the backward re-gather and the row gradients (SURVEY 8d); target = the "
                                 "slower of HBM bytes / measured copy peak and NVLink bytes / 770 GB/s"},
            "config": {"workload": "BASELINE.json configs[3]: NeuMF E=64 (MLP 128-64-32-16, BN, dropout 0.2), 20M users x 2M items, "
                                   "uniform ids, lazy Adam", "local_batch": B,
                       "parallelism": f"tables row-sharded x{world} (owner = id mod G) in NVLink peer-mapped memory; dense block mirrored"}}


def c5_topk_block(dev, world, rank, peaks):
    """BASELINE.json configs[4]: 1 M users x 2 M items, d = 64, k = 10; items RANGE-SHARDED over the ranks, every rank
    scores all users against its range (tcgen05 scoring + fused top-K, scores never reach HBM), the per-shard [U, k]
    lists are all-gathered and merged (score desc, id asc: identical to an unsharded scan).  Strong scaling."""
    import torch.distributed as dist
    from binrec_b200 import hotpath as H, distributed as D
    U, I, d, k, chunk = 1_000_000, 2_000_000, 64, 10, 131072
    g = torch.Generator(device=dev); g.manual_seed(5)                # same queries on every rank
    Q = torch.randn(U, d, generator=g, device=dev)
    lo, hi = D.local_slice(I)
    gi = torch.Generator(device=dev); gi.manual_seed(100 + rank)
    C = torch.randn(hi - lo, d, generator=gi, device=dev)
    idx = H.BruteForceIndex(k).index(C, id_offset=lo)

    def sweep():
        outs = []
        for s0 in range(0, U, chunk):
            v, i = idx(Q[s0:s0 + chunk])
            pv, pi = D.gather_topk_parts(v, i)
            outs.append(H.topk_merge(pv, pi))
        return outs

    sweep(); torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); sweep(); e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    s = float(t.item()) * 1e-3
    del Q, C, idx
    torch.cuda.empty_cache()
    flops_gpu = 2.0 * U * (hi - lo) * d
    return {"metric": "top-K users/sec (1M users x 2M items, d=64, k=10)", "value": U / s, "unit": "users/s", "n_gpus": world,
            "ms": s * 1e3, "scaling": "strong",
            "roofline": _tensor_roofline("score_topk_kernel (per rank; + all-gather of [U,k] lists + topk_merge_kernel)", flops_gpu, s, peaks,
                                         "per GPU, all-gather of the lists and merge included; the selection epilogue is the limiter (DESIGN.md section 4.1)"),
            "config": {"workload": "BASELINE.json configs[4]: full-catalog top-K sweep, bf16 operands, fp32 scores",
                       "parallelism": f"items range-sharded x{world}, NCCL all-gather of the [U, k] (score, id) lists, merge on every rank"}}


def parity_multi_block(dev, world, rank):
    """Parity of the multi-GPU paths INSIDE the bench run (the driver's GPU test lease has one GPU): every rank also runs the
    single-process model on the global batches and compares.  (a) mirrored data-parallel BPR (the headline's kernel):
    3 steps, global batch = world x 2048; (b) row-sharded NeuMF (tensor-core path, He-free class graph E=32 without
    dropout; BatchNorm statistics are per replica, so the comparison is on the forward loss of one step and on the dense
    gradient norm) -- losses against the unsharded NeuMFNet on this rank's batch."""
    import torch.distributed as dist
    from binrec_b200 import distributed as D
    from binrec_b200.BPRModel import BPRNet
    from binrec_b200.NeuMFModel import NeuMFNet
    from binrec_b200.sharded import ShardedNeuMFNet
    out = {}
    U, I, d, B = 6040, 3706, 64, 2048
    rng = np.random.default_rng(3)
    dp = BPRNet(U, I, d, seed=42, device=dev)                   # peer arenas (world > 1)
    os.environ["BRK_DP"] = "nccl"
    single = None
    try:
        # a single-process replica on this rank: no peer arena, no all-reduce -- built with torch.distributed hidden
        import binrec_b200.distributed as Dm
        real_ws, real_rk = Dm.world_size, Dm.rank
        Dm.world_size, Dm.rank = (lambda: 1), (lambda: 0)
        single = BPRNet(U, I, d, seed=42, device=dev)
        for step in range(3):
            u = rng.integers(0, U, world * B).astype(np.int32); p = rng.integers(0, I, world * B).astype(np.int32)
            n = rng.integers(0, I, world * B).astype(np.int32)
            single.train_on_batch(*(torch.from_numpy(x).to(dev) for x in (u, p, n)))
            Dm.world_size, Dm.rank = real_ws, real_rk
            lo, hi = D.local_slice(world * B)
            dp.train_on_batch(*(torch.from_numpy(x[lo:hi]).to(dev) for x in (u, p, n)))
            Dm.world_size, Dm.rank = (lambda: 1), (lambda: 0)
    finally:
        Dm.world_size, Dm.rank = real_ws, real_rk
        os.environ.pop("BRK_DP", None)
    torch.cuda.synchronize()
    if dp.peer is not None:
        dp.peer.check()
    err = torch.stack([(dp.user.w - single.user.w).abs().max(), (dp.item.w - single.item.w).abs().max()]).max().view(1).double()
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    out["mirrored_bpr"] = {"max_abs_weight_diff_vs_single_gpu": float(err.item()), "steps": 3, "global_batch": world * B,
                           "tolerance": 2e-6, "ok": bool(err.item() <= 2e-6)}
    del dp, single
    # (b) row-sharded NeuMF against the unsharded model on the same batch (forward loss, one step, no dropout)
    Un, In, E, Bn = 3000, 2000, 32, 4096
    sh = ShardedNeuMFNet(Un, In, E, dropout=0.0, device=dev, mode="peer", tensor_cores=True, seed=42)
    full = {name: torch.from_numpy(t.full_weights()).to(dev) for name, t in zip(("uMLP", "iMLP", "uMF", "iMF"), sh._tables())}
    rng2 = np.random.default_rng(100 + rank)
    u = torch.from_numpy(rng2.integers(0, Un, Bn).astype(np.int32)).to(dev)
    i = torch.from_numpy(rng2.integers(0, In, Bn).astype(np.int32)).to(dev)
    y = torch.from_numpy((rng2.random(Bn) < 0.3).astype(np.float32)).to(dev)
    if full is not None:
        Dm.world_size, Dm.rank = (lambda: 1), (lambda: 0)
        try:
            ref = NeuMFNet(Un, In, E, dropout=0.0, device=dev, tensor_cores=True, seed=42)
        finally:
            Dm.world_size, Dm.rank = real_ws, real_rk
        for name in ("uMLP", "iMLP", "uMF", "iMF"):
            getattr(ref, name).w.copy_(full[name])
        ref.dense.w.copy_(sh.dense.w)
        lr, _ = ref.forward_backward(u, i, y, global_batch=world * Bn)
        ls, _ = sh.train_on_batch(u, i, y)
        sh.check()
        dl = (ls - lr).abs().view(1).double() / lr.abs().double()
        dist.all_reduce(dl, op=dist.ReduceOp.MAX)
        out["sharded_neumf"] = {"max_rel_loss_diff_vs_unsharded": float(dl.item()), "tolerance": 1e-5, "ok": bool(dl.item() <= 1e-5),
                                "batch_per_rank": Bn}
    else:
        out["sharded_neumf"] = {"skipped": "ShardedTable.gather_full unavailable"}
    del sh
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="brk", choices=["brk", "reference", "cpu_legs"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "brk":
        ap.error("--dump-outputs applies to --impl brk")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        reference_arm(args)
    elif args.impl == "cpu_legs":
        cpu_legs_main(args)
    else:
        product_arm(args)


if __name__ == "__main__":
    main()
