"""Biased-SVD epoch kernel (csrc/svd.cu): epoch time against residency (warps per SM), on the ML-1M-shaped file
(power-law head) and on a uniform file of the same size; prints the critical path so that the time per chain link can
be read off.   python profiles/svd_case.py [once]      (once: a single epoch, for ncu)"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from binrec_b200 import SVD as S          # noqa: E402
from binrec_b200 import synth             # noqa: E402


def epoch_ms(frame, P, Q, bu, bi, mu, warps, iters=3):
    S.fit_model(frame, P, Q, bu, bi, mu, warps_per_sm=warps)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        S.fit_model(frame, P, Q, bu, bi, mu, warps_per_sm=warps)
    e1.record(); torch.cuda.synchronize()
    S.check_fit(frame)
    return e0.elapsed_time(e1) / iters


def main():
    once = len(sys.argv) > 1 and sys.argv[1] == "once"
    U, I, d = synth.ML1M_USERS, synth.ML1M_ITEMS, 50
    for skew in (True,) if once else (True, False):
        u, i = synth.make_interactions(skew=skew)
        r = np.random.default_rng(5).integers(1, 6, len(u)).astype(np.float64)
        t0 = time.perf_counter()
        frame = S.Ratings(u, i, r, num_users=U, num_items=I)
        torch.cuda.synchronize()
        t_sched = time.perf_counter() - t0
        P, Q, bu, bi = S.init_parameters(U, I, d, seed=0)
        mu = float(r.mean())
        if once:
            S.fit_model(frame, P, Q, bu, bi, mu); torch.cuda.synchronize(); S.check_fit(frame)
            return
        chain = frame.critical_path()
        print(f"skew={skew}: n={len(u)} critical path {chain} (max item count {np.bincount(i).max()}, max user count "
              f"{np.bincount(u).max()}), schedule build {t_sched * 1e3:.1f} ms (incl. H2D)", flush=True)
        for warps in (0, 24, 16, 8):
            ms = epoch_ms(frame, P, Q, bu, bi, mu, warps)
            print(f"  warps_per_sm={warps:2d}: {ms:8.3f} ms/epoch  {len(u) / ms / 1e3:8.2f} M ratings/s  "
                  f"{ms * 1e6 / chain:7.1f} ns per chain link", flush=True)


if __name__ == "__main__":
    main()
