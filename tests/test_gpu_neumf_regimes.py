"""The NeuMF tensor-core step in every regime its batch size selects, against the TF32-operand oracle.

With n = ceil(B / 128) tiles and S SMs the launchers pick (csrc/neumf_fused.cu nfz::run, csrc/neumf_tc.cu ntc::run,
csrc/neumf_loop.cu brk_neumf_train_step):
  class spec F = 32 / 64, He variant, n <= S     one cooperative launch, grid S: helper CTAs, one CTA per SM, Adam inside
  class spec, n > S                               the five-kernel path; past occ * S tiles its persistent kernels loop
  He variant, n > S                               independent tiles (atomics + last-CTA ticket), Adam as its own launch
  inference, any n                                independent tiles
A cooperative grid is bounded by the occupancy the launcher queries.  On a B200 that is one CTA per SM for all three
instances, although F = 32 and the He variant take ~108 KB of shared memory and at most 128 registers a thread, so no
cooperative launch covers more than S tiles.
Each case proves which regime ran from BRK_NEUMF_TRACE (block 0 stamps word 0 at entry and word 10 inside the cooperative
dense reduction; block b < 480 writes its SM id to word 32 + b), then holds the step to oracle/neumf.py at the tolerances
of tests/test_gpu_tc.py.  The tables are small (300 x 200) and the ids skewed, so every row collects hundreds of samples
and one sample's ReLU gate flip stays inside the per-row budget of _check_step_against_oracle."""
import numpy as np
import pytest
import torch

from test_gpu_tc import _check_step_against_oracle, _tf32_matmul

pytestmark = pytest.mark.gpu

U, I, TS = 300, 200, 128
SPECS = {"F32": dict(E=32, dropout=0.2, kw=dict(tensor_cores=True)),
         "F64": dict(E=64, dropout=0.0, kw=dict(tensor_cores=True)),
         "He": dict(E=32, dropout=0.0, kw=dict(mf_dim=8, mf_mode="hadamard", batch_norm=False))}

# (spec, tiles = a * S + b, samples in the last tile, regime, sparse_adam)
#   spread: cooperative, grid max(n, S), every CTA on an SM of its own
#   five:   fused_step never ran
#   tiles:  fused_step ran as independent tiles (no cooperative reduction)
CASES = [("F32", (1, -1), 77, "spread", "keras"), ("F32", (1, 0), 128, "spread", "keras"),
         ("F32", (1, 1), 1, "five", "keras"), ("F32", (2, 0), 127, "five", "keras"),
         ("F32", (2, 1), 50, "five", "keras"), ("F32", (4, 1), 77, "five", "keras"),
         ("F64", (1, 0), 100, "spread", "keras"), ("F64", (1, 1), 77, "five", "keras"),
         ("F64", (4, 1), 77, "five", "keras"), ("F64", (4, 1), 77, "five", "lazy"),
         ("He", (1, -1), 77, "spread", "keras"), ("He", (1, 1), 77, "tiles", "keras"), ("He", (2, 0), 77, "tiles", "keras"),
         ("He", (2, 1), 77, "tiles", "keras"), ("He", (4, 1), 77, "tiles", "keras")]


def _case_id(c):
    a, b = c[1]
    return f"{c[0]}-{a}S{b:+d}-last{c[2]}-{c[3]}-{c[4]}".replace("+0", "")


def _sm_count(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


def _batch(B, seed):
    rng = np.random.default_rng(seed)
    u = (U * rng.random(B) ** 2).astype(np.int32); i = (I * rng.random(B) ** 2).astype(np.int32)
    y = (rng.random(B) < 0.25).astype(np.float32)
    return u, i, y


def _net(dev, spec, sparse_adam="keras"):
    from binrec_b200.NeuMFModel import NeuMFNet
    s = SPECS[spec]
    return NeuMFNet(U, I, s["E"], dropout=s["dropout"], seed=42, dropout_seed=11, device=dev, sparse_adam=sparse_adam, **s["kw"])


def _oracle(spec, lazy=False, dtype=torch.float32):
    from oracle import neumf as ON
    s = SPECS[spec]
    kw = {k: v for k, v in s["kw"].items() if k != "tensor_cores"}
    mm = _tf32_matmul() if dtype == torch.float32 else torch.matmul
    return ON.NeuMFOracle(U, I, emb=s["E"], seed=42, dropout=s["dropout"], dropout_seed=11, lazy_adam=lazy, dtype=dtype,
                          matmul=mm, **kw)


class _Trace:
    """BRK_NEUMF_TRACE around one call: words 0..31 zeroed, 32..511 set to -1."""

    def __init__(self, dev, monkeypatch):
        self.buf = torch.full((512,), -1, dtype=torch.int64, device=dev)
        self.buf[:32] = 0
        self.mp = monkeypatch

    def __enter__(self):
        torch.cuda.synchronize()
        self.mp.delenv("BRK_NEUMF_NO_FUSED", raising=False)
        self.mp.setenv("BRK_NEUMF_TRACE", hex(self.buf.data_ptr()))
        return self

    def __exit__(self, *exc):
        torch.cuda.synchronize()
        self.mp.delenv("BRK_NEUMF_TRACE")
        w = self.buf.cpu().numpy()
        sms = w[32:][w[32:] >= 0]
        self.fused, self.coop = bool(w[0] != 0), bool(w[10] != 0)
        self.grid = int(sms.size)                                   # CTAs that ran fused_step (counted up to 480)
        self.n_sms = int(np.unique(sms).size)
        self.max_per_sm = int(np.bincount(sms).max()) if sms.size else 0   # CTAs the busiest SM ran, over the launch
        return False

    def __repr__(self):
        return f"fused={self.fused} coop={self.coop} grid={self.grid} sms={self.n_sms} max_per_sm={self.max_per_sm}"


def _assert_regime(tr, regime, n, S, tag):
    print(f"{tag}: {tr}")
    if regime == "spread":
        assert tr.fused and tr.coop and tr.grid == max(n, S) == S, (tag, tr)
        assert tr.n_sms == S and tr.max_per_sm == 1, (tag, tr)      # the 120 KB request keeps one CTA per SM
    elif regime == "five":
        assert not tr.fused and tr.grid == 0, (tag, tr)
    else:                                                           # independent tiles
        assert tr.fused and not tr.coop and tr.grid == min(n, 480), (tag, tr)


@pytest.mark.parametrize("case", CASES, ids=[_case_id(c) for c in CASES])
def test_neumf_step_regime_matches_tf32_oracle(dev, monkeypatch, case):
    spec, (a, b), last, regime, sparse_adam = case
    S = _sm_count(dev)
    n = a * S + b
    B = TS * (n - 1) + last
    tag = f"{_case_id(case)} S={S} tiles={n} B={B}"
    if a == 4:
        # five-kernel path: past 4 S tiles every persistent grid (tc_head <= 4 S CTAs, tc_bwd2 / tc_bwd1 <= 2 S) has a CTA
        # that takes two tiles or more, and tc_bwd1 prefetches a ragged last tile
        assert n > 4 * S and last < TS
    lazy = sparse_adam == "lazy"

    # ---- forward + backward on a fresh net: predictions, loss, every gradient
    if not lazy:
        net, orc = _net(dev, spec), _oracle(spec)
        u, i, y = _batch(B, seed=n)
        with _Trace(dev, monkeypatch) as tr:
            _check_step_against_oracle(dev, net, orc, u, i, y, 4096, 3, f"{tag} forward_backward")
        _assert_regime(tr, regime, n, S, f"{tag} forward_backward")
        assert not net._bufs["acc"].any().item()                    # accumulators left zero for the next step

    # ---- three Adam steps on a fresh net against the TF32 and the fp64 oracle
    net = _net(dev, spec, sparse_adam)
    orc, o64 = _oracle(spec, lazy), _oracle(spec, lazy, torch.float64)
    rng_seed = 1000 + n
    for step in range(3):
        u, i, y = _batch(B, seed=rng_seed + step)
        lref, _ = orc.step(u, i, y, first_index=step * B, epoch=1)
        l64, _ = o64.step(u, i, y, first_index=step * B, epoch=1)
        args = [torch.from_numpy(x).to(dev) for x in (u, i, y)]
        if step == 0:
            with _Trace(dev, monkeypatch) as tr:
                lgot, _ = net.train_on_batch(*args, first_index=0, epoch=1)
            # a cooperative training launch is one only when Adam runs inside it (otherwise brk_neumf_train_step takes
            # an independent-tile launch or the five-kernel path, then the optimizer kernels)
            _assert_regime(tr, regime, n, S, f"{tag} train_on_batch")
        else:
            lgot, _ = net.train_on_batch(*args, first_index=step * B, epoch=1)
        print(f"{tag} step {step}: loss device {lgot.item():.7f} tf32 oracle {lref:.7f} fp64 {l64:.7f}")
        np.testing.assert_allclose(lgot.item(), lref, rtol=2e-3)
        np.testing.assert_allclose(lgot.item(), l64, rtol=2e-3)
    ref, ref64 = orc.p.numpy(), o64.p.numpy()
    for name, tab in zip(("uMLP", "iMLP", "uMF", "iMF"), net.tables()):
        w = tab.w.cpu().numpy()
        err_dev, err_orc = np.abs(w - ref64[name]).max(), np.abs(ref[name] - ref64[name]).max()
        print(f"{tag} {name} max |w - fp64|: device {err_dev:.2e} tf32 oracle {err_orc:.2e}")
        assert err_dev <= 3 * err_orc + 1e-4, (tag, name, err_dev, err_orc)
        if tab.touched is not None:
            assert not tab.touched.any().item(), (tag, name)
    if SPECS[spec]["kw"].get("batch_norm", True):
        np.testing.assert_allclose(net.bn_moving.cpu().numpy(),
                                   np.concatenate([orc.p.mm1.numpy(), orc.p.mv1.numpy(), orc.p.mm2.numpy(), orc.p.mv2.numpy()]),
                                   rtol=2e-3, atol=1e-5)
    assert int(net.optimizer.state[0].item()) == 3
    assert not net.grad_arena.any().item()                          # every gradient consumed by the optimizer


@pytest.mark.parametrize("spec", sorted(SPECS))
def test_neumf_inference_past_four_waves_matches_oracle(dev, monkeypatch, spec):
    """Inference runs as independent tiles at any batch: 4 S + 1 tiles with a ragged last tile, after two training steps
    so that the BatchNorm moving statistics are not their initial values."""
    S = _sm_count(dev)
    n = 4 * S + 1
    B = TS * (n - 1) + 77
    net, orc = _net(dev, spec), _oracle(spec)
    for step in range(2):
        u, i, y = _batch(2048, seed=70 + step)
        lref, _ = orc.step(u, i, y, first_index=step * 2048, epoch=0)
        lgot, _ = net.train_on_batch(*(torch.from_numpy(x).to(dev) for x in (u, i, y)), first_index=step * 2048, epoch=0)
        np.testing.assert_allclose(lgot.item(), lref, rtol=2e-3)
    u, i, _ = _batch(B, seed=n)
    with _Trace(dev, monkeypatch) as tr:
        p, _ = net.predict_on_batch(torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev))
    _assert_regime(tr, "tiles", n, S, f"{spec} inference tiles={n} B={B}")
    got, want = p.cpu().numpy(), orc.predict(u, i)
    print(f"{spec} inference B={B}: max |err| {np.abs(got - want).max():.2e}")
    np.testing.assert_allclose(got, want, rtol=5e-3, atol=1e-4)
