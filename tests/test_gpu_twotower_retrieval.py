"""The two-tower step with tfrs Retrieval's options -- temperature, candidate sampling probabilities, sample weights, and the
on-device streaming frequency estimator (brk_twotower_step_retrieval / brk_twotower_train_step_retrieval) -- on both
paths: the one cooperative launch (csrc/twotower_fused.cu, fused_step<false, true>) and the multi-kernel step
(csrc/twotower.cu, tt_logq_kernel + inbatch_softmax_kernel<true>), against oracle/twotower_retrieval.py."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U, I = 400, 150


def _tf32():
    from oracle import tf32
    return tf32.matmul                                                 # truncated TF32 operands (test_gpu_tc.TF32_MODE)


def _model(dev, E, S, tc, **kw):
    from binrec_b200.twoTower import TwoTowerModel
    return TwoTowerModel(E, I, U, "u", "i", list(range(U)), list(range(I)), semb=S, device=dev, tensor_cores=tc, **kw)


def _oracle(m, E, S, tc, tau):
    from oracle import twotower_retrieval as OR
    o = OR.RetrievalOracle(U, I, E, S, seed=42, temperature=tau, matmul=_tf32() if tc else torch.matmul)
    with torch.no_grad():
        o.t["Eu"].copy_(m.userTower.emb.w.cpu()); o.t["Ei"].copy_(m.itemTower.emb.w.cpu())
        for tw, wn, bn in ((m.userTower, "Wu", "bu"), (m.itemTower, "Wi", "bi")):
            flat = tw.dense.w.view(-1).cpu()
            o.t[wn].copy_(flat[:E * S].view(E, S)); o.t[bn].copy_(flat[E * S:E * S + S])
    return o


def _inputs(dev, B, seed=3):
    g = torch.Generator(device=dev); g.manual_seed(seed)
    uid = torch.randint(2, U + 2, (B,), generator=g, device=dev, dtype=torch.int32)
    iid = torch.randint(2, I + 2, (B,), generator=g, device=dev, dtype=torch.int32)          # repeated items: accidental hits
    rng = np.random.default_rng(seed)
    p = (rng.random(B) ** 4).astype(np.float32)                       # skewed; some below the 1e-6 clip
    p[rng.integers(0, B, 5)] = 1e-9
    w = rng.uniform(0.0, 2.0, B).astype(np.float32)
    w[rng.integers(0, B, 3)] = 0.0
    return uid, iid, torch.from_numpy(p).to(dev), torch.from_numpy(w).to(dev)


def _grads(m, E, S):
    return [m.userTower.emb.g, m.itemTower.emb.g, m.userTower.dense.g.view(-1)[:E * S].view(E, S),
            m.itemTower.dense.g.view(-1)[:E * S].view(E, S), m.userTower.dense.g.view(-1)[E * S:E * S + S]]


def _zero(m):
    for t in (m.userTower.emb, m.itemTower.emb, m.userTower.dense, m.itemTower.dense):
        t.g.zero_()
    for t in (m.userTower.emb, m.itemTower.emb):
        t.touched.zero_()


def _close_to_oracle(m, o, E, S, lgot, lref):
    np.testing.assert_allclose(lgot, float(lref), rtol=2e-3)
    for got, name in zip(_grads(m, E, S), ("Eu", "Ei", "Wu", "Wi", "bu")):
        g0, g1 = o.t[name].grad.numpy(), got.cpu().numpy()
        scale = max(float(np.abs(g0).max()), 1e-20)
        mx = float(np.abs(g1 - g0).max()) / scale
        fro = float(np.linalg.norm(g1 - g0) / max(np.linalg.norm(g0), 1e-20))
        assert mx <= 1e-2 and fro <= 1e-2, (name, mx, fro)


@pytest.mark.parametrize("B,tc,no_fused,tau", [(129, True, False, 0.2), (333, True, False, 3.0), (1000, True, False, 0.5),
                                               (1536, True, False, 1.0), (2048, True, False, 0.5), (1000, True, True, 0.2),
                                               (333, False, False, 0.2)])
def test_options_match_the_oracle(dev, monkeypatch, B, tc, no_fused, tau):
    """Against the TF32 oracle (fp32 oracle for tc=False) with the tolerances of
    test_gpu_tc.py::test_twotower_tensor_core_step_matches_tf32_oracle: one launch at B <= 1536, the multi-kernel step at
    2048 and under BRK_TT_NO_FUSED=1, the fp32 products."""
    if no_fused:
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    E = S = 64 if B != 1000 else 128
    m = _model(dev, E, S, tc, temperature=tau, candidateProbKey="p", weightKey="w")
    o = _oracle(m, E, S, tc, tau)
    uid, iid, p, w = _inputs(dev, B)
    lgot = m._step(uid, iid, None, True, extras=(p, w)).item()
    ic = iid.cpu().numpy()
    lref = o.loss_and_grads(uid.cpu().numpy(), ic, cand_ids=ic, cand_prob=p.cpu().numpy(), sample_weight=w.cpu().numpy())
    _close_to_oracle(m, o, E, S, lgot, lref)
    # forward only: the same loss, nothing accumulated
    _zero(m)
    np.testing.assert_allclose(m._step(uid, iid, None, False, extras=(p, w)).item(), lgot, rtol=1e-5)
    assert all(float(g.abs().max()) == 0.0 for g in _grads(m, E, S))


def _run_paths(dev, monkeypatch, B, E, S, kw, extras_fn, paths=("fused", "multi")):
    out = {}
    for path in paths:
        if path == "multi":
            monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
        else:
            monkeypatch.delenv("BRK_TT_NO_FUSED", raising=False)
        m = _model(dev, E, S, True, **kw)
        uid, iid, p, w = _inputs(dev, B, seed=5)
        loss = m._step(uid, iid, None, True, extras=extras_fn(p, w)).item()
        out[path] = (loss, [g.clone() for g in _grads(m, E, S)])
    return out


def test_one_launch_equals_the_multi_kernel_step_with_options(dev, monkeypatch):
    """Same inputs and options on both paths, tolerances of test_twotower_one_launch_step_equals_the_multi_kernel_step."""
    r = _run_paths(dev, monkeypatch, 1000, 128, 128, dict(temperature=0.5, candidateProbKey="p", weightKey="w"),
                   lambda p, w: (p, w))
    np.testing.assert_allclose(r["fused"][0], r["multi"][0], rtol=1e-5)
    for a, b in zip(r["fused"][1], r["multi"][1]):
        assert (a - b).abs().max().item() <= 5e-4 * b.abs().max().item()


@pytest.mark.parametrize("B", [1000, 2048])
def test_neutral_options_equal_the_option_free_step(dev, B):
    """tau = 1, p = 1, w = 1 against the model without options (the option-free kernels): loss rtol 1e-6.  Gradients: the
    float REDs of dq / dc and of the row gradients sum in a different order from run to run, which moves the option-free
    step itself by up to ~2e-5 of the largest entry (measured on a B200); the bound is 1e-4 of it, and the run-to-run
    difference of two option-free steps is printed beside the neutral one, with whether the results are bit-equal."""
    E = S = 128
    res = []
    for kw in ({}, dict(temperature=1.0, candidateProbKey="p", weightKey="w"), {}):
        m = _model(dev, E, S, True, **kw)
        uid, iid, _, _ = _inputs(dev, B, seed=7)
        ones = torch.ones(B, dtype=torch.float32, device=dev)
        loss = m._step(uid, iid, None, True, extras=(ones, ones) if kw else None).item()
        res.append((loss, [g.clone() for g in _grads(m, E, S)]))
    np.testing.assert_allclose(res[1][0], res[0][0], rtol=1e-6)
    bit = res[1][0] == res[0][0]
    worst, noise = 0.0, 0.0
    for a, b, c in zip(res[1][1], res[0][1], res[2][1]):
        scale = b.abs().max().item()
        worst = max(worst, (a - b).abs().max().item() / scale)
        noise = max(noise, (c - b).abs().max().item() / scale)
        bit = bit and torch.equal(a, b)
    print(f"neutral options B={B}: gradients within {worst:.1e} of the largest entry (two option-free runs: {noise:.1e}); "
          f"bit-equal: {bit}")
    assert worst <= 1e-4


@pytest.mark.parametrize("path", ["fused", "multi"])
def test_weights_scale_the_loss_and_gradients(dev, monkeypatch, path):
    B, E, S = 1000, 128, 128
    two = _run_paths(dev, monkeypatch, B, E, S, dict(temperature=0.5, weightKey="w"),
                     lambda p, w: (None, torch.full_like(w, 2.0)), paths=(path,))[path]
    one = _run_paths(dev, monkeypatch, B, E, S, dict(temperature=0.5, weightKey="w"),
                     lambda p, w: (None, torch.ones_like(w)), paths=(path,))[path]
    np.testing.assert_allclose(two[0], 2 * one[0], rtol=1e-6)
    for a, b in zip(two[1], one[1]):                                   # RED order: see test_neutral_options_...
        assert (a - 2 * b).abs().max().item() <= 1e-4 * 2 * b.abs().max().item()
    # a single weight of 0 removes that row's loss term
    k = 17
    m = _model(dev, E, S, True, temperature=0.5, weightKey="w")
    o = _oracle(m, E, S, True, 0.5)
    uid, iid, _, _ = _inputs(dev, B, seed=5)
    w = torch.ones(B, dtype=torch.float32, device=dev); w[k] = 0.0
    lz = m._step(uid, iid, None, False, extras=(None, w)).item()
    with torch.no_grad():
        q, c = o.towers(uid.cpu().numpy(), iid.cpu().numpy())
        s = o.mm(q, c.T) / 0.5
        ids = iid.cpu()
        s = s + ((ids[:, None] == ids[None, :]).float() - torch.eye(B)) * (float(np.finfo(np.float32).min) / 100.0)
        rows = torch.nn.functional.cross_entropy(s, torch.arange(B), reduction="none").double()
    np.testing.assert_allclose(lz, float(rows.sum() - rows[k]), rtol=2e-3)
    np.testing.assert_allclose(m._step(uid, iid, None, False, extras=(None, torch.ones_like(w))).item() - lz, float(rows[k]),
                               rtol=5e-2, atol=1e-2 * abs(lz) / B)


@pytest.mark.parametrize("path,B", [("fused", 333), ("multi", 333), ("multi", 2048)])
def test_streaming_estimator_state_equals_the_oracle(dev, monkeypatch, path, B):
    """Ten training steps (step + Adagrad, brk_twotower_train_step_retrieval) with repeated ids: last, gap and the step
    counter equal Algorithm 2's sequential loop bit for bit; duplicates update once; test_step changes nothing; the loss
    uses the updated probabilities."""
    from oracle import twotower_retrieval as OR
    if path == "multi":
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
    E = S = 64
    m = _model(dev, E, S, True, temperature=0.5, streamingFrequency=0.05)
    m.compile("Adagrad", learningRate=0.1)
    f = OR.StreamingFrequency(I + 2, alpha=0.05)
    g = torch.Generator(device=dev); g.manual_seed(11)
    for step in range(10):
        uid = torch.randint(2, U + 2, (B,), generator=g, device=dev, dtype=torch.int32)
        iid = torch.randint(2, 40 + 2 * step, (B,), generator=g, device=dev, dtype=torch.int32)   # heavy repeats, shifting
        if step == 9:                                                  # the last step's loss against the oracle
            o = _oracle(m, E, S, True, 0.5)
        loss = m._train_ids(uid, iid, None).item()
        f.update(iid.cpu().numpy())
    torch.cuda.synchronize()
    assert np.array_equal(m._freq["last"].cpu().numpy(), f.last)
    assert np.array_equal(m._freq["gap"].cpu().numpy().view(np.int32), f.gap.view(np.int32))
    assert int(m._freq["step"].item()) == 10
    ic = iid.cpu().numpy()
    lref = o.loss(uid.cpu().numpy(), ic, cand_ids=ic, cand_prob=f.probability(ic))
    state = [t.clone() for t in m._freq.values()]
    lt = m.test_step({"u": list(uid.cpu().numpy() - 2), "i": list(ic - 2)})["loss"].item()
    for a, b in zip(state, m._freq.values()):
        assert torch.equal(a, b)                                       # test_step leaves the state alone
    np.testing.assert_allclose(loss, float(lref), rtol=2e-3)          # step 10 scored with the probabilities it updated
    assert np.isfinite(lt)


def test_estimator_loss_uses_the_updated_probabilities(dev):
    from oracle import twotower_retrieval as OR
    B, E, S = 333, 64, 64
    m = _model(dev, E, S, True, streamingFrequency=0.3)
    f = OR.StreamingFrequency(I + 2, alpha=0.3)
    g = torch.Generator(device=dev); g.manual_seed(12)
    for step in range(3):
        uid = torch.randint(2, U + 2, (B,), generator=g, device=dev, dtype=torch.int32)
        iid = torch.randint(2, 60, (B,), generator=g, device=dev, dtype=torch.int32)
        o = _oracle(m, E, S, True, None)
        f.update(iid.cpu().numpy())
        _zero(m)
        lgot = m._step(uid, iid, None, True).item()
        ic = iid.cpu().numpy()
        lref = o.loss_and_grads(uid.cpu().numpy(), ic, cand_ids=ic, cand_prob=f.probability(ic))
        _close_to_oracle(m, o, E, S, lgot, lref)
        # computeLossTfrs reads the same state
        info = {"u": list(uid.cpu().numpy() - 2), "i": list(ic - 2)}
        qe, ce = m.computeEmb(info)
        np.testing.assert_allclose(m.computeLossTfrs(qe, ce, info).item(), float(lref), rtol=2e-3)


def test_graph_replayed_fit_equals_eager_steps(dev):
    B, E, S, n = 256, 64, 64, 6
    rng = np.random.default_rng(13)
    batches = [{"u": list(rng.integers(0, U, B)), "i": list(rng.integers(0, 50, B)), "w": list(rng.uniform(0, 2, B))}
               for _ in range(n)]
    a = _model(dev, E, S, True, temperature=0.3, weightKey="w", streamingFrequency=0.1).compile("Adagrad", learningRate=0.1)
    b = _model(dev, E, S, True, temperature=0.3, weightKey="w", streamingFrequency=0.1).compile("Adagrad", learningRate=0.1)
    a.fit(batches, epochs=2, graph=True)
    eager = []
    for e in range(2):
        ls = [b.train_step(info)["loss"].item() for info in batches]
        eager.append(sum(ls) / n)
    for k in ("last", "gap", "step"):
        assert torch.equal(a._freq[k], b._freq[k]), k
    assert int(a._freq["step"].item()) == 2 * n
    np.testing.assert_allclose(a.history["loss"], eager, rtol=1e-4)
    for ta, tb in zip((a.userTower.emb, a.itemTower.emb, a.userTower.dense), (b.userTower.emb, b.itemTower.emb, b.userTower.dense)):
        assert (ta.w - tb.w).abs().max().item() <= 1e-3


@pytest.mark.parametrize("B", [1000, 2048])
def test_train_step_with_adagrad_equals_step_plus_adagrad(dev, B):
    """brk_twotower_train_step_retrieval (Adagrad in the same launch at 1000, step + optimizer kernels at 2048) against
    brk_twotower_step_retrieval followed by the library's Adagrad passes, five steps."""
    E = S = 128
    kw = dict(temperature=2.0, candidateProbKey="p", weightKey="w")
    a = _model(dev, E, S, True, **kw).compile("Adagrad", learningRate=0.1)
    b = _model(dev, E, S, True, **kw).compile("Adagrad", learningRate=0.1)
    uid, iid, p, w = _inputs(dev, B, seed=9)
    la, lb = [], []
    for k in range(5):
        uk, ik, pk, wk = torch.roll(uid, k), torch.roll(iid, 2 * k), torch.roll(p, 3 * k), torch.roll(w, k)
        la.append(a._train_ids(uk, ik, None, extras=(pk, wk)).item())
        lb.append(b._step(uk, ik, None, True, extras=(pk, wk)).item())
        b.optimizer.apply([b.userTower.emb, b.itemTower.emb], dense=[b.userTower.dense, b.itemTower.dense])
    np.testing.assert_allclose(la, lb, rtol=1e-4)
    for ta, tb in zip((a.userTower.emb, a.itemTower.emb, a.userTower.dense, a.itemTower.dense),
                      (b.userTower.emb, b.itemTower.emb, b.userTower.dense, b.itemTower.dense)):
        assert (ta.w - tb.w).abs().max().item() <= 5e-3
        assert ta.g.abs().max().item() == 0.0                           # accumulators left clean


def test_rejections(dev):
    from binrec_b200 import _native as N
    with pytest.raises(ValueError, match="rdZero"):
        _model(dev, 16, 16, True, rdZero=True, resKey="r", temperature=0.5)
    with pytest.raises(ValueError, match="global_negatives"):
        _model(dev, 16, 16, True, global_negatives=True, weightKey="w")
    with pytest.raises(ValueError, match="both"):
        _model(dev, 16, 16, True, candidateProbKey="p", streamingFrequency=0.01)
    for tau in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError, match="temperature"):
            _model(dev, 16, 16, True, temperature=tau)
    with pytest.raises(ValueError, match="alpha"):
        _model(dev, 16, 16, True, streamingFrequency=1.5)
    # the C ABI
    m = _model(dev, 16, 16, True, streamingFrequency=0.01)
    B = 64
    uid, iid, p, w = _inputs(dev, B)
    ws = m._workspace(B)
    ut, it = m.userTower.c_struct(), m.itemTower.c_struct()
    loss = torch.empty(1, dtype=torch.float32, device=dev)

    def call(mode=0x100, **over):
        rt = m._rt((None, None))
        for k, v in over.items():
            setattr(rt, k, v)
        return N.lib().brk_twotower_step_retrieval(N.ctx(dev), C.byref(ut), C.byref(it), N.ptr(uid), N.ptr(iid), N.ptr(iid),
                                                   N.ptr(w), B, mode, 1, C.byref(ws), N.ptr(loss), N.stream_ptr(), C.byref(rt))

    def rejected(msg, **kw):
        assert call(**kw) == -1
        assert msg in N.lib().brk_last_error().decode(), N.lib().brk_last_error()

    rejected("temperature", inv_temperature=0.0)
    rejected("temperature", inv_temperature=float("inf"))
    rejected("temperature", inv_temperature=float("nan"))
    rejected("exclusive", cand_prob=p.data_ptr())
    rejected("rdZero", mode=0x101)
    rejected("item table has", rows=I + 1)
    rejected("step counter", step=None)
    rejected("step counter", gap=None)
    rejected("alpha", alpha=0.0)
    assert int(m._freq["step"].item()) == 0                            # nothing ran
    assert call() == 0
    torch.cuda.synchronize()
    assert int(m._freq["step"].item()) == 1


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    dist.init_process_group("nccl", device_id=dev)
    try:
        from binrec_b200 import distributed as D
        E = S = 64
        n = 600
        rng = np.random.default_rng(21)
        info = {"u": list(rng.integers(0, U, n)), "i": list(rng.integers(0, 80, n)),
                "p": list((rng.random(n) ** 3).astype(np.float32)), "w": list(rng.uniform(0, 2, n).astype(np.float32))}
        lo, hi = D.local_slice(n)
        mine = {k: v[lo:hi] for k, v in info.items()}
        m = _model(dev, E, S, True, temperature=0.5, candidateProbKey="p", weightKey="w").compile("Adagrad", learningRate=0.1)
        o = _oracle(m, E, S, True, 0.5)
        got = m.train_step(mine)["loss"].item()
        ic = np.asarray(mine["i"]) + 2
        ref = float(o.loss(np.asarray(mine["u"]) + 2, ic, cand_ids=ic, cand_prob=np.asarray(mine["p"]),
                           sample_weight=np.asarray(mine["w"])))
        ret[rank] = (got, ref)
    except Exception as e:                                             # pragma: no cover - reported by the parent
        ret[rank] = repr(e)
    finally:
        dist.destroy_process_group()


def test_mirrored_per_replica_loss_with_options_two_gpus():
    """Mirrored data parallelism on 2 GPUs: each rank passes its slice's probabilities and weights to the same kernels;
    its per-replica loss equals the oracle over its slice."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
    for r in range(2):
        assert not isinstance(ret.get(r), str) and r in ret, ret.get(r)
        got, ref = ret[r]
        np.testing.assert_allclose(got, ref, rtol=2e-3)
