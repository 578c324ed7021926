"""The grid barrier of the cooperative step kernels (brk_grid_barrier) keeps its state per context in device memory: the
counter base and, for NeuMF, the tag of the self-validating BatchNorm slot words are read by the kernel at entry and
written back by it.  So a captured NeuMF step replays correctly from a CUDA graph and mixes with eager launches, and each
device of a process has its own barrier words.

The NeuMF batches hold every user and every item at most once: each embedding-gradient element then receives exactly one
RED, and the one-launch step, whose other sums run in a fixed order, is bit-reproducible, so the runs compared here must
agree bit for bit.  With repeated rows the order of the REDs changes from run to run, and over several steps the TF32
products and BatchNorm amplify those last-bit differences to ~1e-3 in the weights, eager run against eager run."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
U, I = 6040, 3706


def _distinct_rows_batch(seed, B):
    rng = np.random.default_rng(seed)
    u = rng.permutation(U)[:B].astype(np.int32)
    i = rng.permutation(I)[:B].astype(np.int32)
    y = (rng.random(B) < 0.2).astype(np.float32)
    return u, i, y


def _neumf_state(net, loss):
    """Loss, weights and Adam moments of the four tables and the dense block, BatchNorm moving statistics (on the host)."""
    tabs = dict(zip(("uMLP", "iMLP", "uMF", "iMF", "dense"), net.tables() + [net.dense]))
    state = {f"{name}.{k}": getattr(t, k).cpu() for name, t in tabs.items() for k in "wmv"}
    state.update(bn_moving=net.bn_moving.cpu(), loss=loss.cpu())
    return state


def _assert_bit_equal(got, want):
    for k in want:
        assert torch.equal(got[k], want[k]), k


# dropout 0: the dropout seed and epoch are host values that a capture bakes in
VARIANTS = {"class_spec": dict(tensor_cores=True),
            "he_et_al": dict(mf_dim=8, mf_mode="hadamard", batch_norm=False)}


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_neumf_graph_replay_equals_eager_steps(dev, variant):
    """3 eager steps, one captured step replayed 5 times, 1 eager step == 9 eager steps.  A replay must wait at the
    grid barrier of its own launch and accept only its own BatchNorm slot words, and the eager step after the replays
    must find the barrier base where they left it.  24 tiles: most CTAs of the grid are helper CTAs (grid = SM count)."""
    from binrec_b200.NeuMFModel import NeuMFNet
    B = 3072
    u, i, y = (torch.from_numpy(x).to(dev) for x in _distinct_rows_batch(8, B))
    a = NeuMFNet(U, I, 32, dropout=0.0, device=dev, **VARIANTS[variant])
    b = NeuMFNet(U, I, 32, dropout=0.0, device=dev, **VARIANTS[variant])
    assert a.tensor_cores
    oa, la = torch.empty(B, device=dev), torch.empty(1, device=dev)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            a.train_on_batch(u, i, y, out=oa, loss_out=la)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            a.train_on_batch(u, i, y, out=oa, loss_out=la)
        for _ in range(5):
            g.replay()
        a.train_on_batch(u, i, y, out=oa, loss_out=la)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(9):
        lb, _ = b.train_on_batch(u, i, y)
    torch.cuda.synchronize()
    assert int(a.optimizer.state[0].item()) == int(b.optimizer.state[0].item()) == 9
    _assert_bit_equal(_neumf_state(a, la), _neumf_state(b, lb))


def _neumf_grads(net, loss, out):
    """Loss, predictions and the gradients of the four tables and the dense block after forward_backward (on the host)."""
    tabs = dict(zip(("uMLP", "iMLP", "uMF", "iMF", "dense"), net.tables() + [net.dense]))
    return dict({f"{name}.g": t.g.cpu().numpy() for name, t in tabs.items()}, loss=loss.cpu().numpy(), out=out.cpu().numpy())


def _run_on(dev, monkeypatch):
    """One NeuMF tensor-core step, one BPR train_steps launch and one two-tower step on `dev`; then the multi-kernel
    launchers whose kernels ask for more than 48 KB of shared memory: the five-kernel tensor-core NeuMF step
    (csrc/neumf_tc.cu), the fp32 tiled one (csrc/neumf2.cu), the script spec's (csrc/neumf.cu) and the multi-kernel
    two-tower step (csrc/gemm_tc.cu)."""
    from binrec_b200.BPRModel import BPRNet
    from binrec_b200.NeuMFModel import NeuMFNet
    from binrec_b200.twoTower import TwoTowerModel
    with torch.cuda.device(dev):
        net = NeuMFNet(U, I, 32, dropout=0.2, device=dev, tensor_cores=True)
        nl, _ = net.train_on_batch(*(torch.from_numpy(x).to(dev) for x in _distinct_rows_batch(3, 2048)), first_index=7, epoch=1)
        neumf = _neumf_state(net, nl)

        multi = {}
        monkeypatch.setenv("BRK_NEUMF_NO_FUSED", "1")
        for name, E, kw in (("five_kernel", 64, dict(tensor_cores=True)), ("fp32_tiled", 32, dict(tensor_cores=False)),
                            ("script_spec", 10, dict(hidden=(100, 50, 10), tensor_cores=False))):
            net = NeuMFNet(U, I, E, dropout=0.2, device=dev, **kw)
            batch = (torch.from_numpy(x).to(dev) for x in _distinct_rows_batch(4, 2048))
            loss, out = net.forward_backward(*batch, first_index=7, epoch=1)
            multi[name] = _neumf_grads(net, loss, out)
        monkeypatch.delenv("BRK_NEUMF_NO_FUSED")

        rng = np.random.default_rng(5)
        Ub, Ib, B = 400, 300, 512
        up, pp, nn = (rng.integers(0, m, 6 * B).astype(np.int32) for m in (Ub, Ib, Ib))
        bpr = BPRNet(Ub, Ib, 64, seed=42, device=dev)
        bpr.set_training_pairs(up, pp)
        bpr.set_negatives(nn)
        bl = bpr.train_steps([2, 0, 5, 1], B).cpu().numpy()
        bpr_out = (bl, {f"{t}.{k}": getattr(getattr(bpr, t), k).cpu().numpy() for t in ("user", "item") for k in "wmv"})

        users = [f"u{j}" for j in range(300)]
        items = [f"m{j}" for j in range(200)]
        tt = TwoTowerModel(32, 200, 300, "CUSTOMER_ID", "MATERIAL", users, items, semb=16, device=dev, tensor_cores=True)
        tt.compile("Adagrad", learningRate=0.1)
        info = {"CUSTOMER_ID": [users[j] for j in rng.integers(0, 300, 256)],
                "MATERIAL": [items[j] for j in (200 * rng.random(256) ** 2).astype(np.int64)]}
        tl = tt.train_step(info)["loss"].item()
        tabs = {f"{n}.{t}": getattr(getattr(tt, n), t) for n in ("userTower", "itemTower") for t in ("emb", "dense")}
        tt_out = (tl, {f"{name}.{k}": getattr(tab, k).cpu().numpy() for name, tab in tabs.items() for k in "wm"})

        # multi-kernel two-tower step: every product through gemm_tf32 (leading dimensions multiples of 4)
        monkeypatch.setenv("BRK_TT_NO_FUSED", "1")
        tt = TwoTowerModel(64, 200, 300, "CUSTOMER_ID", "MATERIAL", users, items, semb=64, device=dev, tensor_cores=True)
        tt.compile("Adagrad", learningRate=0.1)
        info = {"CUSTOMER_ID": [users[j] for j in rng.integers(0, 300, 512)],
                "MATERIAL": [items[j] for j in (200 * rng.random(512) ** 2).astype(np.int64)]}
        tl = tt.train_step(info)["loss"].item()
        monkeypatch.delenv("BRK_TT_NO_FUSED")
        tabs = {f"{n}.{t}": getattr(getattr(tt, n), t) for n in ("userTower", "itemTower") for t in ("emb", "dense")}
        multi["twotower"] = (tl, {f"{name}.{k}": getattr(tab, k).cpu().numpy() for name, tab in tabs.items() for k in "wm"})
        torch.cuda.synchronize()
    return neumf, bpr_out, tt_out, multi


def _assert_twotower_close(t1, t0):
    np.testing.assert_allclose(t1[0], t0[0], rtol=1e-5)
    for k in t0[1]:
        np.testing.assert_allclose(t1[1][k], t0[1][k], rtol=1e-4, atol=2e-5 if k.endswith(".w") else 1e-6, err_msg=k)


def test_cooperative_steps_on_two_devices_in_one_process(monkeypatch):
    """Each device's context has its own barrier words and its own shared-memory opt-in of the kernels: the same steps
    on cuda:1, after cuda:0 ran them in this process, give what cuda:0 gave.  BPR and two-tower repeat rows, so they are
    held to the tolerances of two runs of the same step (tests/test_gpu_bpr_staged.py, tests/test_gpu_twotower.py).  The
    multi-kernel NeuMF steps sum their dense gradients with REDs in no fixed order: their loss and predictions are held to
    rtol 1e-5, each gradient tensor to 1e-5 of its largest entry (compared before the optimizer: Adam would turn the
    last-bit noise of a near-zero gradient into a step of +-lr)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    (n0, b0, t0, m0), (n1, b1, t1, m1) = _run_on(torch.device("cuda:0"), monkeypatch), _run_on(torch.device("cuda:1"), monkeypatch)
    _assert_bit_equal(n1, n0)
    np.testing.assert_allclose(b1[0], b0[0], rtol=1e-5, atol=1e-7)
    for k in b0[1]:
        np.testing.assert_allclose(b1[1][k], b0[1][k], rtol=1e-5, atol=1e-7, err_msg=k)
    _assert_twotower_close(t1, t0)
    _assert_twotower_close(m1.pop("twotower"), m0.pop("twotower"))
    for name in m0:
        for k, want in m0[name].items():
            got = m1[name][k]
            if k.endswith(".g"):
                assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max(), (name, k)
            else:
                np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-7, err_msg=f"{name} {k}")
