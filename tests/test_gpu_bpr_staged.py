"""The one-launch BPR step with its Adam operands staged in shared memory (bpr_steps_coop, default path) against the NumPy
oracle, against the global-memory Adam of BRK_BPR_NO_SMEM_ADAM=1 and against the separate kernels of BRK_NO_COOP=1: losses,
tables and Adam moments, over launch sizes, table shapes that stress the per-CTA slicing, the large-table fallback and the
self-sampling (host-fed / mapped) paths.  A launch that ends without its trailing grid barrier must leave the barrier base
where the next launch expects it; a wrong base traps the next launch, which raises here."""
import contextlib
import os

import numpy as np
import pytest
import torch

from oracle import bpr as OB
from oracle import philox as OP

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-5, 1e-6                 # losses vs the oracle (tests/test_gpu_kernels.py)
W_RTOL, W_ATOL = 1e-4, 2e-6             # tables vs the oracle after several steps
P_RTOL, P_ATOL = 1e-5, 1e-7             # two GPU paths: same REDs, only their order differs


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch.device("cuda:0")


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update(kv)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def frame(U, I, total, seed):
    rng = np.random.default_rng(seed)
    return tuple(rng.integers(0, m, total).astype(np.int32) for m in (U, I, I))


def net_for(dev, U, I, d, u, p, n):
    from binrec_b200.BPRModel import BPRNet
    net = BPRNet(U, I, d, seed=42, device=dev)
    net.set_training_pairs(u, p); net.set_negatives(n)
    return net


def train(net, launches, B, **kv):
    """launches: list of batch-index lists, one cooperative launch each; returns all step losses.  The launches run with
    BRK_COOP_TRACE=1, so that adam_path() can tell which Adam the last one ran."""
    with env(BRK_COOP_TRACE="1", **kv):
        out = [net.train_steps(order, B).cpu().numpy() for order in launches]
    torch.cuda.synchronize()
    return np.concatenate(out)


def adam_path():
    """'smem' or 'global': the Adam of the last traced single-GPU cooperative launch (word 4 of its stamps)."""
    import ctypes
    from binrec_b200 import _native as N
    lib = N.lib(); lib.brk_coop_trace_read.argtypes = [ctypes.c_void_p, ctypes.c_int32]
    buf = (ctypes.c_uint64 * 8)()
    assert lib.brk_coop_trace_read(buf, 8) == 0
    return {1: "smem", 0: "global"}[int(buf[4])]


def oracle_run(U, I, d, u, p, n, B, order):
    orc = OB.BPROracle(U, I, d, seed=42)
    ref = []
    for b in order:
        sl = slice(b * B, min(len(u), (b + 1) * B))
        ref.append(orc.step(u[sl], p[sl], n[sl]))
    return orc, np.array(ref)


def check_oracle(net, orc, losses, ref):
    np.testing.assert_allclose(losses, ref, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(net.user.w.cpu().numpy(), orc.user, rtol=W_RTOL, atol=W_ATOL)
    np.testing.assert_allclose(net.item.w.cpu().numpy(), orc.item, rtol=W_RTOL, atol=W_ATOL)
    np.testing.assert_allclose(net.user.m.cpu().numpy(), orc.mu, rtol=1e-4, atol=1e-8)
    np.testing.assert_allclose(net.user.v.cpu().numpy(), orc.vu, rtol=1e-4, atol=1e-12)
    np.testing.assert_allclose(net.item.m.cpu().numpy(), orc.mi, rtol=1e-4, atol=1e-8)
    np.testing.assert_allclose(net.item.v.cpu().numpy(), orc.vi, rtol=1e-4, atol=1e-12)
    assert not net.grad_arena.any().item()


def check_same(a, b, la, lb):
    np.testing.assert_allclose(la, lb, rtol=P_RTOL, atol=P_ATOL)
    for x, y in ((a.user, b.user), (a.item, b.item)):
        for t in ("w", "m", "v"):
            np.testing.assert_allclose(getattr(x, t).cpu().numpy(), getattr(y, t).cpu().numpy(), rtol=P_RTOL, atol=P_ATOL)
    assert a.optimizer.step.item() == b.optimizer.step.item()


def test_single_step_launches_equal_one_long_launch_and_separate_kernels(dev):
    U, I, d, B = 400, 300, 64, 512
    total = 5 * B + 77                                      # ragged last batch
    u, p, n = frame(U, I, total, 1)
    order = [(3 * k + 1) % 6 for k in range(20)]
    orc, ref = oracle_run(U, I, d, u, p, n, B, order)
    nets, losses = {}, {}
    for name, launches, kv in (("one_per_launch", [[b] for b in order], {}),
                               ("one_launch", [order], {}),
                               ("no_smem", [order], {"BRK_BPR_NO_SMEM_ADAM": "1"}),
                               ("no_coop", [order], {"BRK_NO_COOP": "1"})):
        nets[name] = net_for(dev, U, I, d, u, p, n)
        losses[name] = train(nets[name], launches, B, **kv)
        if name != "no_coop":
            assert adam_path() == ("global" if name == "no_smem" else "smem")
        check_oracle(nets[name], orc, losses[name], ref)
    for name in ("one_launch", "no_smem", "no_coop"):
        check_same(nets["one_per_launch"], nets[name], losses["one_per_launch"], losses[name])


def test_moments_survive_a_checkpoint_between_launches(dev, tmp_path):
    from binrec_b200 import checkpoint as CK
    U, I, d, B = 400, 300, 64, 512
    u, p, n = frame(U, I, 6 * B, 2)
    first, second = [0, 3, 5, 1, 2, 4, 0], [2, 5, 1, 3, 3]
    orc, ref = oracle_run(U, I, d, u, p, n, B, first + second)
    a = net_for(dev, U, I, d, u, p, n)
    la = train(a, [first], B)
    # moments written back at the end of the launch: what the oracle has after the same steps
    orc1, _ = oracle_run(U, I, d, u, p, n, B, first)
    check_oracle(a, orc1, la, ref[:len(first)])
    CK.save_state_dict(str(tmp_path / "cp"), a.state_dict())
    b = net_for(dev, U, I, d, u, p, n)
    b.load_state_dict({k: v.to(dev) for k, v in CK.load_state_dict(str(tmp_path / "cp")).items()})
    lb = train(b, [second], B)
    lc = train(a, [second], B)
    check_oracle(b, orc, np.concatenate([la, lb]), ref)
    check_same(a, b, lc, lb)


@pytest.mark.parametrize("U,I,d,B,path", [
    (401, 299, 4, 1024, "smem"),          # rows * d not a multiple of grid * 4
    (7, 5, 4, 4096, "smem"),              # tables smaller than one float4 per CTA: most CTAs own nothing
    (333, 211, 32, 700, "smem"),
    (400, 300, 64, 512, "smem"),
    (257, 129, 128, 1000, "smem"),
    (3000, 400, 64, 512, "global"),       # slices too large for the shared-memory budget: global-memory Adam
    (2000, 1500, 128, 512, "global"),     # the same at d = 128
])
def test_table_shapes_match_oracle_and_global_adam(dev, U, I, d, B, path):
    total = 4 * B + 33
    u, p, n = frame(U, I, total, U + d)
    order = [4, 0, 2, 1, 3, 4]
    orc, ref = oracle_run(U, I, d, u, p, n, B, order)
    a = net_for(dev, U, I, d, u, p, n)
    la = train(a, [order[:1], order[1:3], order[3:]], B)
    assert adam_path() == path
    check_oracle(a, orc, la, ref)
    b = net_for(dev, U, I, d, u, p, n)
    lb = train(b, [order[:1], order[1:3], order[3:]], B, BRK_BPR_NO_SMEM_ADAM="1")
    assert adam_path() == "global"
    check_same(a, b, la, lb)


@pytest.mark.parametrize("path", ["copy", "mapped"])
def test_sampling_mode_37_steps(dev, path):
    """Host-fed launches of 2, 4, 8, 16 and 7 steps, and one mapped launch of 37: the stager threads fill step s + 1
    while the others run Adam over the CTA's whole slice."""
    from binrec_b200.BPRModel import BPRNet
    U, I, d, B = 300, 200, 64, 256
    rng = np.random.default_rng(31)
    key = np.unique(rng.integers(0, U * I, 4000))
    u, p = (key // I).astype(np.int32), (key % I).astype(np.int32)
    perm = rng.permutation(len(u)); u, p = u[perm], p[perm]
    nb = len(u) // B + 1
    order = [(5 * k + 2) % nb for k in range(37)]
    hu, hp = torch.from_numpy(u).pin_memory(), torch.from_numpy(p).pin_memory()
    res = {}
    for name, kv in (("smem", {}), ("global", {"BRK_BPR_NO_SMEM_ADAM": "1"})):
        net = BPRNet(U, I, d, seed=42, device=dev)
        net.set_training_pairs(u, p)
        with env(BRK_COOP_TRACE="1", **kv):
            fn = net.train_steps_from_host if path == "copy" else net.train_steps_mapped
            losses = fn(hu, hp, order, B, 7, 5)
            torch.cuda.synchronize()
        assert adam_path() == name
        res[name] = (net, losses.numpy().copy())
    orc = OB.BPROracle(U, I, d, seed=42)
    indptr, sitems = OP.build_csr(u, p, U)
    ref = []
    for b in order:
        sl = slice(b * B, min(len(u), (b + 1) * B))
        ref.append(orc.step(u[sl], p[sl], OP.bpr_negatives(u[sl], 7, 5, I, indptr, sitems, first_index=b * B)))
    net, losses = res["smem"]
    np.testing.assert_allclose(losses, np.array(ref), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(net.user.w.cpu().numpy(), orc.user, rtol=W_RTOL, atol=W_ATOL)
    np.testing.assert_allclose(net.item.w.cpu().numpy(), orc.item, rtol=W_RTOL, atol=W_ATOL)
    np.testing.assert_allclose(net.item.m.cpu().numpy(), orc.mi, rtol=1e-4, atol=1e-8)
    np.testing.assert_allclose(net.item.v.cpu().numpy(), orc.vi, rtol=1e-4, atol=1e-12)
    check_same(res["smem"][0], res["global"][0], res["smem"][1], res["global"][1])


def test_launch_sizes_keep_the_barrier_base(dev):
    """Launches of 1, 2, 37, 1 and 16 steps back to back, alternating with the path that keeps the trailing barrier:
    every launch must start from the base the previous one left (a wrong one traps or stalls the launch)."""
    U, I, d, B = 400, 300, 64, 512
    u, p, n = frame(U, I, 6 * B, 5)
    sizes = [1, 2, 37, 1, 16]
    order = [(7 * k + 3) % 6 for k in range(sum(sizes))]
    launches, at = [], 0
    for s in sizes:
        launches.append(order[at:at + s]); at += s
    orc, ref = oracle_run(U, I, d, u, p, n, B, order)
    a = net_for(dev, U, I, d, u, p, n)
    got = []
    for i, ln in enumerate(launches):
        got.append(train(a, [ln], B, **({"BRK_BPR_NO_SMEM_ADAM": "1"} if i % 2 else {})))
    check_oracle(a, orc, np.concatenate(got), ref)
    assert a.optimizer.step.item() == len(order)
