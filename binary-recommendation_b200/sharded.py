"""Row-sharded embedding tables across GPUs (BASELINE.json configs[3]: NeuMF with 20M x 2M x 64 tables).

The reference mirrors every variable on every worker (tf.distribute MultiWorkerMirroredStrategy,
/root/reference/src/models/RModel.py:119-121) and all-reduces full-table gradients; tables of this size
do not fit that scheme.  Here row r of a table lives on rank r % G at local row r // G and a batch is
split over the ranks (data parallel).  Two ways to move rows and row gradients between ranks:

  mode "peer" (the product path): every shard (weights, gradient accumulator, touched bitmask) is
      allocated in NVLink peer-mapped symmetric memory; the fused NeuMF kernels gather peer rows with
      ordinary loads and send row gradients as REDs into the owner's accumulator
      (brk_neumf_step_sharded).  The exchange is carried by the gather / scatter instructions
      themselves -- no staging buffers, no separate all-to-all.  Per step:
          fused fwd/bwd  ->  brk_peer_barrier  ->  lazy Adam on the owned shards  ->
          brk_dp_adam_peer on the (mirrored) dense block, whose own barriers also fence the next step.
  mode "nccl" (the baseline the above is measured against): all-to-all of ids, owners gather rows,
      all-to-all of rows, fused step on the received rows, all-to-all of row gradients, owners
      scatter-add (NCCL all_to_all_single around brk_gather_rows / brk_scatter_add_rows).

The dense MLP / BatchNorm parameters are mirrored; their gradients are summed and Adam applied by the
fused peer kernel (or one NCCL all-reduce in mode "nccl").  BatchNorm statistics stay per replica
(MirroredStrategy's default).  Row-sparse (lazy) Adam on the tables: the exact Keras dense-equivalent
pass over 20M-row tables every step is not an option (SURVEY.md section 0.4).

`emulate=G` builds all G shards inside ONE process on one GPU (pointers are plain local pointers) so that
the sharded addressing can be checked against the unsharded model on a single-GPU box.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _native as N
from . import distributed as D
from . import hotpath as H
from .twoTower import Tower, TwoTowerModel


def shard_rows(rows, G):
    """Rows per shard (equal on every rank, as symmetric memory needs)."""
    return (rows + G - 1) // G


def save_sharded_model(dirpath, tables, replicated, G, rank, emulate, meta=None):
    """Checkpoint of a row-sharded model (checkpoint.py; SURVEY.md section 8 row f3): every rank writes its shards of
    the weights and optimizer slots, rank 0 the replicated tensors and -- after a barrier -- the manifest.
    tables: {name: ShardedTable}."""
    from . import checkpoint as CK
    ranks = list(range(G - 1, -1, -1)) if emulate else [rank]          # emulation: rank 0 (the manifest) goes last
    barrier = None
    if not emulate and G > 1:
        torch.cuda.synchronize()
        barrier = dist.barrier
    for r in ranks:
        shd = {}
        for name, t in tables.items():
            tab = t.tables[r]
            shd[name] = (tab.w, t.rows)
            if tab.m is not None:
                shd[name + "_m"] = (tab.m, t.rows)
            if tab.v is not None:
                shd[name + "_v"] = (tab.v, t.rows)
        CK.save_checkpoint(dirpath, replicated=replicated if r == 0 else None, sharded=shd, rank=r, world=G,
                           meta=meta, barrier=barrier)
    return dirpath


def load_sharded_model(dirpath, tables, G, rank, emulate):
    """Restores the shards this process owns -- whatever world size wrote the checkpoint.  Returns (replicated, meta)."""
    from . import checkpoint as CK
    rep, meta = {}, {}
    for r in (range(G) if emulate else [rank]):
        rep, shd, meta = CK.load_checkpoint(dirpath, r, G)
        for name, t in tables.items():
            tab = t.tables[r]
            tab.w.copy_(torch.from_numpy(shd[name]))
            if tab.m is not None and name + "_m" in shd:
                tab.m.copy_(torch.from_numpy(shd[name + "_m"]))
            if tab.v is not None and name + "_v" in shd:
                tab.v.copy_(torch.from_numpy(shd[name + "_v"]))
    if not emulate and G > 1:
        torch.cuda.synchronize()
        dist.barrier()                                   # nobody gathers peer rows before every owner has loaded
    return rep, meta


class ShardedTable:
    """One row-sharded embedding table: local shard as an H.Table plus every rank's shard pointers.
    slots / slot_init: optimizer slots of every shard, as H.Table (default: Adam's m and v at zero)."""

    def __init__(self, rows, d, G, rank, device, full_init=None, init_seed=0, symmetric=True, emulate=False, slots=2,
                 slot_init=0.0):
        self.rows, self.d, self.G, self.rank, self.device = int(rows), int(d), int(G), int(rank), device
        self.local_rows = shard_rows(rows, G)
        n = self.local_rows * d
        nt = (self.local_rows + 31) // 32
        self.emulate = emulate
        owners = range(G) if emulate else [rank]
        self.tables = {}
        self._keep = []
        ptr_w, ptr_g, ptr_t = [0] * G, [0] * G, [0] * G
        for r in owners:
            if symmetric and not emulate:
                import torch.distributed._symmetric_memory as symm_mem
                group = dist.group.WORLD.group_name
                w = symm_mem.empty(n, dtype=torch.float32, device=device)
                g = symm_mem.empty(n, dtype=torch.float32, device=device)
                t = symm_mem.empty(nt, dtype=torch.int32, device=device)
                hs = [symm_mem.rendezvous(x, group) for x in (w, g, t)]
                self._keep.append(hs)
                ptr_w, ptr_g, ptr_t = (list(h.buffer_ptrs) for h in hs)
            else:
                w = torch.empty(n, dtype=torch.float32, device=device)
                g = torch.empty(n, dtype=torch.float32, device=device)
                t = torch.empty(nt, dtype=torch.int32, device=device)
                ptr_w[r], ptr_g[r], ptr_t[r] = w.data_ptr(), g.data_ptr(), t.data_ptr()
            g.zero_(); t.zero_()
            w2 = w.view(self.local_rows, d)
            if full_init is not None:                       # shard r = rows r, r+G, r+2G, ... of the full matrix
                part = np.ascontiguousarray(full_init[r::G])
                w2.zero_()
                w2[:part.shape[0]].copy_(torch.from_numpy(part))
            else:                                           # Keras Embedding init U(-0.05, 0.05), generated on the device
                gen = torch.Generator(device=device); gen.manual_seed(int(init_seed) * 1000003 + r)
                w2.uniform_(-0.05, 0.05, generator=gen)
            tab = H.Table(w2, slots=slots, touched=False, slot_init=slot_init, g=g)
            tab.touched = t
            self.tables[r] = tab
        self.ptr_w, self.ptr_g, self.ptr_t = ptr_w, ptr_g, ptr_t

    @property
    def local(self):
        return self.tables[self.rank]

    def c_shards(self):
        s = N.brk_shards()
        for p in range(self.G):
            s.w[p], s.g[p], s.touched[p] = self.ptr_w[p], self.ptr_g[p], self.ptr_t[p]
        s.world, s.rank = self.G, self.rank
        return s

    def full_weights(self, which="w"):
        """The whole table on the host (tests): all-gather of the shards, re-interleaved.  which: "w" or an optimizer
        slot ("m", "v")."""
        if self.emulate or self.G == 1:
            parts = [getattr(self.tables[r], which).cpu().numpy() for r in range(self.G)]
        else:
            mine = getattr(self.local, which).contiguous()
            parts_t = [torch.empty_like(mine) for _ in range(self.G)]
            dist.all_gather(parts_t, mine)
            parts = [p.cpu().numpy() for p in parts_t]
        out = np.zeros((self.rows, self.d), dtype=np.float32)
        for r in range(self.G):
            n = len(range(r, self.rows, self.G))
            out[r::self.G] = parts[r][:n]
        return out


class ShardedNeuMFNet:
    """NeuMF (class spec, src/models/NeuMFModel.py:53-100) with row-sharded tables; see the module docstring."""

    def __init__(self, numUser, numItem, numFactor, act="relu", loss="mse", learning_rate=1e-3, dropout=0.0,
                 seed=42, dropout_seed=11, device=None, mode="peer", emulate=0, full_init=None, tensor_cores=False):
        from .NeuMFModel import NeuMFNet
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        self.mode = mode
        self.tensor_cores = bool(tensor_cores)
        self.emulate = int(emulate)
        if self.emulate:
            self.G, self.rank = self.emulate, 0
        else:
            self.G, self.rank = D.world_size(), D.rank()
        E = int(numFactor)
        self.E, self.hidden = E, (E, E // 2, E // 4)
        self.numUser, self.numItem = int(numUser), int(numItem)
        self.act, self.loss, self.dropout, self.dropout_seed = act, loss, float(dropout), dropout_seed
        dev, G, r = self.device, self.G, self.rank
        symmetric = (mode == "peer") and not self.emulate and G > 1
        fi = full_init or {}
        mk = lambda name, rows, k: ShardedTable(rows, E, G, r, dev, full_init=fi.get(name), init_seed=seed * 16 + k,
                                                symmetric=symmetric, emulate=bool(self.emulate))
        self.uMLP, self.iMLP = mk("uMLP", self.numUser, 0), mk("iMLP", self.numItem, 1)
        self.uMF, self.iMF = mk("uMF", self.numUser, 2), mk("iMF", self.numItem, 3)
        # dense block: identical on every rank (same seed); layout and init as NeuMFNet
        h1, h2, h3 = self.hidden
        n_dense = int(N.lib().brk_neumf_dense_floats(E, h1, h2, h3))
        npad = (n_dense + 3) // 4 * 4
        flat = fi.get("dense")
        if flat is None:
            flat = NeuMFNet.initial_dense(E, self.hidden, np.random.Generator(np.random.Philox(key=seed + 77)))
        flat = np.pad(np.asarray(flat, dtype=np.float32), (0, npad - n_dense))
        self.peer = None
        if symmetric:
            self.peer = D.PeerArena(npad, dev)
            self.peer.w.copy_(torch.from_numpy(flat))
            self.dense = H.Table(self.peer.w.view(1, -1), slots=0, touched=False, g=self.peer.g)
            import torch.distributed._symmetric_memory as symm_mem
            self._bar_flags = symm_mem.empty(64, dtype=torch.int32, device=dev)
            self._bar_h = symm_mem.rendezvous(self._bar_flags, dist.group.WORLD.group_name)
            self._bar_flags.zero_()
            self._bar_ptrs = torch.tensor(list(self._bar_h.buffer_ptrs), dtype=torch.int64, device=dev)
            self._bar_sync = torch.zeros(4, dtype=torch.int32, device=dev)
            torch.cuda.synchronize(dev)
            dist.barrier()
        else:
            self.dense = H.Table(torch.from_numpy(flat).to(dev).view(1, -1), touched=False)
        bn = np.concatenate([np.zeros(h1), np.ones(h1), np.zeros(h2), np.ones(h2)]).astype(np.float32)
        self.bn_moving = torch.from_numpy(bn).to(dev)
        self.optimizer = H.Adam(learning_rate, sparse="lazy", device=dev)
        self._ws_batch = 0
        self._net_cls = NeuMFNet

    # ---- C structs -------------------------------------------------------------------------------------
    def _tables(self):
        return [self.uMLP, self.iMLP, self.uMF, self.iMF]

    def _c_model(self, tabs=None):
        h1, h2, h3 = self.hidden
        t = tabs or [x.local for x in self._tables()]
        return N.brk_neumf_model(t[0].c_struct(), t[1].c_struct(), t[2].c_struct(), t[3].c_struct(),
                                 self.dense.c_struct(), self.bn_moving.data_ptr(), self.E, h1, h2, h3,
                                 0 if self.act == "relu" else 1, 0 if self.loss == "mse" else 1,
                                 1 if self.dropout > 0 else 0, 1 if self.tensor_cores else 0)

    def _c_shards(self):
        return N.brk_neumf_shards(*[t.c_shards() for t in self._tables()])

    def _workspace(self, batch):
        if batch > self._ws_batch:
            h1, h2, _ = self.hidden
            dev = self.device
            acc_n = int(N.lib().brk_neumf_acc_doubles(h1, h2))
            self._bufs = dict(h1=torch.empty(h1 * batch, device=dev), h2=torch.empty(h2 * batch, device=dev),
                              dy1=torch.empty(h1 * batch, device=dev), dy2=torch.empty(h2 * batch, device=dev),
                              acc=torch.zeros(acc_n, dtype=torch.float64, device=dev))
            self._ws_batch = batch
        b = self._bufs
        return N.brk_neumf_workspace(b["h1"].data_ptr(), b["h2"].data_ptr(), b["dy1"].data_ptr(), b["dy2"].data_ptr(),
                                     b["acc"].data_ptr())

    # ---- one training step on this rank's slice of the global batch --------------------------------------
    def train_on_batch(self, u, i, y, first_index=0, epoch=0, out=None, loss_out=None):
        B = u.numel()
        dev = self.device
        out = out if out is not None else torch.empty(B, dtype=torch.float32, device=dev)
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=dev)
        gb = B * self.G if (self.G > 1 and not self.emulate) else 0
        if self.mode == "peer":
            self._step_peer(u, i, y, B, gb, first_index, epoch, out, loss_out)
        else:
            self._step_nccl(u, i, y, B, gb, first_index, epoch, out, loss_out)
        return loss_out, out

    def _step_peer(self, u, i, y, B, gb, first_index, epoch, out, loss_out):
        lib, ctx, st = N.lib(), N.ctx(self.device), N.stream_ptr()
        m, sh, ws = self._c_model(), self._c_shards(), self._workspace(B)
        N.check(lib.brk_neumf_step_sharded(ctx, C.byref(m), C.byref(sh), N.ptr(H._i32(u, "u")), N.ptr(H._i32(i, "i")),
                                           N.ptr(H._f32(y, "y")), B, gb, first_index, 1, self.dropout_seed & 0xFFFFFFFF,
                                           epoch & 0xFFFFFFFF, C.byref(ws), N.ptr(out), N.ptr(loss_out), st),
                "brk_neumf_step_sharded")
        if self.emulate:                                      # all G owners' optimizer passes, in this one process
            tabs = [t.tables[r] for r in range(self.G) for t in self._tables()]
            h, state = self.optimizer.h, N.ptr(self.optimizer.state)
            N.check(lib.brk_adam_dense_keras(ctx, H._pack([self.dense]), 1, h, state, 0, st), "brk_adam_dense_keras")
            for k in range(0, len(tabs), 16):
                chunk = tabs[k:k + 16]
                N.check(lib.brk_adam_rows(ctx, H._pack(chunk), len(chunk), h, state, 1 if k + 16 >= len(tabs) else 0, st),
                        "brk_adam_rows")
            return
        if self.peer is None:                                # G == 1
            self.optimizer.apply([t.local for t in self._tables()], dense=[self.dense])
            return
        # every rank's REDs have landed in my accumulators once all ranks passed the barrier
        N.check(lib.brk_peer_barrier(ctx, N.ptr(self._bar_ptrs), N.ptr(self._bar_sync), self.rank, self.G, st),
                "brk_peer_barrier")
        tabs = [t.local for t in self._tables()]
        N.check(lib.brk_adam_rows(ctx, H._pack(tabs), len(tabs), self.optimizer.h, N.ptr(self.optimizer.state), 0, st),
                "brk_adam_rows")
        # dense block: fused reduce-scatter + Adam + all-gather; its barriers also order the shard updates of
        # all ranks before anybody's next gather, and it advances the shared step counter
        self.peer.adam_step(self.optimizer.h, self.optimizer.state)

    def _step_nccl(self, u, i, y, B, gb, first_index, epoch, out, loss_out):
        """Baseline: explicit all-to-all exchange of ids, rows and row gradients around the same kernels."""
        lib, ctx, st = N.lib(), N.ctx(self.device), N.stream_ptr()
        G, dev, E = self.G, self.device, self.E
        ident = torch.arange(B, dtype=torch.int32, device=dev)
        lu, li = D.ShardedLookup(u, G), D.ShardedLookup(i, G)
        tmp = []
        for tab, lk in ((self.uMLP, lu), (self.iMLP, li), (self.uMF, lu), (self.iMF, li)):
            rows = lk.forward(lambda ids, w=tab.local.w: H.gather_rows(w, ids.to(torch.int32)))
            tmp.append(H.Table(rows, slots=0, touched=False))
        m, ws = self._c_model(tmp), self._workspace(B)
        N.check(lib.brk_neumf_step(ctx, C.byref(m), N.ptr(ident), N.ptr(ident), N.ptr(H._f32(y, "y")), B, gb, first_index,
                                   1, self.dropout_seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, C.byref(ws), N.ptr(out),
                                   N.ptr(loss_out), st), "brk_neumf_step")
        for tab, lk, t in zip(self._tables(), (lu, li, lu, li), tmp):
            lk.backward(t.g, lambda ids, vals, T=tab.local: H.scatter_add_rows(T.g, ids.to(torch.int32), vals.contiguous(),
                                                                              T.touched))
        if G > 1:
            D.all_reduce_sum_(self.dense.g)
        self.optimizer.apply([t.local for t in self._tables()], dense=[self.dense])

    def check(self):
        if self.peer is not None:
            self.peer.check()
            if int(self._bar_sync[1].item()) != 0:
                raise RuntimeError("brk_peer_barrier timed out (a rank did not reach the step)")


    # ---- checkpoint (SURVEY.md section 8 row f3) -----------------------------------------------------------
    def _dense_slots(self):
        """(m, v) of the dense block as full-length host arrays: local slots, or -- in peer mode, where every rank
        keeps the Adam moments of its own slice only (distributed.PeerArena) -- the slices summed over ranks."""
        n = self.dense.w.numel()
        if self.peer is None:
            return self.dense.m.view(-1).cpu().numpy(), self.dense.v.view(-1).cpu().numpy()
        out = []
        for part in (self.peer.m, self.peer.v):
            full = torch.zeros(n, dtype=torch.float32, device=self.device)
            lo, hi = self.peer.slice_lo, self.peer.slice_hi
            full[lo:hi] = part[:hi - lo]
            dist.all_reduce(full)
            out.append(full.cpu().numpy())
        return tuple(out)

    def save_checkpoint(self, dirpath):
        m, v = self._dense_slots()
        rep = {"dense": self.dense.w.view(-1), "dense_m": m, "dense_v": v, "bn_moving": self.bn_moving,
               "opt_state": self.optimizer.state}
        tabs = dict(zip(("uMLP", "iMLP", "uMF", "iMF"), self._tables()))
        return save_sharded_model(dirpath, tabs, rep, self.G, self.rank, self.emulate,
                                  meta={"model": "ShardedNeuMFNet", "E": self.E, "numUser": self.numUser,
                                        "numItem": self.numItem, "act": self.act, "loss": self.loss})

    def load_checkpoint(self, dirpath):
        tabs = dict(zip(("uMLP", "iMLP", "uMF", "iMF"), self._tables()))
        rep, meta = load_sharded_model(dirpath, tabs, self.G, self.rank, self.emulate)
        n = self.dense.w.numel()
        self.dense.w.view(-1).copy_(torch.from_numpy(rep["dense"][:n]))
        m, v = torch.from_numpy(rep["dense_m"][:n]).to(self.device), torch.from_numpy(rep["dense_v"][:n]).to(self.device)
        if self.peer is None:
            self.dense.m.view(-1).copy_(m); self.dense.v.view(-1).copy_(v)
        else:
            lo, hi = self.peer.slice_lo, self.peer.slice_hi
            self.peer.m[:hi - lo].copy_(m[lo:hi]); self.peer.v[:hi - lo].copy_(v[lo:hi])
            torch.cuda.synchronize(self.device)
            dist.barrier()
        self.bn_moving.copy_(torch.from_numpy(rep["bn_moving"]))
        self.optimizer.state.copy_(torch.from_numpy(rep["opt_state"]))
        return meta


class PeerBarrier:
    """brk_peer_barrier with its symmetric flag block (one instance per model)."""

    def __init__(self, device):
        import torch.distributed._symmetric_memory as symm_mem
        self.device = device
        self.flags = symm_mem.empty(64, dtype=torch.int32, device=device)
        self._h = symm_mem.rendezvous(self.flags, dist.group.WORLD.group_name)
        self.flags.zero_()
        self.ptrs = torch.tensor(list(self._h.buffer_ptrs), dtype=torch.int64, device=device)
        self.sync = torch.zeros(4, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier()

    def __call__(self):
        N.check(N.lib().brk_peer_barrier(N.ctx(self.device), N.ptr(self.ptrs), N.ptr(self.sync), D.rank(), D.world_size(),
                                         N.stream_ptr()), "brk_peer_barrier")

    def check(self):
        if int(self.sync[1].item()) != 0:
            raise RuntimeError("brk_peer_barrier timed out (a rank did not reach the step)")


class ShardedBPRNet:
    """BPR matrix factorisation (src/models/BPRModel.py:49-74,124-144) with row-sharded user / item tables and
    row-sparse (lazy) Adam: fused fwd/bwd over peer memory -> barrier -> every owner updates its shards -> barrier."""

    def __init__(self, numUser, numItem, numFactor, learning_rate=1e-3, seed=42, device=None, emulate=0, full_init=None):
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        self.emulate = int(emulate)
        self.G, self.rank = (self.emulate, 0) if self.emulate else (D.world_size(), D.rank())
        self.d = int(numFactor)
        symmetric = not self.emulate and self.G > 1
        fi = full_init or {}
        self.user = ShardedTable(numUser, self.d, self.G, self.rank, self.device, full_init=fi.get("user"), init_seed=seed * 16,
                                 symmetric=symmetric, emulate=bool(self.emulate))
        self.item = ShardedTable(numItem, self.d, self.G, self.rank, self.device, full_init=fi.get("item"), init_seed=seed * 16 + 1,
                                 symmetric=symmetric, emulate=bool(self.emulate))
        self.optimizer = H.Adam(learning_rate, sparse="lazy", device=self.device)
        self.barrier = PeerBarrier(self.device) if symmetric else None

    def train_on_batch(self, u, p, n, loss_out=None):
        B = u.numel()
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
        us, it = self.user.c_shards(), self.item.c_shards()
        gb = B * self.G if (self.G > 1 and not self.emulate) else 0
        N.check(N.lib().brk_bpr_fwd_bwd_sharded(N.ctx(self.device), C.byref(us), C.byref(it), self.d, N.ptr(H._i32(u, "u")),
                                                N.ptr(H._i32(p, "p")), N.ptr(H._i32(n, "n")), B, gb, N.ptr(loss_out),
                                                N.stream_ptr()), "brk_bpr_fwd_bwd_sharded")
        if self.emulate:
            self.optimizer.apply([t.tables[r] for r in range(self.G) for t in (self.user, self.item)])
            return loss_out
        if self.barrier is not None:
            self.barrier()                     # every rank's REDs have landed in my accumulators
        self.optimizer.apply([self.user.local, self.item.local])
        if self.barrier is not None:
            self.barrier()                     # every owner has updated its shards before anybody's next gather
        return loss_out

    def check(self):
        if self.barrier is not None:
            self.barrier.check()

    def save_checkpoint(self, dirpath):
        return save_sharded_model(dirpath, {"user": self.user, "item": self.item}, {"opt_state": self.optimizer.state},
                                  self.G, self.rank, self.emulate, meta={"model": "ShardedBPRNet", "d": self.d})

    def load_checkpoint(self, dirpath):
        rep, meta = load_sharded_model(dirpath, {"user": self.user, "item": self.item}, self.G, self.rank, self.emulate)
        self.optimizer.state.copy_(torch.from_numpy(rep["opt_state"]))
        return meta


class ShardedTwoTowerNet:
    """Two-tower retrieval model (twoTower.TwoTowerModel: Embedding -> linear Dense(semb) per tower, in-batch softmax or
    rdZero BCE, Keras Adagrad) with row-sharded embedding tables, for catalogs too large to mirror on every GPU.

    Semantics, per step on a global batch split over the G ranks (D.local_slice):
      * every rank trains its slice; the in-batch softmax uses that slice's items as negatives (MirroredStrategy's
        per-replica loss, what the mirrored TwoTowerModel.fit does); accidental hits compare global item ids within
        the slice;
      * each replica's loss is SUM-reduced; gradients are summed over ranks, never scaled;
      * row r of a table (numUser + 2 / numItem + 2 rows: the StringLookup offset) lives on rank r % G at local row
        r // G; a rank's row gradients land in the owner's accumulator as REDs and set the owner's touched bits;
      * every owner applies row-sparse Keras Adagrad (accumulator initial value 0.1, in `m`) to the touched rows of its
        shards.  Adagrad leaves rows with g = 0 unchanged, so this is the mirrored dense pass up to summation order;
      * the two Dense blocks (W [E][S], then b [S]) are mirrored; their gradients are summed over ranks by
        brk_allreduce_dense_peer (fixed order: bit-identical replicas) and every replica applies brk_adagrad_dense.
    So G GPUs give the mirrored TwoTowerModel's result on the same global batches.  `emulate=G` holds all G shards in
    one process on one GPU and trains the whole batch as one replica: the unsharded single-GPU TwoTowerModel's result.

    Ids arrive as int32 table rows (already looked up).  full_init: {"user", "item": full tables [rows, E];
    "user_dense", "item_dense": flat Dense blocks as Tower.init_dense lays them out}; without it the tables are
    U(-0.05, 0.05) and the Dense blocks Glorot-uniform from Philox(seed + 77)."""

    def __init__(self, numUser, numItem, embedDim, semb, learning_rate=0.1, rdZero=False, tensor_cores=True, seed=42,
                 device=None, emulate=0, full_init=None):
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        self.emulate = int(emulate)
        self.G, self.rank = (self.emulate, 0) if self.emulate else (D.world_size(), D.rank())
        self.embedDim, self.semb = int(embedDim), int(semb)
        self.numUser, self.numItem = int(numUser), int(numItem)
        self.rdZero, self.tensor_cores = bool(rdZero), bool(tensor_cores)
        self.optimizer = H.Adagrad(learning_rate)
        dev, E, S = self.device, self.embedDim, self.semb
        symmetric = not self.emulate and self.G > 1
        fi = full_init or {}
        mk = lambda name, rows, k: ShardedTable(rows, E, self.G, self.rank, dev, full_init=fi.get(name), init_seed=seed * 16 + k,
                                                symmetric=symmetric, emulate=bool(self.emulate), slots=1,
                                                slot_init=H.Adagrad.INITIAL_ACCUMULATOR)
        self.user, self.item = mk("user", self.numUser + 2, 0), mk("item", self.numItem + 2, 1)
        rng = np.random.Generator(np.random.Philox(key=seed + 77))
        self.dense = []
        for name in ("user_dense", "item_dense"):
            t = Tower.__new__(Tower)
            t.E, t.S = E, S
            t.init_dense(rng, dev)
            if name in fi:
                t.dense.w.view(-1).copy_(torch.from_numpy(np.asarray(fi[name], dtype=np.float32).reshape(-1)))
            self.dense.append(t.dense)
        # the Dense gradients are views of ONE flat arena, summed over the ranks once per step (peer memory, no NCCL)
        self.grad_arena = self._reducer = None
        self.barrier = None
        if symmetric:
            sizes = [t.w.numel() for t in self.dense]
            self.grad_arena, self._reducer = D.gradient_arena(sum(sizes), dev)
            for t, v in zip(self.dense, torch.split(self.grad_arena[:sum(sizes)], sizes)):
                t.g = v.view(t.rows, t.d)
            self.barrier = PeerBarrier(dev)
        self._ws_batch = 0

    _workspace = TwoTowerModel._workspace               # the mirrored model's step buffers (same attribute names)

    def _towers(self):
        return [N.brk_tower(N.brk_table(), d.c_struct(), self.embedDim, self.semb) for d in self.dense]

    def _shards(self):
        return N.brk_twotower_shards(self.user.c_shards(), self.item.c_shards())

    def train_on_batch(self, u, i, labels=None, loss_out=None):
        """One step on this rank's slice (u, i: int32 table rows; labels: rdZero targets).  Every rank must call it, an
        empty slice included.  Returns the slice's loss as a device scalar."""
        loss_out = self.forward_backward(u, i, labels, loss_out)
        self.apply_gradients()
        return loss_out

    def forward_backward(self, u, i, labels=None, loss_out=None):
        """The step without the optimizer: row gradients in the owners' accumulators (touched bits set there), Dense
        gradients in this rank's Dense blocks."""
        B = u.numel()
        dev = self.device
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=dev)
        lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()
        if B > 0:
            if self.rdZero and labels is None:
                raise ValueError("rdZero training needs labels")
            ws = self._workspace(B)
            ut, it = self._towers()
            sh = self._shards()
            u, i = H._i32(u, "u"), H._i32(i, "i")
            N.check(lib.brk_twotower_step_sharded(ctx, C.byref(ut), C.byref(it), C.byref(sh), N.ptr(u), N.ptr(i), N.ptr(i),
                                                  N.ptr(H._f32(labels, "labels")) if self.rdZero else None, B,
                                                  (1 if self.rdZero else 0) | (0x100 if self.tensor_cores else 0),
                                                  C.byref(ws), N.ptr(loss_out), st), "brk_twotower_step_sharded")
        else:
            loss_out.zero_()
        return loss_out

    def apply_gradients(self):
        """Row-sparse Adagrad on the owned shards, Dense gradients summed over ranks, Adagrad on the Dense blocks."""
        lib, ctx, st = N.lib(), N.ctx(self.device), N.stream_ptr()
        opt = self.optimizer
        if self.barrier is None:                            # every shard lives in this process (emulation, or G == 1)
            tabs = [t.tables[r] for t in (self.user, self.item) for r in range(self.G)]
            for k in range(0, len(tabs), 16):
                N.check(lib.brk_adagrad_rows(ctx, H._pack(tabs[k:k + 16]), len(tabs[k:k + 16]), opt.lr, opt.eps, st),
                        "brk_adagrad_rows")
            N.check(lib.brk_adagrad_dense(ctx, H._pack(self.dense), 2, opt.lr, opt.eps, st), "brk_adagrad_dense")
            return
        self.barrier()                                      # every rank's REDs have landed in my shards
        mine = [self.user.local, self.item.local]
        N.check(lib.brk_adagrad_rows(ctx, H._pack(mine), 2, opt.lr, opt.eps, st), "brk_adagrad_rows")
        # The all-reduce also fences the next step: its entry barrier is reached by a rank only after that rank's row
        # pass above (stream order), and nobody leaves the all-reduce before every rank has reached it.  So no rank
        # gathers rows of the next step before every owner has updated its shards and zeroed their accumulators.
        D.all_reduce_sum_(self.grad_arena, self._reducer)
        N.check(lib.brk_adagrad_dense(ctx, H._pack(self.dense), 2, opt.lr, opt.eps, st), "brk_adagrad_dense")

    def check(self):
        """Raises when a cross-GPU barrier or the Dense all-reduce timed out (call at epoch ends, not per step)."""
        if self.barrier is not None:
            self.barrier.check()
        if self._reducer is not None:
            self._reducer.check()

    def _tower_forward(self, k, ids):
        ids = H._i32(ids, "ids")
        n = ids.numel()
        emb = torch.empty(n, self.embedDim, dtype=torch.float32, device=self.device)
        out = torch.empty(n, self.semb, dtype=torch.float32, device=self.device)
        if n == 0:
            return out
        t, sh = self._towers()[k], (self.user, self.item)[k].c_shards()
        N.check(N.lib().brk_tower_forward_sharded(N.ctx(self.device), C.byref(t), C.byref(sh), N.ptr(ids), n, N.ptr(emb),
                                                  N.ptr(out), N.stream_ptr()), "brk_tower_forward_sharded")
        return out

    def score_vectors(self, user_rows, item_rows):
        """(user vectors [n, S], item vectors [m, S]) of int32 table rows, for hotpath.BruteForceIndex / topKmetrics."""
        return self._tower_forward(0, user_rows), self._tower_forward(1, item_rows)

    # ---- checkpoint: shards of the tables and their accumulators, replicated Dense blocks and theirs ------------
    def save_checkpoint(self, dirpath):
        rep = {}
        for name, t in zip(("user_dense", "item_dense"), self.dense):
            rep[name], rep[name + "_m"] = t.w.view(-1), t.m.view(-1)
        return save_sharded_model(dirpath, {"user": self.user, "item": self.item}, rep, self.G, self.rank, self.emulate,
                                  meta={"model": "ShardedTwoTowerNet", "E": self.embedDim, "S": self.semb,
                                        "numUser": self.numUser, "numItem": self.numItem})

    def load_checkpoint(self, dirpath):
        rep, meta = load_sharded_model(dirpath, {"user": self.user, "item": self.item}, self.G, self.rank, self.emulate)
        for name, t in zip(("user_dense", "item_dense"), self.dense):
            t.w.view(-1).copy_(torch.from_numpy(rep[name]))
            t.m.view(-1).copy_(torch.from_numpy(rep[name + "_m"]))
        return meta
