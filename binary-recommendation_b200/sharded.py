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
from .NeuMFModel import NeuMFTopKIndex, NeuMFTopKIndexFP32
from .twoTower import (GlobalNegatives, SampledNegatives, Tower, TwoTowerModel, check_retrieval_options,
                       check_sampled_options)


def shard_rows(rows, G):
    """Rows per shard (equal on every rank, as symmetric memory needs)."""
    return (rows + G - 1) // G


def save_sharded_model(dirpath, tables, replicated, G, rank, emulate, meta=None, extra=None):
    """Checkpoint of a row-sharded model (checkpoint.py; SURVEY.md section 8 row f3): every rank writes its shards of
    the weights and optimizer slots, rank 0 the replicated tensors and -- after a barrier -- the manifest.
    tables: {name: ShardedTable}; extra: {name: (shard(r) -> rank r's [local_rows, d] tensor, global rows)}, other
    row-sharded state."""
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
        for name, (shard, rows) in (extra or {}).items():
            shd[name] = (shard(r), rows)
        CK.save_checkpoint(dirpath, replicated=replicated if r == 0 else None, sharded=shd, rank=r, world=G,
                           meta=meta, barrier=barrier)
    return dirpath


def load_sharded_model(dirpath, tables, G, rank, emulate, extra=None):
    """Restores the shards this process owns -- whatever world size wrote the checkpoint.  Returns (replicated, meta).
    extra: {name: shard(r) -> rank r's tensor}, restored where the checkpoint has the entry and zeroed where not."""
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
        for name, shard in (extra or {}).items():
            if name in shd:
                shard(r).copy_(torch.from_numpy(shd[name]))
            else:
                shard(r).zero_()
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

    # the reference class graph: NeuMFNet's attributes of the same names (the top-k indexes read them)
    variant, mf_mode, batch_norm = False, "dot", True

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
        self.EMF = E
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

    def param(self, name):
        """View of the dense block's parameter `name` (NeuMFNet.DENSE_ORDER, NeuMFNet's layout)."""
        E, (h1, h2, h3) = self.E, self.hidden
        shapes = dict(W1=(2 * E, h1), b1=(h1,), g1=(h1,), be1=(h1,), W2=(h1, h2), b2=(h2,), g2=(h2,), be2=(h2,),
                      W3=(h2, h3), b3=(h3,), W4=(h3 + 1, 1), b4=(1,))
        off = 0
        for key in self._net_cls.DENSE_ORDER:
            n = int(np.prod(shapes[key]))
            if key == name:
                return self.dense.w.view(-1)[off:off + n].view(*shapes[key])
            off += n
        raise KeyError(name)

    def _gather_rows(self, names, ids):
        """Rows `ids` (global row ids, int32 on this device) of the tables `names`: peer loads from the owners' shards, or
        in mode "nccl" the all-to-all of distributed.ShardedLookup (collective: every rank calls it)."""
        tabs = [getattr(self, n) for n in names]
        if self.mode == "peer" or self.emulate or self.G == 1:
            return [_gather_rows_sharded(t, ids) for t in tabs]
        lk = D.ShardedLookup(ids, self.G)
        gather = lambda w: (lambda x: H.gather_rows(w, x.to(torch.int32)) if x.numel() else w.new_empty((0, self.E)))
        return [lk.forward(gather(t.local.w)) for t in tabs]

    # ---- full-catalog top-k (collective: every rank calls with the same arguments) ---------------------------------
    def topk_index(self, itemsId=None):
        """Top-k index of a tensor-core model (tensor_cores=True) over itemsId (default: every item): see
        ShardedTopKIndex.  Per query 1 <= k <= 32; the lists equal NeuMFNet.topk_index's over the full tables."""
        if not self.tensor_cores:
            raise ValueError("the model computes in fp32 (tensor_cores=False): rank it with ShardedNeuMFNet.topk_index_fp32")
        return ShardedNeuMFTopKIndex(self, itemsId, NeuMFTopKIndex)

    def topk_index_fp32(self, itemsId=None):
        """Top-k index of an fp32 model (tensor_cores=False) over itemsId: see ShardedTopKIndex.  The lists equal
        NeuMFNet.topk_index_fp32's over the full tables."""
        if self.tensor_cores:
            raise ValueError("the model computes with TF32 tensor-core products (tensor_cores=True): rank it with "
                             "ShardedNeuMFNet.topk_index")
        return ShardedNeuMFTopKIndex(self, itemsId, NeuMFTopKIndexFP32)

    def score_all(self, usersId, itemsId, k, exclude=None):
        """(scores [U, k], positions in itemsId [U, k]) for topKRatings: a one-off top-k index over itemsId.  `exclude`:
        an (indptr, ids) CSR of positions per user (hotpath.exclusion_csr).  Collective."""
        index = self.topk_index(itemsId) if self.tensor_cores else self.topk_index_fp32(itemsId)
        return index(usersId, k) if exclude is None else index.query_with_exclusions(usersId, exclude, k)

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

    def topk_index(self, itemsId=None, k=10):
        """Top-k index over itemsId (default: every item) by the dot product of user and item rows: see ShardedTopKIndex.
        The lists equal BruteForceIndex(k).index(item_w[itemsId])(user_w[usersId]) over the full tables; k up to
        hotpath.fused_k_cap of the row width."""
        return ShardedDotTopKIndex(self, itemsId, k, lambda which, ids: _gather_rows_sharded((self.user, self.item)[which], ids),
                                   self.d, self.item.rows)

    def score_all(self, usersId, itemsId, k, exclude=None):
        """(scores [U, k], positions in itemsId [U, k]) for topKRatings: a one-off top-k index over itemsId.  `exclude`:
        an (indptr, ids) CSR of positions per user (hotpath.exclusion_csr).  Collective."""
        index = self.topk_index(itemsId, k)
        return index(usersId, k) if exclude is None else index.query_with_exclusions(usersId, exclude, k)

    def save_checkpoint(self, dirpath):
        return save_sharded_model(dirpath, {"user": self.user, "item": self.item}, {"opt_state": self.optimizer.state},
                                  self.G, self.rank, self.emulate, meta={"model": "ShardedBPRNet", "d": self.d})

    def load_checkpoint(self, dirpath):
        rep, meta = load_sharded_model(dirpath, {"user": self.user, "item": self.item}, self.G, self.rank, self.emulate)
        self.optimizer.state.copy_(torch.from_numpy(rep["opt_state"]))
        return meta


class ShardedEstimator:
    """The streaming frequency estimator of Yi et al. (brk_tt_retrieval's, one slot per item-table row) with its state
    sharded like the item table: last (int64) and gap (fp32) of row y live on rank y % G at local row y // G, in
    symmetric memory on real ranks and as G local arrays under emulation (as ShardedTable).  `step` is this process's
    training-step counter, equal on every rank."""

    def __init__(self, rows, G, rank, device, alpha, symmetric, emulate):
        self.rows, self.G, self.rank, self.device, self.alpha = int(rows), int(G), int(rank), device, float(alpha)
        self.local_rows = shard_rows(rows, G)
        self.emulate = emulate
        self.last, self.gap, self._keep = {}, {}, []
        ptr_l, ptr_g = [0] * G, [0] * G
        for r in (range(G) if emulate else [rank]):
            if symmetric and not emulate:
                import torch.distributed._symmetric_memory as symm_mem
                group = dist.group.WORLD.group_name
                last = symm_mem.empty(self.local_rows, dtype=torch.int64, device=device)
                gap = symm_mem.empty(self.local_rows, dtype=torch.float32, device=device)
                hs = [symm_mem.rendezvous(x, group) for x in (last, gap)]
                self._keep.append(hs)
                ptr_l, ptr_g = (list(h.buffer_ptrs) for h in hs)
            else:
                last = torch.empty(self.local_rows, dtype=torch.int64, device=device)
                gap = torch.empty(self.local_rows, dtype=torch.float32, device=device)
                ptr_l[r], ptr_g[r] = last.data_ptr(), gap.data_ptr()
            last.zero_(); gap.zero_()
            self.last[r], self.gap[r] = last, gap
        self.step = torch.zeros(1, dtype=torch.int64, device=device)
        self.c = N.brk_tt_estimator_sharded()
        for p in range(G):
            self.c.last[p], self.c.gap[p] = ptr_l[p], ptr_g[p]
        self.c.rows, self.c.world, self.c.rank = self.local_rows, G, self.rank

    def update(self, ids):
        """The training-step update for this rank's slice `ids` (int32 item rows; may be empty)."""
        N.check(N.lib().brk_tt_estimator_update_sharded(N.ctx(self.device), C.byref(self.c), N.ptr(ids) if ids.numel() else None,
                                                         ids.numel(), self.alpha, N.ptr(self.step), N.stream_ptr()),
                "brk_tt_estimator_update_sharded")

    def state(self):
        """(last [rows] int64, gap [rows] float32, step) of the whole table on the host; collective on real ranks."""
        if self.emulate or self.G == 1:
            parts = [(self.last[r].cpu().numpy(), self.gap[r].cpu().numpy()) for r in range(self.G)]
        else:
            gathered = []
            for mine in (self.last[self.rank], self.gap[self.rank]):
                ts = [torch.empty_like(mine) for _ in range(self.G)]
                dist.all_gather(ts, mine)
                gathered.append([t.cpu().numpy() for t in ts])
            parts = list(zip(*gathered))
        last, gap = np.zeros(self.rows, np.int64), np.zeros(self.rows, np.float32)
        for r, (lr, gr) in enumerate(parts):
            n = len(range(r, self.rows, self.G))
            last[r::self.G], gap[r::self.G] = lr[:n], gr[:n]
        return last, gap, int(self.step.item())


class ShardedTwoTowerNet:
    """Two-tower retrieval model (twoTower.TwoTowerModel: Embedding -> linear Dense(semb) per tower, in-batch softmax or
    rdZero BCE, Keras Adagrad) with row-sharded embedding tables, for catalogs too large to mirror on every GPU.

    Semantics, per step on a global batch split over the G ranks (D.local_slice):
      * every rank trains its slice; the in-batch softmax uses that slice's items as negatives (MirroredStrategy's
        per-replica loss, what the mirrored TwoTowerModel.fit does); accidental hits compare global item ids within
        the slice.  With global_negatives=True every rank's queries are scored against the items of the whole global
        batch instead (GlobalNegatives, brk_twotower_step_global): the label of global row o is column o, accidental
        hits are masked across slices, and the ranks' losses sum to the one-GPU loss of the global batch;
      * each replica's loss is SUM-reduced; gradients are summed over ranks, never scaled;
      * row r of a table (numUser + 2 / numItem + 2 rows: the StringLookup offset) lives on rank r % G at local row
        r // G; a rank's row gradients land in the owner's accumulator as REDs and set the owner's touched bits;
      * every owner applies row-sparse Keras Adagrad (accumulator initial value 0.1, in `m`) to the touched rows of its
        shards.  Adagrad leaves rows with g = 0 unchanged, so this is the mirrored dense pass up to summation order;
      * the two Dense blocks (W [E][S], then b [S]) are mirrored; their gradients are summed over ranks by
        brk_allreduce_dense_peer (fixed order: bit-identical replicas) and every replica applies brk_adagrad_dense.
    So G GPUs give the mirrored TwoTowerModel's result on the same global batches.  `emulate=G` holds all G shards in
    one process on one GPU and trains the whole batch as one replica: the unsharded single-GPU TwoTowerModel's result.
    With global_negatives=True, `emulate=G` splits each batch with local_slice over the G emulated ranks and runs the
    three phases of brk_twotower_step_global rank by rank; with one rank (G = 1) the flag changes nothing.

    tfrs Retrieval's sampling-bias correction (brk_twotower_step_sharded_retrieval), per replica as the softmax above:
    temperature=tau, per-call candidate sampling probabilities `cand_prob` and sample weights `weights` ([b] float32 device
    tensors of this rank's slice; under emulation of the whole batch), or streamingFrequency=alpha (True: 0.01): the
    streaming frequency estimator (ShardedEstimator) updated on the GLOBAL batch -- every rank updates the rows of its
    slice, a cross-GPU barrier, then every replica's step reads p_y = 1 / gap[y] at the owner -- so its state equals the
    single-process estimator's on the global batch bit for bit.  Not offered with rdZero or global_negatives.

    sampledNegatives=M (brk_twotower_step_sharded_sampled): every training step draws M item rows uniformly from
    [2, numItem + 2) and adds them as candidate columns of every row of the replica's slice, with temperature and weights
    as above.  Each replica draws its own rows (Philox keyed by (seed, rank); rank 0 under emulation and at G = 1, so
    `emulate=G` gives TwoTowerModel(sampledNegatives=M)'s result); the sampled rows are gathered from and their gradients
    sent to their owners like the batch's.  The sampler's step counter is checkpointed as a replicated entry.  Not
    offered with rdZero, global_negatives, cand_prob or streamingFrequency.

    Ids arrive as int32 table rows (already looked up).  full_init: {"user", "item": full tables [rows, E];
    "user_dense", "item_dense": flat Dense blocks as Tower.init_dense lays them out}; without it the tables are
    U(-0.05, 0.05) and the Dense blocks Glorot-uniform from Philox(seed + 77)."""

    def __init__(self, numUser, numItem, embedDim, semb, learning_rate=0.1, rdZero=False, tensor_cores=True, seed=42,
                 device=None, emulate=0, full_init=None, global_negatives=False, temperature=None, streamingFrequency=None,
                 sampledNegatives=None):
        self.sampledNegatives = check_sampled_options(sampledNegatives, rdZero, global_negatives, streamingFrequency, False)
        if global_negatives and rdZero:
            raise ValueError("global_negatives needs the in-batch softmax: rdZero has no in-batch negatives")
        if streamingFrequency is False:
            streamingFrequency = None
        self.temperature, self.streamingFrequency = temperature, streamingFrequency
        self._retrieval = temperature is not None or streamingFrequency is not None
        alpha = check_retrieval_options(rdZero, global_negatives, temperature, streamingFrequency, False) \
            if self._retrieval else None
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        self.emulate = int(emulate)
        self.G, self.rank = (self.emulate, 0) if self.emulate else (D.world_size(), D.rank())
        self.global_negatives = bool(global_negatives)
        self.embedDim, self.semb = int(embedDim), int(semb)
        self.numUser, self.numItem = int(numUser), int(numItem)
        self.rdZero, self.tensor_cores = bool(rdZero), bool(tensor_cores)
        self.optimizer = H.Adagrad(learning_rate)
        dev, E, S = self.device, self.embedDim, self.semb
        symmetric = not self.emulate and self.G > 1
        fi = full_init or {}
        # before the peer barrier below: its set-up barrier fences the zeroed estimator shards too
        self._est = ShardedEstimator(self.numItem + 2, self.G, self.rank, dev, alpha, symmetric, bool(self.emulate)) \
            if alpha is not None else None
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
        self._global = GlobalNegatives(self.G, self.rank, E, S, dev, emulate=bool(self.emulate), barrier=self.barrier) \
            if self.global_negatives and self.G > 1 else None
        self._smp = SampledNegatives(self.sampledNegatives, self.numItem + 2, seed, self.rank, dev) \
            if self.sampledNegatives else None
        self._ws_batch = 0

    _workspace = TwoTowerModel._workspace               # the mirrored model's step buffers (same attribute names)

    def _towers(self):
        return [N.brk_tower(N.brk_table(), d.c_struct(), self.embedDim, self.semb) for d in self.dense]

    def _shards(self):
        return N.brk_twotower_shards(self.user.c_shards(), self.item.c_shards())

    def train_on_batch(self, u, i, labels=None, loss_out=None, split=None, cand_prob=None, weights=None):
        """One step on this rank's slice (u, i: int32 table rows; labels: rdZero targets).  Every rank must call it, an
        empty slice included.  Returns the slice's loss as a device scalar.  With global_negatives on real ranks, `split`
        lists the slice sizes of all G ranks (default: every slice has this one's size); under emulation u, i are the
        global batch and the loss is the sum over the emulated ranks.  cand_prob / weights: the slice's candidate
        sampling probabilities and sample weights (see the class docstring)."""
        loss_out = self.forward_backward(u, i, labels, loss_out, split, cand_prob, weights)
        self.apply_gradients()
        return loss_out

    def _rt(self, B, cand_prob, weights):
        """brk_tt_retrieval_sharded of one step, or None without any option (the option-free step)."""
        if not self._retrieval and cand_prob is None and weights is None:
            return None
        check_sampled_options(self.sampledNegatives or None, self.rdZero, self.global_negatives, self.streamingFrequency,
                              cand_prob is not None)
        check_retrieval_options(self.rdZero, self.global_negatives, None, self.streamingFrequency, cand_prob is not None)
        cols = []
        for name, v in (("cand_prob", cand_prob), ("weights", weights)):
            if v is not None and v.numel() != B:
                raise ValueError(f"{name} has {v.numel()} entries, the slice {B}")
            cols.append(H._f32(v, name) if v is not None else None)
        rt = N.brk_tt_retrieval_sharded()
        rt.cand_prob, rt.row_weight = (N.ptr(v).value if v is not None and B > 0 else None for v in cols)
        rt._cols = cols                                     # alive as long as the struct
        rt.inv_temperature = 1.0 / float(self.temperature) if self.temperature is not None else 1.0
        if self._est is not None:
            rt.est = C.pointer(self._est.c)
        return rt

    def forward_backward(self, u, i, labels=None, loss_out=None, split=None, cand_prob=None, weights=None):
        """The step without the optimizer: row gradients in the owners' accumulators (touched bits set there), Dense
        gradients in this rank's Dense blocks.  With the estimator, every rank's update of the global batch, then a
        cross-GPU barrier, comes first."""
        B = u.numel()
        dev = self.device
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=dev)
        lib, ctx, st = N.lib(), N.ctx(dev), N.stream_ptr()
        rt = self._rt(B, cand_prob, weights)
        if self._smp is not None:                           # every rank draws, an empty slice included
            u, i = H._i32(u, "u"), H._i32(i, "i")
            ws = self._workspace(max(B, 1))
            ut, it = self._towers()
            sh = self._shards()
            smp = self._smp.c_struct()
            N.check(lib.brk_twotower_step_sharded_sampled(ctx, C.byref(ut), C.byref(it), C.byref(sh), N.ptr(u), N.ptr(i), B,
                                                          0x100 if self.tensor_cores else 0, C.byref(ws), N.ptr(loss_out), st,
                                                          C.byref(smp), C.byref(rt) if rt is not None else None),
                    "brk_twotower_step_sharded_sampled")
        elif rt is not None:
            u, i = H._i32(u, "u"), H._i32(i, "i")
            if self._est is not None:
                self._est.update(i)
                if self.barrier is not None:
                    self.barrier()                          # every rank's update has landed before any step reads gap
            if B > 0:
                ws = self._workspace(B)
                ut, it = self._towers()
                sh = self._shards()
                N.check(lib.brk_twotower_step_sharded_retrieval(ctx, C.byref(ut), C.byref(it), C.byref(sh), N.ptr(u), N.ptr(i),
                                                                N.ptr(i), None, B, 0x100 if self.tensor_cores else 0,
                                                                C.byref(ws), N.ptr(loss_out), st, C.byref(rt)),
                        "brk_twotower_step_sharded_retrieval")
            else:
                loss_out.zero_()
        elif self._global is not None:
            u, i = H._i32(u, "u"), H._i32(i, "i")
            if self.emulate:
                bounds = {r: D.local_slice(B, r, self.G) for r in range(self.G)}
                parts = {r: (u[lo:hi], i[lo:hi]) for r, (lo, hi) in bounds.items()}
                split = [hi - lo for lo, hi in bounds.values()]
            else:
                parts = {self.rank: (u, i)}
                split = split if split is not None else [B] * self.G

            def shards(r):
                sh = self._shards()
                sh.user.rank = sh.item.rank = r
                return sh
            ut, it = self._towers()
            self._global.step(ut, it, shards, parts, split, self.tensor_cores, loss_out)
        elif B > 0:
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

    def estimator_state(self):
        """(last [rows] int64, gap [rows] float32, step) of the streaming frequency estimator on the host (None without
        it); collective on real ranks, like ShardedTable.full_weights."""
        return self._est.state() if self._est is not None else None

    def check(self):
        """Raises when a cross-GPU barrier (the estimator's included: it shares the model's flag block) or the Dense
        all-reduce timed out (call at epoch ends, not per step)."""
        if self.barrier is not None:
            self.barrier.check()
        if self._reducer is not None:
            self._reducer.check()
        if self._global is not None:
            self._global.check()

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

    def topk_index(self, itemsId=None, k=10):
        """Top-k index over the item table rows itemsId (default: every row) by the dot product of the tower outputs: see
        ShardedTopKIndex.  The lists equal a BruteForceIndex over score_vectors' outputs; k up to hotpath.fused_k_cap
        of semb."""
        return ShardedDotTopKIndex(self, itemsId, k, self._tower_forward, self.semb, self.item.rows)

    # ---- checkpoint: shards of the tables and their accumulators, replicated Dense blocks and theirs ------------
    # With the estimator also its state: last / gap as row-sharded [rows, 1] entries (re-sharded across world sizes
    # like the tables) and the step counter replicated.  With sampled negatives the sampler's step counter, replicated.
    def _estimator_shards(self):
        e = self._est
        if e is None:
            return {}
        return {"estimator_last": lambda r: e.last[r].view(-1, 1), "estimator_gap": lambda r: e.gap[r].view(-1, 1)}

    def save_checkpoint(self, dirpath):
        rep = {}
        for name, t in zip(("user_dense", "item_dense"), self.dense):
            rep[name], rep[name + "_m"] = t.w.view(-1), t.m.view(-1)
        if self._est is not None:
            rep["estimator_step"] = self._est.step
        if self._smp is not None:
            rep["sampler_step"] = self._smp.step
        extra = {name: (shard, self._est.rows) for name, shard in self._estimator_shards().items()}
        return save_sharded_model(dirpath, {"user": self.user, "item": self.item}, rep, self.G, self.rank, self.emulate,
                                  meta={"model": "ShardedTwoTowerNet", "E": self.embedDim, "S": self.semb,
                                        "numUser": self.numUser, "numItem": self.numItem}, extra=extra)

    def load_checkpoint(self, dirpath):
        """Restores what save_checkpoint wrote, whatever world size wrote it.  A model with the estimator that loads a
        checkpoint without its state (one saved without streamingFrequency) starts the estimator from zero: every row
        unseen and the step counter at 0."""
        rep, meta = load_sharded_model(dirpath, {"user": self.user, "item": self.item}, self.G, self.rank, self.emulate,
                                       extra=self._estimator_shards())
        for name, t in zip(("user_dense", "item_dense"), self.dense):
            t.w.view(-1).copy_(torch.from_numpy(rep[name]))
            t.m.view(-1).copy_(torch.from_numpy(rep[name + "_m"]))
        if self._est is not None:
            self._est.step.fill_(int(rep["estimator_step"][0]) if "estimator_step" in rep else 0)
        if self._smp is not None:                           # a checkpoint saved without sampled negatives: counter 0
            self._smp.step.fill_(int(rep["sampler_step"][0]) if "sampler_step" in rep else 0)
        return meta


# ---- full-catalog top-k over item ranges of the row-sharded models ------------------------------------------------------
def _gather_rows_sharded(table, ids):
    """Rows `ids` (global row ids, int32 on the device) of a ShardedTable: peer loads from the owners' shards (plain local
    loads under emulation or with one GPU)."""
    if ids.numel() == 0:
        return torch.empty((0, table.d), dtype=torch.float32, device=ids.device)
    return H.gather_rows_sharded(table.c_shards(), table.d, ids)


class _ListBuffers:
    """The exchange buffers of ShardedTopKIndex: two alternating slots per range, each [header: 4 int32][scores: cap fp32]
    [ids: cap int32], and per slot the DEVICE pointer arrays (scores, ids, headers of every range) that
    brk_topk_merge_peer reads.  Symmetric (NVLink peer-mapped) memory with one slot pair per rank in a multi-GPU run,
    `G` plain local buffers in one process."""

    def __init__(self, G, device, cap, symmetric):
        self.cap = int(cap)
        self.slot = 4 + 2 * self.cap
        n = 2 * self.slot
        if symmetric:
            import torch.distributed._symmetric_memory as symm_mem
            buf = symm_mem.empty(n, dtype=torch.float32, device=device)
            self._handle = symm_mem.rendezvous(buf, dist.group.WORLD.group_name)
            self.mine = {D.rank(): buf}
            bases = list(self._handle.buffer_ptrs)
        else:
            self.mine = {r: torch.empty(n, dtype=torch.float32, device=device) for r in range(G)}
            bases = [self.mine[r].data_ptr() for r in range(G)]
        for b in self.mine.values():
            b.zero_()
        self.ptrs = []
        for s in (0, 1):
            o = s * self.slot
            self.ptrs.append(torch.tensor([[p + 4 * (o + 4) for p in bases], [p + 4 * (o + 4 + self.cap) for p in bases],
                                           [p + 4 * o for p in bases]], dtype=torch.int64, device=device))

    def views(self, r, s, U, k):
        """(header int32 [4], scores [U, k], ids [U, k]) of range r's slot s."""
        b, o = self.mine[r], s * self.slot
        return (b[o:o + 4].view(torch.int32), b[o + 4:o + 4 + U * k].view(U, k),
                b[o + 4 + self.cap:o + 4 + self.cap + U * k].view(torch.int32).view(U, k))


class ShardedTopKIndex:
    """Full-catalog top-k of a row-sharded model (ShardedNeuMFNet, ShardedBPRNet, ShardedTwoTowerNet) over item ranges.

        index = net.topk_index(itemsId)                  # collective: every rank passes the same itemsId
        scores, ids = index(usersId, k=10)               # collective; ids: positions in itemsId
        scores, ids = index.query_with_exclusions(usersId, hotpath.exclusion_csr(rows, ids, len(usersId), dev))

    Rank r of G indexes the positions [lo, hi) = distributed.local_slice(len(itemsId), r, G): it gathers those items'
    rows from their owners (row-sharded tables: row i on rank i % G) and builds its item side as the unsharded index
    does, with id_offset = lo.  A query gathers the users' rows from the shards, scores them against the local range with
    the model's fused top-k kernel, pads the list to exactly k entries with (-inf, -1), publishes it in a symmetric
    buffer and merges every rank's list from the peers' memory (brk_topk_merge_peer).  Every rank gets the same
    [U, min(k, len(itemsId))] lists, equal bit for bit to the single-GPU index over the full tables.

    Protocol (mode "peer"): the build and every query start with a cross-GPU barrier, so that no rank reads a shard
    while its owner's optimizer pass may still be running.  Users go in chunks of CHUNK_ENTRIES // k; chunk c is
    published in slot c % 2 with a header {seq, U, k}, then a barrier, then the merge.  A rank reaches chunk c + 1's
    barrier only after its merge of chunk c (stream order), so nobody overwrites a slot a peer may still read, with one
    barrier per chunk.  The merge checks every rank's header against its own and the query raises ValueError when they
    differ (a rank skipped a call, or the ranks passed different users or k).  ShardedNeuMFNet(mode="nccl") gathers
    rows with the all-to-all of distributed.ShardedLookup and exchanges the lists with an NCCL all-gather +
    brk_topk_merge, as does a run where symmetric memory is unavailable.  `emulate=G` (and G = 1) scores all ranges in
    one process into local buffers and runs the same merge kernel.

    The index is a snapshot of the item rows: rebuild it after training."""

    CHUNK_ENTRIES = 1 << 21          # list entries (score + id, 8 B) per exchange slot: 16 MB, two slots

    def __init__(self, net, itemsId, k_cap, k=10):
        self.net, self.device = net, net.device
        self.G, self.rank = net.G, net.rank
        self.multi = not net.emulate and self.G > 1
        self.k_cap = int(k_cap)
        self.k = self._check_k(k)
        if itemsId is None:
            items = np.arange(self._num_items(), dtype=np.int32)
        else:
            items = (itemsId.cpu().numpy() if isinstance(itemsId, torch.Tensor) else np.asarray(itemsId)).astype(np.int32).reshape(-1)
        if items.size == 0:
            raise ValueError(f"{type(self).__name__}: no items")
        self.num_candidates = int(items.size)
        self._bufs, self._barrier, self._nccl = None, None, False
        if not self.multi:
            self._bufs = _ListBuffers(self.G, self.device, self.CHUNK_ENTRIES, symmetric=False)
        elif self._peer_rows():
            try:
                self._bufs = _ListBuffers(self.G, self.device, self.CHUNK_ENTRIES, symmetric=True)
                self._barrier = PeerBarrier(self.device)
            except Exception as e:                # pragma: no cover - depends on the box
                self._bufs, self._nccl = None, True
                if self.rank == 0:
                    print(f"[binrec_b200] symmetric memory unavailable ({e!r}); exchanging top-k lists over NCCL", flush=True)
        else:
            self._nccl = True
        self._err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._seq = 0
        self._sync()
        self.parts = {}                                    # range -> (lo, scorer or None for an empty range)
        for r in (range(self.G) if not self.multi else [self.rank]):
            lo, hi = D.local_slice(self.num_candidates, r, self.G)
            self.parts[r] = (lo, self._build_part(items[lo:hi], lo))

    # ---- model-specific hooks ----------------------------------------------------------------------------------------
    def _num_items(self):
        raise NotImplementedError

    def _peer_rows(self):
        """True when rows are gathered with peer loads (the tables live in symmetric memory)."""
        return True

    def _build_part(self, items, lo):
        """Scorer of the positions [lo, lo + len(items)) (items: table rows, host int32; may be empty)."""
        raise NotImplementedError

    def _query(self, users):
        """The user side of a chunk of users (int32 table rows on the device); collective in a multi-GPU run."""
        raise NotImplementedError

    def _score(self, part, query, U, k, exclusions):
        """(scores, ids) [U, min(k, part's items)] of one range; ids are global positions."""
        raise NotImplementedError

    # ---- collective query --------------------------------------------------------------------------------------------
    def _check_k(self, k):
        k = self.k if k is None else int(k)
        if k < 1 or k > self.k_cap:
            raise ValueError(f"k={k}: the sharded top-k of {type(self.net).__name__} keeps 1..{self.k_cap} entries per user")
        return k

    def _sync(self):
        """Cross-GPU barrier: in stream order on the peer path, a host rendezvous after a device synchronise otherwise."""
        if self._barrier is not None:
            self._barrier()
        elif self.multi:
            torch.cuda.synchronize(self.device)
            dist.barrier()

    def __call__(self, usersId, k=None):
        """(scores [U, k], ids [U, k]) for the users usersId (rows of the user tables); ids are positions in itemsId, best
        first, ties to the lower position.  Collective: every rank passes the same users and k."""
        return self._run(usersId, k, None)

    def query_with_exclusions(self, usersId, exclusions, k=None):
        """As the call, with row r's listed positions left out: `exclusions` is an (indptr int64 [>= U+1], ids int32) CSR
        of global positions, ascending within each row (hotpath.exclusion_csr), the same on every rank.  Rows with
        fewer than k remaining items are padded with (-inf, -1)."""
        return self._run(usersId, k, exclusions)

    def _run(self, usersId, k, exclusions):
        k = min(self._check_k(k), self.num_candidates)
        dev = self.device
        users = torch.as_tensor(np.asarray(usersId, dtype=np.int32) if not isinstance(usersId, torch.Tensor) else usersId)
        users = H._i32(users.to(dev).reshape(-1), "usersId")
        U = users.numel()
        vals = torch.empty((U, k), dtype=torch.float32, device=dev)
        ids = torch.empty((U, k), dtype=torch.int32, device=dev)
        if U == 0:
            return vals, ids
        if exclusions is not None:
            exclusions = H._check_csr(exclusions, U, dev)
        self._sync()
        step = max(1, self.CHUNK_ENTRIES // k)
        for s0 in range(0, U, step):
            n = min(U, s0 + step) - s0
            q = self._query(users[s0:s0 + n])
            ex = None if exclusions is None else (exclusions[0][s0:], exclusions[1])
            lists = {r: (self._score(part, q, n, k, ex) if part is not None else None) for r, (lo, part) in self.parts.items()}
            self._exchange(lists, n, k, vals[s0:s0 + n], ids[s0:s0 + n])
        if self._bufs is not None:
            err = int(self._err.item())
            if self._barrier is not None:
                self._barrier.check()
            if err:
                self._err.zero_()
                raise ValueError(f"sharded top-k: rank {err - 1}'s list header differs from this rank's (a rank skipped a "
                                 "query, or the ranks passed different users or k); no result was written")
        return vals, ids

    @staticmethod
    def _pad(lst, dst_v, dst_i):
        """Writes a range's list into [n, k] buffers, padded with (-inf, -1) (a range shorter than k, or empty)."""
        if lst is None or lst[0].shape[1] < dst_v.shape[1]:
            dst_v.fill_(float("-inf")); dst_i.fill_(-1)
        if lst is not None:
            w = lst[0].shape[1]
            dst_v[:, :w].copy_(lst[0]); dst_i[:, :w].copy_(lst[1])

    def _exchange(self, lists, n, k, out_v, out_i):
        dev = self.device
        if self._nccl:
            v = torch.empty((n, k), dtype=torch.float32, device=dev)
            i = torch.empty((n, k), dtype=torch.int32, device=dev)
            self._pad(lists[self.rank], v, i)
            mv, mi = H.topk_merge(*D.gather_topk_parts(v, i))
            out_v.copy_(mv); out_i.copy_(mi)
            return
        slot, seq = self._seq & 1, self._seq & 0x7FFFFFFF
        self._seq += 1
        for r, lst in lists.items():
            hdr, bv, bi = self._bufs.views(r, slot, n, k)
            self._pad(lst, bv, bi)
            hdr[0].fill_(seq); hdr[1].fill_(n); hdr[2].fill_(k)
        if self._barrier is not None:
            self._barrier()                               # every rank's list of this chunk is in its slot
        p = self._bufs.ptrs[slot]
        N.check(N.lib().brk_topk_merge_peer(N.ctx(dev), N.ptr(p[0]), N.ptr(p[1]), N.ptr(p[2]), self.G, n, k, N.ptr(out_v),
                                            N.ptr(out_i), N.ptr(self._err), N.stream_ptr()), "brk_topk_merge_peer")


class ShardedNeuMFTopKIndex(ShardedTopKIndex):
    """ShardedNeuMFNet.topk_index / topk_index_fp32: each range is a NeuMFTopKIndex / NeuMFTopKIndexFP32 whose rows come
    from the shards; a query computes the user half of the factored first layer once (uMLP rows gathered from the
    shards) and hands the kernel a model whose uMF table is the gathered rows.  BatchNorm statistics are per replica in
    sharded training; the index uses rank 0's, broadcast at build time -- those save_checkpoint keeps, so the index
    equals the single-GPU index of the restored checkpoint."""

    def __init__(self, net, itemsId, part_cls):
        part_cls.check_model(net)                      # on every rank, whether or not its range is empty
        self._part_cls = part_cls
        self.bn = D.broadcast_(net.bn_moving.clone(), 0) if (not net.emulate and net.G > 1) else net.bn_moving.clone()
        super().__init__(net, itemsId, H.MAX_FUSED_K)

    def _num_items(self):
        return self.net.numItem

    def _peer_rows(self):
        return self.net.mode == "peer"

    def _build_part(self, items, lo):
        if items.size == 0:
            if self._nccl:                               # join the all-to-all lookups of the ranks that do have items
                self.net._gather_rows(["iMLP"], torch.empty(0, dtype=torch.int32, device=self.device))
                self.net._gather_rows(["iMF"], torch.empty(0, dtype=torch.int32, device=self.device))
            return None
        return _RANGE_CLS[self._part_cls](self.net, items, lo)

    def _query(self, users):
        net = self.net
        uMLP, uMF = net._gather_rows(["uMLP", "uMF"], users)
        n, h1 = users.numel(), net.hidden[0]
        user_side = self._part_cls._product(uMLP, net.param("W1")[:net.E], torch.empty((n, h1), dtype=torch.float32,
                                                                                       device=self.device))
        m = net._c_model()
        m.uMF = N.brk_table(uMF.data_ptr(), None, None, None, None, n, uMF.shape[1], 0)
        m.bn_moving = self.bn.data_ptr()
        return user_side, m, torch.arange(n, dtype=torch.int32, device=self.device), uMF

    def _score(self, part, query, U, k, exclusions):
        return part._score(query[:3], U, min(k, part.num_candidates), exclusions)


class _ShardRows:
    """Row source of a NeuMF index over one item range: the rows are gathered from the shards of ShardedNeuMFNet."""

    def _rows(self, table, ids):
        return self.net._gather_rows([table], ids)[0]


class _NeuMFRange(_ShardRows, NeuMFTopKIndex):
    pass


class _NeuMFRangeFP32(_ShardRows, NeuMFTopKIndexFP32):
    pass


_RANGE_CLS = {NeuMFTopKIndex: _NeuMFRange, NeuMFTopKIndexFP32: _NeuMFRangeFP32}


class ShardedDotTopKIndex(ShardedTopKIndex):
    """ShardedBPRNet.topk_index / ShardedTwoTowerNet.topk_index: each range is a hotpath.BruteForceIndex over the bf16
    candidates of its items (BPR: the item rows; two-tower: the item tower's outputs), queried with the users' rows
    (two-tower: user tower outputs), all gathered from the shards."""

    def __init__(self, net, itemsId, k, vectors, dim, num_items):
        self._vectors, self._num = vectors, num_items
        super().__init__(net, itemsId, H.fused_k_cap(int(N.lib().brk_bf16_padded_dim(dim))), k)

    def _num_items(self):
        return self._num

    def _build_part(self, items, lo):
        if items.size == 0:
            return None
        return H.BruteForceIndex(self.k).index(self._vectors(1, torch.from_numpy(items).to(self.device)), id_offset=lo)

    def _query(self, users):
        return self._vectors(0, users)

    def _score(self, part, query, U, k, exclusions):
        return part(query, k) if exclusions is None else part.query_with_exclusions(query, exclusions, k)
