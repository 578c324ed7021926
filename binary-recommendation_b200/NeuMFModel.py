"""NeuMF (GMF + MLP) -- drop-in mirror of the reference's src/models/NeuMFModel.py (class, method
names, call shapes, return values) and of the script variant trainers/NFC_plain.py.

Underneath: four embedding tables and one flat dense-parameter block resident in HBM, the fused
five-kernel forward/backward of csrc/neumf.cu, Philox negative sampling (csrc/sampler.cu) and one
fused Keras-Adam launch over all parameters (csrc/optim.cu), all through the C ABI.

Differences from the reference, stated once:
  * negatives come from the counter-based sampler (same marginals as NeuMFModel.py:104-105: user and
    item both follow the positives' empirical popularity, no collision check), so runs are reproducible;
    `rejectCollisions = True` on the model re-draws negatives that are known positives (SURVEY.md 8 f1);
  * the merged frame of an epoch (sampling + labels + row shuffle) is written on the device by one kernel
    (csrc/pipeline.cu) instead of pandas on the host;
  * dropout masks come from Philox with keep probability 205/256 (oracle/neumf.py); TensorFlow's
    dropout stream is not reproducible, so rate 0.2 is matched in distribution, not bit for bit;
  * `train` works without a distributedConfig (the reference raises NameError, RModel.py:139);
  * predictForUser sorts by the numeric score (the reference sorts the string form of the score,
    NeuMFModel.py:146,150) and scores each product once (the reference scores 4x redundantly through
    bootstrapDataset's negatives, NeuMFModel.py:135 -> RModel.py:168-170).
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import _torchext as T
from . import distributed as D
from . import hotpath as H
from . import pipeline as PL
from . import synth
from .RModel import RModel

TC_SPECS = {(64, 64, 32, 16), (32, 32, 16, 8)}
# He et al. variant instances of the one-launch tensor-core kernel (csrc/neumf_fused.cu): (E, EMF, hidden)
FUSED_VARIANTS = {(32, 8, (32, 16, 8))}


class NeuMFNet:
    """The 'Keras model' of NeuMFModel.compileModel: inputs {'user','item'}, sigmoid output."""

    DENSE_ORDER = ("W1", "b1", "g1", "be1", "W2", "b2", "g2", "be2", "W3", "b3", "W4", "b4")

    def __init__(self, numUser, numItem, numFactor, hidden=None, act="relu", loss="mse", learning_rate=1e-3,
                 dropout=0.2, seed=42, dropout_seed=11, sparse_adam="keras", device=None, head_order="h3_mf",
                 tensor_cores=False, mf_dim=None, mf_mode="dot", batch_norm=True):
        """mf_dim / mf_mode / batch_norm select the He et al. variant BASELINE.json configs[0] names (not in the
        reference tree): mf_mode="hadamard" feeds the element-wise product uMF[u] * iMF[i] (mf_dim wide) to the head
        instead of the scalar Dot of NeuMFModel.py:79, batch_norm=False drops both BatchNormalization layers."""
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        E = int(numFactor)
        h1, h2, h3 = hidden or (E, E // 2, E // 4)
        EMF = E if mf_dim is None else int(mf_dim)
        if mf_mode not in ("dot", "hadamard"):
            raise ValueError(f"mf_mode {mf_mode!r}: 'dot' or 'hadamard'")
        self.variant = EMF != E or mf_mode != "dot" or not batch_norm
        if min(E, EMF, h1, h2, h3) < 1:
            raise ValueError(f"numFactor {numFactor}: every layer needs at least one unit (hidden={(h1, h2, h3)})")
        if self.variant and (E, EMF, (h1, h2, h3)) in FUSED_VARIANTS and mf_mode == "hadamard" and not batch_norm and act == "relu":
            tensor_cores = True                              # the built instance of the variant is the one-launch kernel
        # every other width runs on the any-width kernels (csrc/neumf_generic.cu): numFactor is free (RModel.py:35)
        self.E, self.hidden, self.EMF, self.mf_mode, self.batch_norm = E, (h1, h2, h3), EMF, mf_mode, bool(batch_norm)
        head_mf = EMF if mf_mode == "hadamard" else 1
        # tensor_cores: the Dense products run on tcgen05 with TF32 operands (csrc/neumf_tc.cu); fp32 otherwise
        if tensor_cores and not self.variant and (E, h1, h2, h3) not in TC_SPECS:
            raise ValueError(f"no tensor-core instance for E={E}, hidden={(h1, h2, h3)}; built: {sorted(TC_SPECS)}")
        self.tensor_cores = bool(tensor_cores)
        self.numUser, self.numItem = int(numUser), int(numItem)
        self.act, self.loss, self.dropout = act, loss, float(dropout)
        self.dropout_seed = dropout_seed
        self.head_order = head_order
        lazy = sparse_adam == "lazy"
        dev = self.device
        rng = np.random.Generator(np.random.Philox(key=seed))
        n_dense = int(N.lib().brk_neumf_dense_floats_ex(E, h1, h2, h3, head_mf))
        npad = (n_dense + 3) // 4 * 4
        # one flat gradient arena (4 tables + dense block): data-parallel replicas all-reduce it once per step
        sizes = [self.numUser * E, self.numItem * E, self.numUser * EMF, self.numItem * EMF, npad]
        # under torch.distributed the arena is NVLink peer-mapped memory and the per-step gradient sum is
        # brk_allreduce_dense_peer (fixed-order sum, bit-identical replicas, no NCCL call on the step's path)
        self.grad_arena, self._reducer = D.gradient_arena(sum(sizes), dev)
        views = list(torch.split(self.grad_arena[:sum(sizes)], sizes))

        def emb(rows, width=E):
            return H.Table(torch.from_numpy(H.keras_embedding_init(rows, width, rng)).to(dev), touched=lazy, g=views.pop(0))

        # draw order = oracle/neumf.py: uMLP, iMLP, uMF, iMF, then the Dense kernels (glorot-uniform)
        self.uMLP, self.iMLP = emb(self.numUser), emb(self.numItem)
        self.uMF, self.iMF = emb(self.numUser, EMF), emb(self.numItem, EMF)

        if lazy and (E, h1, h2, h3) == (10, 100, 50, 10) and not self.variant:
            raise ValueError("row-sparse Adam needs the touched-row marking of the tiled kernels (csrc/neumf2.cu); "
                             "the (10;100,50,10) script spec runs on the first-generation kernels")
        parts = self.initial_dense_parts(E, (h1, h2, h3), rng, head_mf)
        flat = np.concatenate([parts[k].reshape(-1) for k in self.DENSE_ORDER])
        assert flat.size == n_dense
        self.dense = H.Table(torch.from_numpy(np.pad(flat, (0, npad - n_dense))).to(dev).view(1, -1), touched=False,
                             g=views.pop(0))
        self._offsets, off = {}, 0
        for k in self.DENSE_ORDER:
            self._offsets[k] = (off, parts[k].shape)
            off += parts[k].size
        bn = np.concatenate([np.zeros(h1), np.ones(h1), np.zeros(h2), np.ones(h2)]).astype(np.float32)
        self.bn_moving = torch.from_numpy(bn).to(dev)
        self.optimizer = H.Adam(learning_rate, sparse=sparse_adam, device=dev)
        self._ws_batch = 0
        self._ws = None
        self.history = {"loss": []}

    @staticmethod
    def initial_dense_parts(E, hidden, rng, head_mf=1):
        """Keras defaults: Dense glorot-uniform kernels / zero biases, BN gamma 1 / beta 0 (draw order W1..W4)."""
        h1, h2, h3 = hidden

        def glorot(i, o):
            lim = np.sqrt(6.0 / (i + o))
            return rng.uniform(-lim, lim, size=(i, o)).astype(np.float32)

        return {"W1": glorot(2 * E, h1), "b1": np.zeros(h1, np.float32), "g1": np.ones(h1, np.float32),
                "be1": np.zeros(h1, np.float32), "W2": glorot(h1, h2), "b2": np.zeros(h2, np.float32),
                "g2": np.ones(h2, np.float32), "be2": np.zeros(h2, np.float32), "W3": glorot(h2, h3),
                "b3": np.zeros(h3, np.float32), "W4": glorot(h3 + head_mf, 1), "b4": np.zeros(1, np.float32)}

    @classmethod
    def initial_dense(cls, E, hidden, rng):
        parts = cls.initial_dense_parts(E, hidden, rng)
        return np.concatenate([parts[k].reshape(-1) for k in cls.DENSE_ORDER])

    # ---- parameter views -------------------------------------------------------------------------
    def param(self, name, grad=False):
        off, shape = self._offsets[name]
        src = self.dense.g if grad else self.dense.w
        return src.view(-1)[off:off + int(np.prod(shape))].view(*shape)

    def tables(self):
        return [self.uMLP, self.iMLP, self.uMF, self.iMF]

    def _c_model(self):
        h1, h2, h3 = self.hidden
        return N.brk_neumf_model(self.uMLP.c_struct(), self.iMLP.c_struct(), self.uMF.c_struct(), self.iMF.c_struct(),
                                 self.dense.c_struct(), self.bn_moving.data_ptr(), self.E, h1, h2, h3,
                                 0 if self.act == "relu" else 1, 0 if self.loss == "mse" else 1,
                                 1 if self.dropout > 0 else 0, 1 if self.tensor_cores else 0,
                                 self.EMF, 1 if self.mf_mode == "hadamard" else 0, 0 if self.batch_norm else 1, 0)

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

    # ---- steps ---------------------------------------------------------------------------------------
    def forward_backward(self, u, i, y, first_index=0, epoch=0, out=None, loss_out=None, global_batch=0):
        """Fused forward + backward on device tensors; gradients land in the tables' accumulators."""
        B = u.numel()
        out = out if out is not None else torch.empty(B, dtype=torch.float32, device=self.device)
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
        m, ws = self._c_model(), self._workspace(B)
        N.check(N.lib().brk_neumf_step(N.ctx(self.device), C.byref(m), N.ptr(H._i32(u, "u")), N.ptr(H._i32(i, "i")),
                                       N.ptr(H._f32(y, "y")), B, global_batch, first_index, 1, self.dropout_seed & 0xFFFFFFFF,
                                       epoch & 0xFFFFFFFF, C.byref(ws), N.ptr(out), N.ptr(loss_out), N.stream_ptr()),
                "brk_neumf_step")
        return loss_out, out

    def train_on_batch(self, u, i, y, first_index=0, epoch=0, out=None, loss_out=None, global_batch=None):
        """One training step.  Under torch.distributed: mirrored synchronous data parallelism
        (RModel.py:119-121) -- u / i / y are THIS rank's rows of the global batch (global_batch rows in all; default
        world * len(u)), gradients are scaled by 1/global_batch, ONE all-reduce of the flat arena, identical Adam step
        on every rank; BatchNorm statistics stay per replica (MirroredStrategy's default)."""
        w = D.world_size()
        if w == 1 and isinstance(self.optimizer, H.Adam):
            # one C call: fused step + optimizer (ONE kernel when the tensor-core instance covers the model)
            B = u.numel()
            out = out if out is not None else torch.empty(B, dtype=torch.float32, device=self.device)
            loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
            m, ws, opt = self._c_model(), self._workspace(B), self.optimizer
            if T.ops() is not None and opt.sparse == "keras":
                # the PyTorch-extension route: one custom op, tensors in (torch.ops.brk.neumf_train_step)
                tabs = self.tables() + [self.dense]
                h1, h2, h3 = self.hidden
                b = self._bufs
                T.ops().neumf_train_step([t.w for t in tabs], [t.g for t in tabs], [t.m for t in tabs], [t.v for t in tabs],
                                         self.bn_moving, [self.E, h1, h2, h3, 0 if self.act == "relu" else 1,
                                                          0 if self.loss == "mse" else 1, 1 if self.dropout > 0 else 0,
                                                          1 if self.tensor_cores else 0, self.EMF,
                                                          1 if self.mf_mode == "hadamard" else 0, 0 if self.batch_norm else 1],
                                         H._i32(u, "u"), H._i32(i, "i"), H._f32(y, "y"), int(first_index),
                                         self.dropout_seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, opt.h.lr, opt.h.beta1, opt.h.beta2,
                                         opt.h.eps, opt.state, b["h1"], b["h2"], b["dy1"], b["dy2"], b["acc"], out, loss_out)
                return loss_out, out
            N.check(N.lib().brk_neumf_train_step(
                N.ctx(self.device), C.byref(m), N.ptr(H._i32(u, "u")), N.ptr(H._i32(i, "i")), N.ptr(H._f32(y, "y")), B,
                first_index, self.dropout_seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, opt.h, N.ptr(opt.state),
                1 if opt.sparse == "lazy" else 0, C.byref(ws), N.ptr(out), N.ptr(loss_out), N.stream_ptr()),
                "brk_neumf_train_step")
            return loss_out, out
        gb = (int(global_batch) if global_batch is not None else w * u.numel()) if w > 1 else 0
        if u.numel() > 0:
            loss, out = self.forward_backward(u, i, y, first_index, epoch, out, loss_out, global_batch=gb)
        else:                                                # this rank's slice of a ragged last batch may be empty
            loss = loss_out if loss_out is not None else torch.zeros(1, dtype=torch.float32, device=self.device)
            loss.zero_()
        if w > 1:
            D.all_reduce_sum_(self.grad_arena, self._reducer)
        self.optimizer.apply(self.tables(), dense=[self.dense])
        return loss, out

    def train_steps(self, u, i, y, batch, order, epoch=0, losses=None, out=None):
        """The inner loop of fit over a resident frame u / i / y: batch b = rows [b * batch, (b + 1) * batch) for b
        in `order`, fused step + optimizer each, enqueued by ONE C call (brk_neumf_train_steps) -- no Python between
        steps.  Single process with the stock Adam only; otherwise the per-step path (train_on_batch) is used."""
        order = np.ascontiguousarray(order, dtype=np.int64)
        n = u.numel()
        losses = losses if losses is not None else torch.empty(len(order), dtype=torch.float32, device=self.device)
        out = out if out is not None else torch.empty(min(batch, n), dtype=torch.float32, device=self.device)
        if D.world_size() > 1 or not isinstance(self.optimizer, H.Adam):
            for k, b in enumerate(order):
                # data parallel: `batch` is the GLOBAL batch (MultiWorkerMirroredStrategy auto-shards the dataset,
                # RModel.py:119-121); this rank trains its local_slice of it, the dropout stream follows the row's
                # position in the frame, so W ranks reproduce the single-process step up to BatchNorm's per-replica statistics
                lo_g, hi_g = int(b) * batch, min(n, (int(b) + 1) * batch)
                lo, hi = D.local_slice(hi_g - lo_g)
                s = slice(lo_g + lo, lo_g + hi)
                self.train_on_batch(u[s], i[s], y[s], first_index=lo_g + lo, epoch=epoch, out=out[:hi - lo],
                                    loss_out=losses[k:k + 1], global_batch=hi_g - lo_g)
            return losses
        m, ws = self._c_model(), self._workspace(min(batch, n))
        opt = self.optimizer
        N.check(N.lib().brk_neumf_train_steps(
            N.ctx(self.device), C.byref(m), N.ptr(H._i32(u, "u")), N.ptr(H._i32(i, "i")), N.ptr(H._f32(y, "y")), n,
            int(batch), order.ctypes.data_as(C.POINTER(C.c_int64)), len(order), self.dropout_seed & 0xFFFFFFFF,
            epoch & 0xFFFFFFFF, opt.h, N.ptr(opt.state), 1 if opt.sparse == "lazy" else 0, C.byref(ws), N.ptr(out),
            N.ptr(losses), N.stream_ptr()), "brk_neumf_train_steps")
        return losses

    @staticmethod
    def pack_host_batches(users, items, labels, batch_size):
        """Batch-major pinned host frame [n_full_batches, 3, batch] of int32 words (user ids, item ids, labels as float
        bits): what a loader producing ({"user": ids, "item": ids}, label) batches writes (NeuMFModel.py:111-117)."""
        nb = len(users) // int(batch_size)
        packed = torch.empty((nb, 3, int(batch_size)), dtype=torch.int32).pin_memory()
        a = packed.numpy()
        n = nb * int(batch_size)
        a[:, 0, :] = np.asarray(users[:n], dtype=np.int32).reshape(nb, -1)
        a[:, 1, :] = np.asarray(items[:n], dtype=np.int32).reshape(nb, -1)
        a[:, 2, :] = np.asarray(labels[:n], dtype=np.float32).view(np.int32).reshape(nb, -1)
        return packed

    def train_steps_from_host(self, packed_host, order, epoch=0, losses_host=None):
        """End-to-end steps from a pack_host_batches() frame in page-locked HOST memory: per step one H2D copy of the
        batch (12 B per sample), the fused step + optimizer, and one D2H copy of all step losses at the end -- all
        enqueued by ONE C call (brk_neumf_train_steps_host); returns the pinned loss tensor (valid after a stream
        synchronize).  Single process with the stock Adam."""
        if D.world_size() > 1 or not isinstance(self.optimizer, H.Adam):
            raise NotImplementedError("host-fed NeuMF steps: single process with the Adam optimizer")
        nb, three, batch = packed_host.shape
        order = np.ascontiguousarray(order, dtype=np.int64)
        k = len(order)
        dev = self.device
        need = int(N.lib().brk_neumf_host_stage_ints(batch))
        if getattr(self, "_stage", None) is None or self._stage.numel() < need:
            self._stage = torch.empty(need, dtype=torch.int32, device=dev)
        d_losses = torch.empty(max(k, 1), dtype=torch.float32, device=dev)
        if losses_host is None:
            losses_host = torch.empty(max(k, 1), dtype=torch.float32).pin_memory()
        out = torch.empty(batch, dtype=torch.float32, device=dev)
        m, ws, opt = self._c_model(), self._workspace(batch), self.optimizer
        N.check(N.lib().brk_neumf_train_steps_host(
            N.ctx(dev), C.byref(m), C.c_void_p(packed_host.data_ptr()), nb, batch, order.ctypes.data_as(C.POINTER(C.c_int64)), k,
            self.dropout_seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, opt.h, N.ptr(opt.state), 1 if opt.sparse == "lazy" else 0,
            C.byref(ws), N.ptr(self._stage), N.ptr(out), N.ptr(d_losses), C.c_void_p(losses_host.data_ptr()), N.stream_ptr()),
            "brk_neumf_train_steps_host")
        self._keep = (d_losses, out)                         # alive until the stream has consumed them
        return losses_host[:k]

    def predict_on_batch(self, u, i, y=None):
        """Inference with the BN moving statistics; returns (predictions, loss or None)."""
        B = u.numel()
        out = torch.empty(B, dtype=torch.float32, device=self.device)
        loss_out = torch.empty(1, dtype=torch.float32, device=self.device) if y is not None else None
        m, ws = self._c_model(), self._workspace(B)
        N.check(N.lib().brk_neumf_step(N.ctx(self.device), C.byref(m), N.ptr(H._i32(u, "u")), N.ptr(H._i32(i, "i")),
                                       N.ptr(y) if y is not None else None, B, 0, 0, 0, 0, 0, C.byref(ws), N.ptr(out),
                                       N.ptr(loss_out) if loss_out is not None else None, N.stream_ptr()),
                "brk_neumf_step")
        return out, loss_out

    # ---- Keras-like API -------------------------------------------------------------------------------
    def fit(self, dataset, validation_data=None, epochs=1, steps_per_epoch=None, verbose=0):
        """dataset: a NeuMFDataset (bootstrapDataset).  One pass per epoch; batch ORDER reshuffled per
        epoch as tf.data's .batch().shuffle() does (NeuMFModel.py:117-121)."""
        for e in range(epochs):
            if e == 0:
                D.barrier()                                  # nobody enters a cross-GPU wait while a rank is still staging
            losses = dataset.run_epoch(self, e, steps_per_epoch)
            mean = float(losses.double().mean().item())
            if getattr(self, "_reducer", None) is not None:
                self._reducer.check()                        # a peer all-reduce that timed out aborted its step: raise here
            self.history["loss"].append(mean)
            if validation_data is not None:
                self.history.setdefault("val_loss", []).append(self.evaluate(validation_data)[0])
            if verbose:
                print(f"epoch {e + 1}: loss {mean:.6f}")
        return self

    def evaluate(self, dataset, steps=None):
        """[loss, mse, mae, binary_accuracy] -- the reference's METRICS list (RModel.py:20,144-147)."""
        tot = 0; acc = np.zeros(4)
        for k, (u, i, y) in enumerate(dataset.batches()):
            if steps is not None and k >= steps:
                break
            out, loss = self.predict_on_batch(u, i, y)
            n = u.numel()
            err = out - y
            acc += n * np.array([float(loss.item()), float((err * err).mean().item()), float(err.abs().mean().item()),
                                 float(((out > 0.5).float() == y).float().mean().item())])
            tot += n
        return list(acc / max(tot, 1))

    def predict(self, dataset):
        return torch.cat([self.predict_on_batch(u, i)[0] for u, i, _ in dataset.batches()]).unsqueeze(1)

    def score_all(self, usersId, itemsId, k, exclude=None):
        """Top-k over the whole catalog for each user (topKRatings' "NFC" path, topKmetrics.py:29-33):
        NeuMF has no factorised scorer, so every (user, item) pair goes through the fused forward.  `exclude`: an
        (indptr, ids) CSR over the rows of usersId listing positions in itemsId to leave out (hotpath.exclusion_csr);
        they are masked in each chunk's scores before the selection, and short rows are padded with (-inf, -1)."""
        dev = self.device
        items = torch.as_tensor(np.asarray(itemsId, dtype=np.int32)).to(dev)
        I = items.numel()
        k = min(k, I)
        vals, idxs = [], []
        chunk = max(1, (1 << 22) // I)
        users = np.asarray(usersId, dtype=np.int32)
        for s in range(0, len(users), chunk):
            uu = torch.as_tensor(users[s:s + chunk]).to(dev)
            out, _ = self.predict_on_batch(uu.repeat_interleave(I), items.repeat(uu.numel()))
            S = out.view(uu.numel(), I)
            if exclude is not None:
                H.mask_excluded(S, exclude[0][s:s + uu.numel() + 1], exclude[1], 0)
            v, ix = H.topk_rows(S, k)
            vals.append(v); idxs.append(ix)
        return torch.cat(vals), torch.cat(idxs)

    def topk_index(self, itemsId=None, id_offset=0):
        """Full-catalog top-k index over itemsId (default: every item): see NeuMFTopKIndex.  It snapshots the item side
        of the model, so rebuild it after training."""
        return NeuMFTopKIndex(self, itemsId, id_offset)

    def topk_index_fp32(self, itemsId=None, id_offset=0):
        """Full-catalog top-k index of an fp32 model (tensor_cores=False) over itemsId (default: every item): see
        NeuMFTopKIndexFP32.  It snapshots the item side of the model, so rebuild it after training."""
        return NeuMFTopKIndexFP32(self, itemsId, id_offset)

    def state_dict(self):
        sd = {"bn_moving": self.bn_moving.cpu(), "opt_state": self.optimizer.state.cpu()}
        for name, t in zip(("uMLP", "iMLP", "uMF", "iMF", "dense"), self.tables() + [self.dense]):
            sd[name] = t.w.cpu(); sd[name + "_m"] = t.m.cpu(); sd[name + "_v"] = t.v.cpu()
        return sd

    def load_state_dict(self, sd):
        """Also accepts the whole-table view of a checkpoint written by sharded.ShardedNeuMFNet (same names)."""
        self.bn_moving.copy_(sd["bn_moving"]); self.optimizer.state.copy_(sd["opt_state"])
        for name, t in zip(("uMLP", "iMLP", "uMF", "iMF", "dense"), self.tables() + [self.dense]):
            for slot, key in ((t.w, name), (t.m, name + "_m"), (t.v, name + "_v")):
                if tuple(sd[key].reshape(-1).shape) != tuple(slot.reshape(-1).shape):
                    raise ValueError(f"checkpoint tensor {key!r} has {sd[key].numel()} elements, the model needs {slot.numel()}")
                slot.copy_(sd[key].reshape(slot.shape))


def _gemm_tf32(a, w, out, bias=None):
    """out [M, N] = a [M, K] @ w [K, N] (+ bias) with TF32 operands and fp32 accumulation (brk_gemm_tf32)."""
    M, K = a.shape
    Nn = w.shape[1]
    N.check(N.lib().brk_gemm_tf32(N.ctx(a.device), N.ptr(a), C.c_void_p(w.data_ptr()), N.ptr(out),
                                  C.c_void_p(bias.data_ptr()) if bias is not None else None, M, Nn, K, K, Nn, Nn, 0, 0,
                                  1.0, 0, N.stream_ptr()), "brk_gemm_tf32")
    return out


def _sgemm(a, w, out, bias=None):
    """out [M, N] = a [M, K] @ w [K, N] (+ bias) in fp32 on the CUDA cores (brk_sgemm); a row of out depends on that row
    of a alone (no split K)."""
    M, K = a.shape
    Nn = w.shape[1]
    N.check(N.lib().brk_sgemm(N.ctx(a.device), N.ptr(a), C.c_void_p(w.data_ptr()), N.ptr(out),
                              C.c_void_p(bias.data_ptr()) if bias is not None else None, M, Nn, K, K, Nn, Nn, 0, 0, 1.0, 0,
                              N.stream_ptr()), "brk_sgemm")
    return out


class _FactoredTopKIndex:
    """What the NeuMF top-k indexes share: the item half of the factored first layer computed once, the user half per
    query, then one scoring + selection launch.  Subclasses name the product and the C entry points."""

    K_MAX = H.MAX_FUSED_K

    def __init__(self, net, itemsId=None, id_offset=0):
        self.net = net
        dev = net.device
        if itemsId is None:
            items = torch.arange(net.numItem, dtype=torch.int32, device=dev)
        else:
            items = torch.as_tensor(np.asarray(itemsId, dtype=np.int32)).to(dev)
        if items.numel() == 0:
            raise ValueError(f"{type(self).__name__}: no items")
        self.num_candidates = items.numel()
        self.id_offset = int(id_offset)
        E = net.E
        W1 = net.param("W1")                                 # [2E, H1]: rows [0, E) act on uMLP, [E, 2E) on iMLP
        self._W1u, self._W1i = W1[:E], W1[E:]
        self.item_side = self._product(self._rows("iMLP", items), self._W1i,
                                       torch.empty((items.numel(), net.hidden[0]), dtype=torch.float32, device=dev),
                                       net.param("b1"))
        self.item_mf = self._rows("iMF", items)

    def _rows(self, table, ids):
        """Rows `ids` (int32, device) of the model's table `table` ("uMLP", "iMLP", "uMF", "iMF"); the indexes of
        sharded.ShardedNeuMFNet gather them from the shards instead."""
        return H.gather_rows(getattr(self.net, table).w, ids)

    @staticmethod
    def _product(a, w, out, bias=None):
        raise NotImplementedError

    def _workspace_bytes(self, lib, ctx, m, U, k):
        raise NotImplementedError

    _SCORE = _SCORE_EXCL = None                              # names of the C entry points

    def _check_k(self, k):
        k = 10 if k is None else int(k)
        if k < 1 or k > self.K_MAX:
            raise ValueError(f"k={k}: the fused NeuMF top-k keeps 1..{self.K_MAX} entries per user; use NeuMFNet.score_all")
        return min(k, self.num_candidates)

    def _run(self, usersId, k, exclusions):
        k = self._check_k(k)
        users = self._users(usersId)
        U = users.numel()
        if U == 0:
            dev = self.net.device
            return torch.empty((0, k), dtype=torch.float32, device=dev), torch.empty((0, k), dtype=torch.int32, device=dev)
        if exclusions is not None:
            exclusions = H._check_csr(exclusions, U, self.net.device)
        return self._score(self._query(users), U, k, exclusions)

    def _users(self, usersId):
        users = torch.as_tensor(np.asarray(usersId, dtype=np.int32) if not isinstance(usersId, torch.Tensor) else usersId)
        return H._i32(users.to(self.net.device).reshape(-1), "usersId")

    def _query(self, users):
        """The user half of a query: (user_side [U, H1], brk_neumf_model, the kernel's user rows)."""
        net = self.net
        user_side = self._product(self._rows("uMLP", users), self._W1u,
                                  torch.empty((users.numel(), net.hidden[0]), dtype=torch.float32, device=net.device))
        return user_side, net._c_model(), users

    def _score(self, query, U, k, exclusions):
        """One scoring + selection launch over this index's items for a prepared query; `exclusions`: a checked CSR or
        None.  Returns (vals, ids) [U, k]."""
        user_side, m, users = query
        dev = self.net.device
        vals = torch.empty((U, k), dtype=torch.float32, device=dev)
        ids = torch.empty((U, k), dtype=torch.int32, device=dev)
        lib, ctx = N.lib(), N.ctx(dev)
        ws_bytes = self._workspace_bytes(lib, ctx, m, U, k)
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        if exclusions is None:
            N.check(getattr(lib, self._SCORE)(ctx, C.byref(m), N.ptr(user_side), N.ptr(users), U, N.ptr(self.item_side),
                                              N.ptr(self.item_mf), self.num_candidates, k, self.id_offset, N.ptr(vals),
                                              N.ptr(ids), N.ptr(ws), ws_bytes, N.stream_ptr()), self._SCORE)
        else:
            indptr, xids = exclusions
            N.check(getattr(lib, self._SCORE_EXCL)(ctx, C.byref(m), N.ptr(user_side), N.ptr(users), U,
                                                   N.ptr(self.item_side), N.ptr(self.item_mf), self.num_candidates, k,
                                                   self.id_offset, N.ptr(indptr), N.ptr(xids), N.ptr(vals), N.ptr(ids),
                                                   N.ptr(ws), ws_bytes, N.stream_ptr()), self._SCORE_EXCL)
        return vals, ids

    def __call__(self, usersId, k=None):
        """(scores [U, k], ids [U, k]) for the users usersId (rows of the user tables)."""
        return self._run(usersId, k, None)

    def query_with_exclusions(self, usersId, exclusions, k=None):
        """As the call, with row r's listed ids left out: `exclusions` is an (indptr int64 [>= U+1], ids int32) CSR of
        global ids (position + id_offset), ascending within each row (hotpath.exclusion_csr).  Rows with fewer than k
        remaining items are padded with (-inf, -1)."""
        return self._run(usersId, k, exclusions)


class NeuMFTopKIndex(_FactoredTopKIndex):
    """Full-catalog NeuMF top-k in one kernel launch (brk_neumf_score_topk): for each queried user, the k items of the
    index with the highest prediction -- the value predict_on_batch returns for the pair, to TF32 rounding -- sorted
    by score, ties to the lower position, scores never materialised.  Shaped like hotpath.BruteForceIndex:

        index = net.topk_index(itemsId)            # item side: iMLP[items] W1[E:2E] + b1 and the items' iMF rows
        scores, ids = index(usersId, k=10)         # ids: positions in itemsId plus id_offset
        scores, ids = index.query_with_exclusions(usersId, hotpath.exclusion_csr(rows, ids, len(usersId), dev))

    The first Dense layer factors over [uMLP[u], iMLP[i]], so building the index computes the item half once and a
    query the user half once; the kernel runs the rest of the network per pair on the tensor cores.  The index is a
    snapshot of the item tables and keeps the model for the dense block, the BatchNorm statistics and the user tables:
    rebuild it after training.  Built for the tensor-core class graph (numFactor 32 or 64, relu) and the He et al.
    variant (E 32, mf_dim 8, hadamard, no BatchNorm); other models, and k > 32, raise ValueError -- rank them with
    NeuMFNet.score_all (the fp32 models: NeuMFNet.topk_index_fp32).

    Item-range shards: rank r indexes its range [lo, hi) with id_offset = lo; the merged lists equal the unsharded
    index's bit for bit:

        index = net.topk_index(np.arange(lo, hi), id_offset=lo)
        scores, ids = distributed.sharded_topk(usersId, None, lo, k, local_topk=lambda q, c, off: index(q, k))

    (or hotpath.topk_merge over the stacked [shards, U, k] lists in one process)."""

    _SCORE, _SCORE_EXCL = "brk_neumf_score_topk", "brk_neumf_score_topk_excl"
    _product = staticmethod(_gemm_tf32)

    def __init__(self, net, itemsId=None, id_offset=0):
        self.check_model(net)
        super().__init__(net, itemsId, id_offset)

    @staticmethod
    def check_model(net):
        """Raises ValueError unless a fused top-k instance covers the model."""
        h1, h2, h3 = net.hidden
        ok = net.act == "relu" and (
            (not net.variant and net.tensor_cores and (net.E, h1, h2, h3) in TC_SPECS) or
            (net.variant and net.mf_mode == "hadamard" and not net.batch_norm and
             (net.E, net.EMF, net.hidden) in FUSED_VARIANTS))
        if not ok:
            raise ValueError(f"no fused top-k instance for E={net.E}, mf_dim={net.EMF}, hidden={net.hidden}, act={net.act}, "
                             f"mf_mode={net.mf_mode}, batch_norm={net.batch_norm}, tensor_cores={net.tensor_cores}; built: "
                             f"tensor-core class graph {sorted(TC_SPECS)} and the He et al. variant {sorted(FUSED_VARIANTS)} "
                             "-- use NeuMFNet.score_all")

    def _workspace_bytes(self, lib, ctx, m, U, k):
        return lib.brk_neumf_topk_workspace_bytes(ctx, U, self.num_candidates, k)


class NeuMFTopKIndexFP32(_FactoredTopKIndex):
    """Full-catalog top-k for the fp32 NeuMF models in one kernel launch on the CUDA cores (brk_neumf_score_topk_fp32):
    for each queried user, the k items of the index with the highest prediction -- the value predict_on_batch returns
    for the pair, to fp32 rounding -- sorted by score, ties to the lower position, scores never materialised.  The
    surface is NeuMFTopKIndex's:

        index = net.topk_index_fp32(itemsId)       # item side: iMLP[items] W1[E:2E] + b1 (fp32) and the items' iMF rows
        scores, ids = index(usersId, k=10)         # ids: positions in itemsId plus id_offset
        scores, ids = index.query_with_exclusions(usersId, hotpath.exclusion_csr(rows, ids, len(usersId), dev))

    Both halves of the factored first layer are fp32 products (brk_sgemm), and the kernel runs the rest of the network
    per pair in fp32.  Covers every fp32 model (tensor_cores=False) up to H1 <= 128, H2 <= 64, H3 <= 32 and
    mf_dim <= 128 (numFactor free): the class graph NeuMFModel builds at any numFactor <= 128, the NFC_plain network of
    NCFModel / fit_nfc_plain (sigmoid, hidden (100, 50, 10)) and the fp32 He-style variants (Hadamard head, with or
    without BatchNorm).  Tensor-core models raise ValueError (use NeuMFNet.topk_index), as do wider models and k > 32
    (use NeuMFNet.score_all).  Like NeuMFTopKIndex the index is a snapshot of the item tables: rebuild it after training.

    Item-range shards: rank r indexes its range [lo, hi) with id_offset = lo; the merged lists equal the unsharded
    index's bit for bit:

        index = net.topk_index_fp32(np.arange(lo, hi), id_offset=lo)
        scores, ids = distributed.sharded_topk(usersId, None, lo, k, local_topk=lambda q, c, off: index(q, k))

    (or hotpath.topk_merge over the stacked [shards, U, k] lists in one process)."""

    MAX_WIDTHS = dict(H1=128, H2=64, H3=32, mf_dim=128)
    _SCORE, _SCORE_EXCL = "brk_neumf_score_topk_fp32", "brk_neumf_score_topk_fp32_excl"
    _product = staticmethod(_sgemm)

    def __init__(self, net, itemsId=None, id_offset=0):
        self.check_model(net)
        super().__init__(net, itemsId, id_offset)

    @classmethod
    def check_model(cls, net):
        """Raises ValueError unless the fp32 kernel covers the model."""
        if net.tensor_cores:
            raise ValueError("the model computes with TF32 tensor-core products (tensor_cores=True): rank it with "
                             "NeuMFNet.topk_index")
        h1, h2, h3 = net.hidden
        cap = cls.MAX_WIDTHS
        if h1 > cap["H1"] or h2 > cap["H2"] or h3 > cap["H3"] or net.EMF > cap["mf_dim"]:
            raise ValueError(f"no fp32 top-k instance for hidden={net.hidden}, mf_dim={net.EMF}; built up to hidden "
                             f"({cap['H1']}, {cap['H2']}, {cap['H3']}) and mf_dim {cap['mf_dim']} -- use NeuMFNet.score_all")

    def _workspace_bytes(self, lib, ctx, m, U, k):
        return lib.brk_neumf_topk_fp32_workspace_bytes(ctx, C.byref(m), U, self.num_candidates, k)


class NeuMFDataset:
    """What bootstrapDataset returns: positives + Philox negatives, labels 1/0, one seeded row shuffle,
    cut into batches; resident on the device.  Iterating yields ({"user": ids, "item": ids}, label)
    like the reference's tf.data pipeline (NeuMFModel.py:111-123).  The whole frame is written by ONE
    kernel (pipeline.neumf_epoch_build: keyed permutation + positive copy / negative draw + label);
    resample(epoch) rebuilds it in place with fresh negatives and a fresh row order (the reference
    samples once per bootstrapDataset call)."""

    def __init__(self, users, items, negRatio, batchSize, shuffle, device, seed=7, epoch=0, reject=False,
                 numUser=None):
        dev = device
        users = np.ascontiguousarray(users, dtype=np.int32)
        items = np.ascontiguousarray(items, dtype=np.int32)
        self.pu = torch.from_numpy(users).to(dev)
        self.pi = torch.from_numpy(items).to(dev)
        P = self.pu.numel()
        self.n_neg = int(round(P * negRatio))
        self.n = P + self.n_neg
        self.batchSize, self.shuffle, self.seed = int(batchSize), shuffle, seed
        self.device = dev
        self.reject = bool(reject)
        self.csr = None
        if self.reject:
            nu = int(numUser) if numUser is not None else int(users.max()) + 1
            indptr, sitems = synth.build_csr(users, items, nu)
            self.csr = (torch.from_numpy(indptr).to(dev), torch.from_numpy(sitems).to(dev))
        self.u = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.i = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.y = torch.empty(self.n, dtype=torch.float32, device=dev)
        self.resample(epoch)

    def resample(self, epoch):
        """mergeDf = concat(pos, neg).sample(frac=1.) (NeuMFModel.py:103-109), seeded by (seed, epoch)."""
        PL.neumf_epoch_build(self.pu, self.pi, self.n_neg, self.seed, epoch, reject=self.reject,
                             csr_indptr=self.csr[0] if self.csr else None,
                             csr_items=self.csr[1] if self.csr else None, out=(self.u, self.i, self.y))
        self.epoch = epoch

    def batch_order(self, epoch):
        """`.batch(batchSize).shuffle(...)` (NeuMFModel.py:117-121): whole batches are permuted per epoch."""
        nb = len(self)
        return PL.epoch_permutation_host(nb, self.seed, epoch, PL.SALT_BATCHES) if self.shuffle else np.arange(nb)

    def __len__(self):
        return (self.n + self.batchSize - 1) // self.batchSize

    def batches(self, order=None):
        nb = len(self)
        for b in (order if order is not None else range(nb)):
            s = slice(b * self.batchSize, min(self.n, (b + 1) * self.batchSize))
            yield self.u[s], self.i[s], self.y[s]

    def __iter__(self):
        for u, i, y in self.batches():
            yield {"user": u, "item": i}, y

    def run_epoch(self, net, epoch, steps=None):
        nb = len(self)
        order = self.batch_order(epoch)
        if steps is not None:
            order = order[:int(steps)]
        if hasattr(net, "train_steps"):                       # one C call for the whole list of batches
            return net.train_steps(self.u, self.i, self.y, self.batchSize, order, epoch=epoch)
        losses = torch.empty(len(order), dtype=torch.float32, device=self.device)
        outs = torch.empty(self.batchSize, dtype=torch.float32, device=self.device)
        for k, b in enumerate(order):                         # nets with their own step (row-sharded tables)
            lo_g, hi_g = int(b) * self.batchSize, min(self.n, (int(b) + 1) * self.batchSize)
            lo, hi = D.local_slice(hi_g - lo_g)              # this rank's rows of the global batch (whole batch when single)
            s = slice(lo_g + lo, lo_g + hi)
            net.train_on_batch(self.u[s], self.i[s], self.y[s], first_index=lo_g + lo, epoch=epoch,
                               out=outs[:hi - lo], loss_out=losses[k:k + 1])
        return losses


class NeuMFModel(RModel):

    def __init__(self, workDir=None):
        super().__init__('NeuMFModel', workDir)
        self.sparseAdam = "keras"
        self.dropout = 0.2
        self.rejectCollisions = False      # reference semantics: no collision check (NeuMFModel.py:104-105)
        self._testProducts, self._testUsers = [], []

    def prepareToTrain(self, distributedConfig, path, rowLimit):
        numItem, numUser, (users, items) = self.readData(path, rowLimit)
        (trU, trI), (teU, teI) = synth.train_test_split(users, items, self.testSize, seed=self.splitSeed)
        self._testProducts = np.unique(teI).tolist()          # pickled in the reference (NeuMFModel.py:34-38)
        self._testUsers = np.unique(teU).tolist()
        print(len(trU), 'train examples')
        print(len(teU), 'testSplit examples')
        if distributedConfig is None:
            trainDataset = self.bootstrapDataset((trU, trI))
            testDataset = self.bootstrapDataset((teU, teI), shuffle=False)
        else:
            trainDataset = self.bootstrapDataset((trU, trI), batchSize=self.batchSize)
            testDataset = self.bootstrapDataset((teU, teI), batchSize=self.batchSize, shuffle=False)
        self.model = self.compileModel(distributedConfig, numUser, numItem, self.numFactor)
        return trainDataset, testDataset, (trU, trI)

    def compileModel(self, distributedConfig, numUser: int, numItem: int, numFactor: int):
        """Adam(1e-3), mean squared error, metrics mse/mae/binary_accuracy (NeuMFModel.py:87-91)."""
        self.model = NeuMFNet(numUser, numItem, numFactor, act="relu", loss="mse", learning_rate=1e-3,
                              dropout=self.dropout, seed=self.seed, sparse_adam=self.sparseAdam)
        return self.model

    def bootstrapDataset(self, df, negRatio=3., batchSize=128, shuffle=True):
        users, items = self._loadPairs(df, None)
        dev = torch.device(f"cuda:{torch.cuda.current_device()}")
        return NeuMFDataset(users, items, negRatio, batchSize, shuffle, dev, seed=self.samplerSeed,
                            reject=self.rejectCollisions)

    def train(self, path, rowLimit, metricDict: dict = {}, distributedConfig=None):
        trainDataset, testDataset, trainSplit = self.prepareToTrain(distributedConfig, path, rowLimit)
        if distributedConfig is None:
            self.model.fit(trainDataset, validation_data=testDataset, epochs=self.epochs)
        else:
            steps = int(len(trainDataset) / self.epochs / self.getNumberOfWorkers(distributedConfig))
            self.model.fit(trainDataset, validation_data=testDataset, epochs=self.epochs, steps_per_epoch=max(steps, 1))
        self.saveCheckPoint()
        print("Evaluating trained model...")
        _, val = synth.train_test_split(trainSplit[0], trainSplit[1], 0.2, seed=self.splitSeed + 1)
        valDataset = self.bootstrapDataset(val, shuffle=False)
        evaluatedMetric = self.model.evaluate(valDataset, steps=self.validationSteps)
        return {'result': 'completed', 'metrics': evaluatedMetric}

    def checkpointMeta(self) -> dict:
        return {"model": self.modelName, "numUser": self.model.numUser, "numItem": self.model.numItem,
                "numFactor": self.model.E, "testProducts": [int(x) for x in self._testProducts],
                "testUsers": [int(x) for x in self._testUsers]}

    def buildFromMeta(self, meta: dict):
        self.compileModel(None, meta["numUser"], meta["numItem"], meta["numFactor"])
        self._testProducts, self._testUsers = list(meta.get("testProducts", [])), list(meta.get("testUsers", []))

    def getPredictableUsers(self) -> list:
        return list(self._testUsers)

    def getPredictDataFrame(self, customerId):
        return {self.PRODUCT_ID: list(self._testProducts), self.CUSTOMER_ID: [customerId] * len(self._testProducts)}

    def predictForUser(self, customerId, numberOfItem=5):
        """[(str(item), str(score)), ...] best first, as NeuMFModel.py:133-150 returns."""
        return self.predictForUsers([customerId], numberOfItem)[0]

    def predictForUsers(self, customerIds, numberOfItem=5):
        """predictForUser for a batch of users in one pass (the serving handoff of SURVEY.md section 8 row f3): every
        (user, product) pair goes through the fused forward in large batches and the per-user top lists come from
        the device top-k kernel (NeuMFNet.score_all); one host read for the whole batch."""
        customerIds = [int(c) for c in customerIds]
        bad = [c for c in customerIds if not 0 <= c < self.model.numUser]
        if bad:
            raise ValueError(f"unknown customer ids {bad[:5]}")
        if not self._testProducts or not customerIds:
            return [[] for _ in customerIds]
        k = min(int(numberOfItem), len(self._testProducts))
        v, ix = self.model.score_all(customerIds, self._testProducts, k)
        v, ix = v.cpu().numpy(), ix.cpu().numpy()
        return [[(str(self._testProducts[j]), str(s)) for s, j in zip(v[r], ix[r])] for r in range(len(customerIds))]
