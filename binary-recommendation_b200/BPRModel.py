"""BPR matrix factorisation -- drop-in mirror of the reference's src/models/BPRModel.py (class,
method names and call shapes) and of the functional script src/models/bpr.py.

What runs underneath: tables in HBM, Philox negative sampling (csrc/sampler.cu), one fused
gather + loss + scatter-add kernel per batch (csrc/bpr.cu) and a fused Keras-Adam pass
(csrc/optim.cu), all through the C ABI.

Differences from the reference, stated once:
  * the reference enumerates every (positive, non-interacted) pair on the host
    (BPRModel.py:111-119) -- O(P*I), infeasible beyond toy sizes; `train` samples one
    non-interacted negative per positive per epoch with the counter-based sampler instead
    (extractPositivesNegatives is kept for small inputs and for tests);
  * BPRModel.train in the reference calls compileModel with 3 arguments against a 4-argument
    signature and stores the returned tuple as the model (BPRModel.py:107 vs :49,74); here the
    signature is the 4-argument one and `self.model` is the model;
  * ids are int32 (the reference casts them to float32, BPRModel.py:101-103).
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import distributed as D
from . import hotpath as H
from . import synth
from .RModel import RModel


class BPRNet:
    """The 'Keras model' of BPRModel.compileModel: inputs customerId_input / pProduct_input /
    nProduct_input, output the per-row triplet loss 1 - sigmoid(x_ui - x_uj)."""

    def __init__(self, numUser, numItem, numFactor, seed=42, learning_rate=1e-3, sparse_adam="keras",
                 device=None):
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        self.numUser, self.numItem, self.numFactor = int(numUser), int(numItem), int(numFactor)
        rng = np.random.Generator(np.random.Philox(key=seed))
        # Keras Embedding default init U(-0.05, 0.05); user table first, then item (same draw order as the oracle)
        lazy = sparse_adam == "lazy"   # the touched-row bitmask is only needed by the row-sparse optimizer
        # one flat gradient arena for both tables: data-parallel replicas sum it with ONE all-reduce
        nu, ni = self.numUser * self.numFactor, self.numItem * self.numFactor
        wu = torch.from_numpy(H.keras_embedding_init(self.numUser, self.numFactor, rng)).to(self.device)
        wi = torch.from_numpy(H.keras_embedding_init(self.numItem, self.numFactor, rng)).to(self.device)
        # multi-rank: weights and gradients live in NVLink peer-mapped arenas and the optimizer step is the
        # fused reduce-scatter + Adam + all-gather kernel (csrc/dp_peer.cu); Adam moments are sharded
        self.peer = None if lazy else D.peer_arena_or_none(nu + ni, self.device)
        if self.peer is not None:
            self.grad_arena = self.peer.g
            self.peer.w[:nu].copy_(wu.view(-1)); self.peer.w[nu:nu + ni].copy_(wi.view(-1))
            self.user = H.Table(self.peer.w[:nu].view(self.numUser, self.numFactor), slots=0, touched=False,
                                g=self.grad_arena[:nu])
            self.item = H.Table(self.peer.w[nu:nu + ni].view(self.numItem, self.numFactor), slots=0, touched=False,
                                g=self.grad_arena[nu:nu + ni])
        else:
            self.grad_arena = torch.zeros(nu + ni, dtype=torch.float32, device=self.device)
            self.user = H.Table(wu, touched=lazy, g=self.grad_arena[:nu])
            self.item = H.Table(wi, touched=lazy, g=self.grad_arena[nu:])
        self.optimizer = H.Adam(learning_rate, sparse=sparse_adam, device=self.device)
        self._pairs = None
        self.history = {"loss": []}

    # ---- data residency ------------------------------------------------------------------------
    def set_training_pairs(self, users, items):
        """Uploads the positive pairs once; they stay resident for all epochs."""
        users = np.ascontiguousarray(users, dtype=np.int32); items = np.ascontiguousarray(items, dtype=np.int32)
        indptr, sitems = synth.build_csr(users, items, self.numUser)
        dev = self.device
        self._pairs = dict(u=torch.from_numpy(users).to(dev), p=torch.from_numpy(items).to(dev),
                           n=torch.empty(len(users), dtype=torch.int32, device=dev),
                           indptr=torch.from_numpy(indptr).to(dev), sitems=torch.from_numpy(sitems).to(dev),
                           total=len(users))

    def sample_negatives(self, seed, epoch):
        pr = self._pairs
        H.philox_bpr_negatives(pr["u"], seed, epoch, self.numItem, pr["indptr"], pr["sitems"], 0, out=pr["n"])
        return pr["n"]

    def set_negatives(self, negs):
        self._pairs["n"].copy_(torch.as_tensor(np.ascontiguousarray(negs, dtype=np.int32)))

    # ---- training -------------------------------------------------------------------------------
    def train_steps(self, batch_indices, batch_size, losses=None, arrays=None):
        """Enqueues len(batch_indices) training steps over the resident triplets; returns the device
        tensor of per-step mean losses (no host sync).  arrays: dict u / p / n / total to train on instead of the
        resident frame (fit passes this rank's slice of every global batch under data parallelism).  In peer mode
        every listed batch must be full (the cooperative launch runs the same number of samples on every rank)."""
        pr = arrays if arrays is not None else self._pairs
        k = len(batch_indices)
        if losses is None:
            losses = torch.empty(k, dtype=torch.float32, device=self.device)
        idx = (C.c_int64 * k)(*[int(b) for b in batch_indices])
        us, it = self.user.c_struct(), self.item.c_struct()
        if self.peer is not None:
            # mirrored data parallelism: one cooperative launch per rank runs all k steps, cross-GPU barriers and
            # the reduce-scatter + Adam + all-gather over NVLink peer memory included (csrc/bpr.cu)
            N.check(N.lib().brk_bpr_train_steps_dp(N.ctx(self.device), C.byref(us), C.byref(it), N.ptr(pr["u"]),
                                                   N.ptr(pr["p"]), N.ptr(pr["n"]), pr["total"], batch_size, idx, k,
                                                   self.optimizer.h, C.byref(self.peer.desc), N.ptr(self.optimizer.state),
                                                   N.ptr(losses), N.stream_ptr()), "brk_bpr_train_steps_dp")
            return losses
        N.check(N.lib().brk_bpr_train_steps(N.ctx(self.device), C.byref(us), C.byref(it), N.ptr(pr["u"]),
                                            N.ptr(pr["p"]), N.ptr(pr["n"]), pr["total"], batch_size, idx, k,
                                            self.optimizer.h, 1 if self.optimizer.sparse == "lazy" else 0,
                                            N.ptr(self.optimizer.state), N.ptr(losses), N.stream_ptr()),
                "brk_bpr_train_steps")
        return losses

    @staticmethod
    def pack_host_batches(users, items, batch_size):
        """Batch-major pinned host layout [n_batches, 2, batch] (each batch's user ids, then its item ids; the
        last block zero-padded): what a loader producing ({"user": ids, "item": ids}) batches writes
        (NeuMFModel.py:111-117).  With it train_steps_from_host moves each step's inputs with ONE copy."""
        users = np.ascontiguousarray(users, dtype=np.int32); items = np.ascontiguousarray(items, dtype=np.int32)
        nb = (len(users) + batch_size - 1) // batch_size
        packed = torch.zeros((nb, 2, batch_size), dtype=torch.int32).pin_memory()
        flat = packed.numpy()
        full = len(users) // batch_size
        flat[:full, 0, :] = users[:full * batch_size].reshape(full, batch_size)
        flat[:full, 1, :] = items[:full * batch_size].reshape(full, batch_size)
        if full < nb:
            r = len(users) - full * batch_size
            flat[full, 0, :r] = users[full * batch_size:]; flat[full, 1, :r] = items[full * batch_size:]
        packed.total = len(users)
        return packed

    def train_steps_from_host(self, u_host, p_host, batch_indices, batch_size, sampler_seed, epoch, losses_host=None):
        """End-to-end steps from page-locked HOST id arrays (torch CPU int32 tensors, pinned): H2D, device
        negative sampling, fused step, Adam and loss D2H are all enqueued by ONE C call; returns the pinned
        host loss tensor (valid after a stream synchronize).  Needs set_training_pairs() for the sampler's
        positive lists.  u_host may be a pack_host_batches() tensor (then p_host is None)."""
        pr = self._pairs
        k = len(batch_indices)
        dev = self.device
        if p_host is None:                                  # batch-major [n_batches, 2, batch]
            total, stride = int(u_host.total), 2 * batch_size
            u_ptr, p_ptr = u_host.data_ptr(), u_host.data_ptr() + 4 * batch_size
        else:
            total, stride = u_host.numel(), batch_size
            u_ptr, p_ptr = u_host.data_ptr(), p_host.data_ptr()
        need = int(N.lib().brk_bpr_host_stage_ints(batch_size))
        if getattr(self, "_stage", None) is None or self._stage.numel() < need:
            self._stage = torch.empty(need, dtype=torch.int32, device=dev)
        d_losses = torch.empty(k, dtype=torch.float32, device=dev)
        if losses_host is None:
            losses_host = torch.empty(k, dtype=torch.float32).pin_memory()
        idx = (C.c_int64 * k)(*[int(b) for b in batch_indices])
        us, it = self.user.c_struct(), self.item.c_struct()
        N.check(N.lib().brk_bpr_train_steps_host(
            N.ctx(dev), C.byref(us), C.byref(it), C.c_void_p(u_ptr), C.c_void_p(p_ptr),
            total, batch_size, stride, idx, k, sampler_seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, self.numItem,
            N.ptr(pr["indptr"]), N.ptr(pr["sitems"]), self.optimizer.h, 1 if self.optimizer.sparse == "lazy" else 0,
            N.ptr(self.optimizer.state), N.ptr(self._stage), N.ptr(d_losses), C.c_void_p(losses_host.data_ptr()),
            C.cast(C.byref(self.peer.desc), C.c_void_p) if self.peer is not None else None,
            N.stream_ptr()), "brk_bpr_train_steps_host")
        self._d_losses = d_losses            # keep alive until the stream has consumed it
        return losses_host

    def train_steps_mapped(self, u_host, p_host, batch_indices, batch_size, sampler_seed, epoch, losses_host=None):
        """Zero-copy variant of train_steps_from_host: the pinned host id arrays stay where they are, ONE
        cooperative launch runs every step and pulls each step's ids over PCIe itself; per-step losses are
        stored straight into the pinned `losses_host` (valid after a stream synchronize)."""
        pr = self._pairs
        k = len(batch_indices)
        if losses_host is None:
            losses_host = torch.empty(k, dtype=torch.float32).pin_memory()
        idx = (C.c_int64 * k)(*[int(b) for b in batch_indices])
        us, it = self.user.c_struct(), self.item.c_struct()
        N.check(N.lib().brk_bpr_train_steps_mapped(
            N.ctx(self.device), C.byref(us), C.byref(it), C.c_void_p(u_host.data_ptr()), C.c_void_p(p_host.data_ptr()),
            u_host.numel(), batch_size, idx, k, sampler_seed & 0xFFFFFFFF, epoch & 0xFFFFFFFF, self.numItem,
            N.ptr(pr["indptr"]), N.ptr(pr["sitems"]), self.optimizer.h, N.ptr(self.optimizer.state),
            C.c_void_p(losses_host.data_ptr()), N.stream_ptr()), "brk_bpr_train_steps_mapped")
        return losses_host

    def train_on_batch(self, u, p, n, loss_out=None):
        """One step on device id tensors; returns the device loss scalar (local-batch mean).
        Under torch.distributed this is the mirrored synchronous step of RModel.py:119-121: each rank
        trains its own slice, gradients are scaled by 1/(world * batch) and summed by one all-reduce,
        every rank applies the same Adam step."""
        w = D.world_size()
        if self.peer is not None:
            # one cooperative launch: fused fwd/bwd + cross-GPU reduce-scatter / Adam / all-gather
            if loss_out is None:
                loss_out = torch.empty(1, dtype=torch.float32, device=self.device)
            idx = (C.c_int64 * 1)(0)
            us, it = self.user.c_struct(), self.item.c_struct()
            N.check(N.lib().brk_bpr_train_steps_dp(N.ctx(self.device), C.byref(us), C.byref(it), N.ptr(H._i32(u, "u")),
                                                   N.ptr(H._i32(p, "p")), N.ptr(H._i32(n, "n")), u.numel(), u.numel(), idx, 1,
                                                   self.optimizer.h, C.byref(self.peer.desc), N.ptr(self.optimizer.state),
                                                   N.ptr(loss_out), N.stream_ptr()), "brk_bpr_train_steps_dp")
            return loss_out
        loss = H.bpr_fwd_bwd(self.user, self.item, u, p, n, loss_out=loss_out, global_batch=w * u.numel() if w > 1 else 0)
        self.apply_gradients()
        return loss

    def apply_gradients(self):
        """Optimizer step on the accumulated gradients (data-parallel aware)."""
        if self.peer is not None:
            self.peer.adam_step(self.optimizer.h, self.optimizer.state)
            return
        if D.world_size() > 1:
            if self.optimizer.sparse == "lazy":
                raise NotImplementedError("mirrored data parallelism uses the dense (Keras) Adam pass")
            D.all_reduce_sum_(self.grad_arena)
        self.optimizer.apply([self.user, self.item])

    def fit(self, X, y=None, batch_size=64, epochs=1, shuffle=True, sampler_seed=7, verbose=0, initial_epoch=0):
        """Keras-like fit (BPRModel.py:109).  X: dict with 'customerId_input', 'pProduct_input' and
        optionally 'nProduct_input'; without the latter a fresh Philox negative is drawn per positive
        per epoch.  y is ignored exactly as identityLoss ignores it (BPRModel.py:125-126).
        Batches are contiguous slices of the given row order; with shuffle=True the batch ORDER is
        permuted per epoch (seeded), which is what tf.data .batch().shuffle() does in the reference's
        other pipeline (NeuMFModel.py:117-121)."""
        if 'user_input' in X:                                   # input names of the script version (bpr.py:215-217)
            X = {'customerId_input': X['user_input'], 'pProduct_input': X['positive_item_input'],
                 'nProduct_input': X.get('negative_item_input')}
        users = np.asarray(X['customerId_input']); pos = np.asarray(X['pProduct_input'])
        self.set_training_pairs(users, pos)
        fixed_neg = X.get('nProduct_input')
        if fixed_neg is not None:
            self.set_negatives(fixed_neg)
        total = self._pairs["total"]
        n_batches = (total + batch_size - 1) // batch_size
        rng = np.random.Generator(np.random.Philox(key=sampler_seed + 1000003))
        W = D.world_size()
        if W > 1:
            return self._fit_data_parallel(batch_size, epochs, shuffle, sampler_seed, verbose, initial_epoch, fixed_neg, rng)
        for e in range(initial_epoch, initial_epoch + epochs):
            if fixed_neg is None:
                self.sample_negatives(sampler_seed, e)
            order = rng.permutation(n_batches) if shuffle else np.arange(n_batches)
            losses = self.train_steps(order, batch_size)
            # Keras reports the running mean of the per-batch losses
            mean = float(losses.double().mean().item())
            self.history["loss"].append(mean)
            if verbose:
                print(f"epoch {e + 1}: loss {mean:.6f}")
        return self

    def _fit_data_parallel(self, batch_size, epochs, shuffle, sampler_seed, verbose, initial_epoch, fixed_neg, rng):
        """fit under torch.distributed -- what MultiWorkerMirroredStrategy does with an auto-sharded dataset
        (RModel.py:119-121): `batch_size` stays the GLOBAL batch, rank r trains rows [r B/W, (r+1) B/W) of every global
        batch, gradients are scaled by 1/B and summed, every rank applies the same Adam step.  Same frame, same
        sampler stream and same batch order on every rank (all seeded), so W GPUs reproduce the single-GPU run up to
        summation order.  The ragged last batch goes through the per-step path with unequal slices."""
        W, r = D.world_size(), D.rank()
        if batch_size % W:
            raise ValueError(f"batch_size {batch_size} is the global batch: it must be a multiple of the {W} ranks")
        pr = self._pairs
        total, lb = pr["total"], batch_size // W
        nfull, n_batches = total // batch_size, (total + batch_size - 1) // batch_size
        dev = self.device
        sel = (torch.arange(nfull, device=dev).view(-1, 1) * batch_size + r * lb + torch.arange(lb, device=dev).view(1, -1)).reshape(-1)
        local = dict(u=pr["u"][sel].contiguous(), p=pr["p"][sel].contiguous(), n=None, total=nfull * lb)
        D.barrier()                                             # nobody enters a cross-GPU wait while a rank is still staging
        for e in range(initial_epoch, initial_epoch + epochs):
            if fixed_neg is None:
                self.sample_negatives(sampler_seed, e)           # counter = position in the GLOBAL frame: independent of W
            local["n"] = pr["n"][sel].contiguous()
            order = rng.permutation(n_batches) if shuffle else np.arange(n_batches)
            parts = []
            k = 0
            while k < len(order):                                # runs of full batches -> one launch; the ragged one on its own
                if order[k] == nfull:
                    parts.append(self._ragged_global_batch(nfull * batch_size, total - nfull * batch_size).view(1))
                    k += 1
                    continue
                j = k
                while j < len(order) and order[j] != nfull:
                    j += 1
                parts.append(self._train_steps_local(order[k:j], lb, local, batch_size))
                k = j
            losses = torch.cat(parts).double()
            if self.peer is not None:
                self.peer.check()
            mean = losses.mean().view(1)
            D.all_reduce_sum_(mean)                              # equal local batches: global mean = mean of the local means
            mean = float(mean.item()) / W
            self.history["loss"].append(mean)
            if verbose and r == 0:
                print(f"epoch {e + 1}: loss {mean:.6f}")
        return self

    def _train_steps_local(self, batch_indices, lb, local, global_batch):
        if self.peer is not None:
            return self.train_steps(batch_indices, lb, arrays=local)
        losses = torch.empty(len(batch_indices), dtype=torch.float32, device=self.device)
        for k, b in enumerate(batch_indices):                   # NCCL fallback: one all-reduce of the flat arena per step
            s = slice(int(b) * lb, (int(b) + 1) * lb)
            H.bpr_fwd_bwd(self.user, self.item, local["u"][s], local["p"][s], local["n"][s], loss_out=losses[k:k + 1],
                          global_batch=global_batch)
            self.apply_gradients()
        return losses

    def _ragged_global_batch(self, first, count):
        """The last, partial global batch: rank r takes its local_slice of the `count` rows (possibly none), the
        gradient scale is 1/count; returns this rank's share of the batch loss scaled so that the ranks' values average
        to the global mean."""
        pr = self._pairs
        lo, hi = D.local_slice(count)
        loss = torch.zeros(1, dtype=torch.float32, device=self.device)
        if hi > lo:
            s = slice(first + lo, first + hi)
            H.bpr_fwd_bwd(self.user, self.item, pr["u"][s], pr["p"][s], pr["n"][s], loss_out=loss, global_batch=count)
            loss = loss * (float(hi - lo) * D.world_size() / float(count))
        self.apply_gradients()
        return loss.view(())

    # ---- inference ------------------------------------------------------------------------------
    def predict(self, X):
        """Model output = per-row triplet loss (BPRModel.py:63,144)."""
        dev = self.device
        u, p, n = (torch.as_tensor(np.ascontiguousarray(X[k], dtype=np.int32)).to(dev)
                   for k in ('customerId_input', 'pProduct_input', 'nProduct_input'))
        x = H.bpr_scores(self.user.w, self.item.w, u, p, n)
        return (1.0 - torch.sigmoid(x)).unsqueeze(1)

    def get_layer_weights(self, name):
        return {"user_embedding": self.user.w, "item_embedding": self.item.w}[name]

    def state_dict(self):
        """Collective under peer-mode data parallelism: the Adam moments are sharded over the ranks (every rank holds the
        slice it applies) and are gathered here; every rank must call it."""
        if self.peer is not None:
            self.peer.check()
            nu, ni = self.numUser * self.numFactor, self.numItem * self.numFactor
            m, v = self.peer.full_moments()
            shp_u, shp_i = (self.numUser, self.numFactor), (self.numItem, self.numFactor)
            return {"user": self.user.w.cpu(), "item": self.item.w.cpu(), "user_m": m[:nu].view(shp_u).cpu(),
                    "user_v": v[:nu].view(shp_u).cpu(), "item_m": m[nu:nu + ni].view(shp_i).cpu(),
                    "item_v": v[nu:nu + ni].view(shp_i).cpu(), "opt_state": self.optimizer.state.cpu()}
        return {"user": self.user.w.cpu(), "item": self.item.w.cpu(), "user_m": self.user.m.cpu(),
                "user_v": self.user.v.cpu(), "item_m": self.item.m.cpu(), "item_v": self.item.v.cpu(),
                "opt_state": self.optimizer.state.cpu()}

    def load_state_dict(self, sd):
        self.user.w.copy_(sd["user"]); self.item.w.copy_(sd["item"])
        if self.peer is not None:
            dev = self.device
            m = torch.zeros(self.peer.n, dtype=torch.float32, device=dev); v = torch.zeros_like(m)
            nu, ni = self.numUser * self.numFactor, self.numItem * self.numFactor
            m[:nu] = sd["user_m"].reshape(-1).to(dev); m[nu:nu + ni] = sd["item_m"].reshape(-1).to(dev)
            v[:nu] = sd["user_v"].reshape(-1).to(dev); v[nu:nu + ni] = sd["item_v"].reshape(-1).to(dev)
            self.peer.load_moments(m, v)
        else:
            self.user.m.copy_(sd["user_m"]); self.user.v.copy_(sd["user_v"])
            self.item.m.copy_(sd["item_m"]); self.item.v.copy_(sd["item_v"])
        self.optimizer.state.copy_(sd["opt_state"])


def bpr_predict(model, user_id, item_ids, user_layer='user_embedding', item_layer='item_embedding'):
    """bpr.py:122-133: scores of one user against item_ids (user vector times item matrix)."""
    dev = model.device
    item_ids = torch.as_tensor(np.ascontiguousarray(item_ids, dtype=np.int32)).to(dev)
    rows = H.gather_rows(model.get_layer_weights(item_layer), item_ids)
    uvec = model.get_layer_weights(user_layer)[int(user_id)]
    return (rows * uvec).sum(-1)


def identity_loss(_, y_pred):
    """bpr.py:136-138."""
    return torch.mean(y_pred)


def bpr_triplet_loss(X):
    """bpr.py:141-157: 1 - sigmoid(<u, p> - <u, n>) per row; the script's argument order is [positive, negative, user]
    (the class version BPRModel.bprTripletLoss takes [user, positive, negative])."""
    positive_item_latent, negative_item_latent, user_latent = X
    pos = (user_latent * positive_item_latent).sum(-1, keepdim=True)
    neg = (user_latent * negative_item_latent).sum(-1, keepdim=True)
    return 1.0 - torch.sigmoid(pos - neg)


def out_shape(shapes):
    """bpr.py:160-161."""
    return shapes[0]


def build_model(num_users: int, num_items: int, latent_dim: int, **kw):
    """bpr.py:164-192: user table + ONE item table shared by the positive and the negative input, output = the
    per-row triplet loss.  Returns the fused device model (BPRNet); its fit takes the script's input names
    ('user_input', 'positive_item_input', 'negative_item_input', bpr.py:215-217) as well as the class version's."""
    return BPRNet(num_users, num_items, latent_dim, **kw)


def rating_triplets(user_ids, movie_ids, ratings, threshold=3):
    """The explicit-rating triplet frame of the script version (bpr.py:96-110): for every user, in order of first
    appearance, each positively rated item (rating > threshold) paired with each negatively rated one
    (rating <= threshold), positives outer / negatives inner, both in file order; users lacking either kind are
    skipped and reported.  Returns (user, positive, negative) int32 arrays -- the customerId_input / pProduct_input /
    nProduct_input columns BPRNet.fit takes (bpr.py:215-217) -- and the list of skipped users.  Host NumPy: input preparation, not the hot path."""
    u = np.asarray(user_ids); m = np.asarray(movie_ids); r = np.asarray(ratings)
    if not (len(u) == len(m) == len(r)):
        raise ValueError("user_ids, movie_ids and ratings differ in length")
    order = np.argsort(u, kind="stable")                          # rows of one user stay in file order
    su = u[order]
    starts = np.flatnonzero(np.r_[True, su[1:] != su[:-1]]) if len(su) else np.zeros(0, np.int64)
    ends = np.r_[starts[1:], len(su)]
    first_row = order[starts] if len(su) else starts
    uu, pp, nn, without = [], [], [], []
    for g in np.argsort(first_row, kind="stable"):               # users in order of first appearance (.unique())
        rows = order[starts[g]:ends[g]]
        pos = m[rows][r[rows] > threshold]; neg = m[rows][r[rows] <= threshold]
        if len(pos) == 0 or len(neg) == 0:
            without.append(su[starts[g]].item())
            continue
        uu.append(np.full(len(pos) * len(neg), su[starts[g]]))
        pp.append(np.repeat(pos, len(neg))); nn.append(np.tile(neg, len(pos)))
    cat = lambda parts: np.concatenate(parts).astype(np.int32) if parts else np.zeros(0, np.int32)
    return cat(uu), cat(pp), cat(nn), without


def _rank_eval(model, ground_truth, items, k, user_layer='user_embedding', item_layer='item_embedding'):
    """(auc [R], ap_at_k [R]) float64 NumPy arrays for the (user, true items) rows of ground_truth: fp32 scores of
    every user against `items` (one SGEMM per chunk of users: bpr_predict for all of them), then ONE counting kernel
    per chunk (brk_rank_eval_rows) instead of sklearn's roc_auc_score and a Python sort of the catalog per user."""
    dev = model.device
    rows = [(int(u), list(t)) for u, t in ground_truth]
    items = list(items)
    pos_of = {}
    for j, it in enumerate(items):
        pos_of.setdefault(it, j)                                   # list.index: the first occurrence
    R, I = len(rows), len(items)
    auc = np.full(R, np.nan); ap = np.full(R, np.nan)
    if R == 0 or I == 0:
        return auc, ap
    indptr = np.zeros(R + 1, dtype=np.int64)
    cols, alen = [], np.zeros(R, dtype=np.int32)
    for r, (u, true_items) in enumerate(rows):
        try:
            c = sorted({pos_of[t] for t in true_items})
        except KeyError as e:
            raise ValueError(f"{e.args[0]} is not in list") from None     # items.index(p) in the reference
        cols.extend(c); indptr[r + 1] = len(cols); alen[r] = len(true_items)
    W_u, W_i = model.get_layer_weights(user_layer), model.get_layer_weights(item_layer)
    d = W_u.shape[1]
    item_rows = H.gather_rows(W_i, torch.as_tensor(np.asarray(items, dtype=np.int32)).to(dev))      # [I, d]
    users = torch.as_tensor(np.asarray([u for u, _ in rows], dtype=np.int32)).to(dev)
    cols_d = torch.as_tensor(np.asarray(cols if cols else [0], dtype=np.int32)).to(dev)
    alen_d = torch.from_numpy(alen).to(dev)
    rank_ws = torch.empty(max(len(cols), 1), dtype=torch.int32, device=dev)
    part_ws = torch.empty(max(len(cols), 1), dtype=torch.float64, device=dev)
    out = torch.empty((R, 2), dtype=torch.float64, device=dev)
    chunk = max(1, min(R, (1 << 26) // I))                       # <= 256 MiB of fp32 scores per pass
    scores = torch.empty((chunk, I), dtype=torch.float32, device=dev)
    lib, ctx = N.lib(), N.ctx(dev)
    for a in range(0, R, chunk):
        b = min(R, a + chunk)
        uv = H.gather_rows(W_u, users[a:b])                      # [b - a, d]
        N.check(lib.brk_sgemm(ctx, N.ptr(uv), N.ptr(item_rows), N.ptr(scores), None, b - a, I, d, d, d, I, 0, 1, 1.0, 0,
                              N.stream_ptr()), "brk_sgemm")
        ip = torch.from_numpy(indptr[a:b + 1] - indptr[a]).to(dev)
        off = int(indptr[a])
        N.check(lib.brk_rank_eval_rows(ctx, N.ptr(scores), b - a, I, N.ptr(ip), N.ptr(cols_d[off:]), N.ptr(alen_d[a:b]), int(k),
                                       N.ptr(rank_ws[off:]), N.ptr(part_ws[off:]), N.ptr(out[a:b]), N.stream_ptr()),
                "brk_rank_eval_rows")
    o = out.cpu().numpy()
    return o[:, 0], o[:, 1]


def full_auc(model, ground_truth, items) -> float:
    """bpr.py:230-253: mean over the users with a non-empty true list of the AUC of that user's scores against the
    whole item list (ties count half, as sklearn's roc_auc_score).  ground_truth: iterable of (user_id, true items)."""
    rows = [(u, t) for u, t in ground_truth]
    auc, _ = _rank_eval(model, rows, items, 1)
    scores = [a for a, (_, t) in zip(auc, rows) if len(t)]
    if any(np.isnan(a) for a in scores):
        raise ValueError("Only one class present in y_true. ROC AUC score is not defined in that case.")   # sklearn's
    return sum(scores) / len(scores)                              # ZeroDivisionError when nobody has a true item


def mean_average_precision_k(model, ground_truth, items, k=100) -> float:
    """bpr.py:256-289: mean over users of average precision at k over the catalog sorted by score (stable: the
    earlier item first among equal scores), each divided by min(len(actual), k)."""
    rows = [(u, t) for u, t in ground_truth]
    if any(len(t) == 0 for _, t in rows):
        raise ZeroDivisionError("float division by zero")         # score / min(len(actual), k)
    _, ap = _rank_eval(model, rows, items, k)
    return float(np.mean(ap))


class BPRModel(RModel):
    def __init__(self, workDir=None):
        super().__init__('BPRModel', workDir)
        self._trainDf = None
        self._productIds: list = []
        self._results: list = []
        self.sparseAdam = "keras"

    @property
    def results(self) -> list:
        return self._results

    @results.setter
    def results(self, value: list):
        self._results = value

    @property
    def productIds(self) -> list:
        return self._productIds

    @productIds.setter
    def productIds(self, value: list):
        self._productIds = value

    @property
    def trainDf(self):
        return self._trainDf

    @trainDf.setter
    def trainDf(self, value):
        self._trainDf = value

    def compileModel(self, distributedConfig, numUser: int, numItem: int, numFactor: int):
        """Returns (model, strategy) like BPRModel.py:49,74; Adam(1e-3) as :70."""
        self.model = BPRNet(numUser, numItem, numFactor, seed=self.seed, learning_rate=1e-3,
                            sparse_adam=self.sparseAdam)
        return self.model, None

    def train(self, path, rowLimit, metricDict: dict = None, distributedConfig=None):
        self.batchSize = 64                                              # BPRModel.py:77
        numItem, numUser, (users, items) = self.readData(path, rowLimit)
        (trU, trI), _ = synth.train_test_split(users, items, self.testSize, seed=self.splitSeed)
        self.trainDf = (trU, trI)
        customerIds = np.unique(trU)
        self.productIds = np.unique(trI).tolist()
        print('Having %s customers and %s products' % (len(customerIds), len(self._productIds)))
        self.compileModel(distributedConfig, int(customerIds.max()) + 1, int(max(self.productIds)) + 1,
                          self.numFactor)
        X = {'customerId_input': trU, 'pProduct_input': trI}
        self.model.fit(X, None, batch_size=self.batchSize, epochs=self.epochs, sampler_seed=self.samplerSeed)
        return {'result': 'completed', 'metrics': [self.model.history["loss"][-1]]}

    def checkpointMeta(self) -> dict:
        return {"model": self.modelName, "numUser": self.model.user.rows, "numItem": self.model.item.rows,
                "numFactor": self.model.user.d, "productIds": [int(x) for x in self._productIds]}

    def buildFromMeta(self, meta: dict):
        self.compileModel(None, meta["numUser"], meta["numItem"], meta["numFactor"])
        self.productIds = list(meta.get("productIds", []))

    def predictForUsers(self, customerIds, numberOfItem=5, excludeSeen=False):
        """Top products for a batch of users (not in the reference, whose BPRModel stops after training; the scores
        are bpr_predict's, src/models/bpr.py:122-133): one bf16 tcgen05 scoring GEMM with the fused top-K epilogue
        over the whole catalog (hotpath.BruteForceIndex) -> [[(str(product), str(score)), ...] per user].
        excludeSeen=True leaves out each user's training pairs (trainDf), so a user with fewer unseen products than
        numberOfItem gets a shorter list; it needs the training pairs (ValueError after a checkpoint restore alone)."""
        if excludeSeen and self._trainDf is None:
            raise ValueError("excludeSeen needs the training pairs (trainDf), which this model does not hold")
        cu = np.asarray([int(c) for c in customerIds], dtype=np.int64)
        users = torch.as_tensor(cu.astype(np.int32)).to(self.model.device)
        if users.numel() and (int(users.min()) < 0 or int(users.max()) >= self.model.user.rows):
            raise ValueError("unknown customer id")
        if users.numel() == 0:
            return []
        index = H.BruteForceIndex(k=numberOfItem).index(self.model.item.w)
        q = H.gather_rows(self.model.user.w, users)
        if excludeSeen:
            # the requested users' rows of the per-user seen lists, in request order
            trU, trI = self._trainDf
            indptr, seen = synth.build_csr(trU, trI, self.model.user.rows)
            starts, lens = indptr[cu], indptr[cu + 1] - indptr[cu]
            ptr = np.zeros(len(cu) + 1, dtype=np.int64)
            np.cumsum(lens, out=ptr[1:])
            ids = seen[np.repeat(starts - ptr[:-1], lens) + np.arange(ptr[-1])]
            dev = self.model.device
            v, ix = index.query_with_exclusions(q, (torch.from_numpy(ptr).to(dev),
                                                    torch.from_numpy(ids.astype(np.int32)).to(dev)))
        else:
            v, ix = index(q)
        v, ix = v.cpu().numpy(), ix.cpu().numpy()
        return [[(str(int(j)), str(s)) for s, j in zip(v[r], ix[r]) if j >= 0] for r in range(len(v))]

    def extractPositivesNegatives(self, customerId) -> list:
        """Exhaustive (positive, non-interacted) pairs of one customer -- BPRModel.py:111-119."""
        trU, trI = self._trainDf
        existing = trI[trU == customerId].tolist()
        have = set(existing)
        entries = []
        for existingProductId in existing:
            for productId in self._productIds:
                if productId not in have:
                    entries.append({'CUSTOMER_ID': customerId, 'pPRODUCT_ID': existingProductId,
                                    'nPRODUCT_ID': productId})
        return entries

    def outShape(self, shapes):
        return shapes[0]

    def identityLoss(self, _, y_pred):
        return torch.mean(y_pred)                                          # BPRModel.py:125-126

    def bprTripletLoss(self, X):
        """1 - sigmoid(<u,p> - <u,n>) on three [B,F] latent tensors -- BPRModel.py:128-144."""
        userLatent, positiveItemLatent, negativeItemLatent = X
        pos = (userLatent * positiveItemLatent).sum(-1, keepdim=True)
        neg = (userLatent * negativeItemLatent).sum(-1, keepdim=True)
        return 1.0 - torch.sigmoid(pos - neg)
