"""Two-tower retrieval model -- drop-in mirror of the reference's trainers/twoTower.py
(TwoTowerModel with the same constructor arguments and method names, splitTrainTest,
crossValidation).

Underneath: two embedding tables + two linear Dense layers resident in HBM; towers, in-batch softmax
(TFRS Retrieval semantics) or rdZero BCE, all gradients in csrc/twotower.cu; Keras Adagrad in
csrc/optim.cu; full-catalog scoring + top-K on tcgen05 (csrc/topk.cu); metrics in csrc/metrics.cu.

Differences from the reference, stated once:
  * `trainers.model_utils.getOptimizer` does not exist in the reference tree (twoTower.py:5); here
    compile() accepts hotpath.Adagrad / hotpath.Adam objects or the strings "Adagrad" / "Adam";
  * crossValidation takes in-memory folds (lists of dicts with the userKey / itemKey [/ resKey]
    columns) instead of prompting for SMB credentials (twoTower.py:130-134);
  * StringLookup: vocabulary entry j -> row j + 2 (0 mask, 1 OOV), as TF 2.3/2.4; looked up by a device hash
    table (csrc/pipeline.cu) for ids with an exact 64-bit key, by a host dictionary for longer strings.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _native as N
from . import distributed as D
from . import hotpath as H
from .topKmetrics import exclusion_pairs_csr, topKMetrics


class StringLookup:
    """tf.keras.layers.experimental.preprocessing.StringLookup(vocabulary=...) (twoTower.py:33,35)."""

    def __init__(self, vocabulary):
        self.vocabulary = list(vocabulary)
        self._map = {v: j + 2 for j, v in enumerate(self.vocabulary)}
        self._dev = None          # pipeline.Vocabulary (device hash table), built on first device lookup
        self._packable = True

    def __call__(self, values):
        return np.fromiter((self._map.get(v, 1) for v in values), dtype=np.int32, count=len(values))

    def lookup_device(self, values, device):
        """int32 device tensor of indices.  Ids that have an exact 64-bit key (integers, strings of <= 8 bytes --
        the reference's CUSTOMER_ID / MATERIAL codes, loadBinaryMovieLens.py:49) are mapped by the device hash table
        (csrc/pipeline.cu); longer strings keep the host dictionary (text handling, not the hot path)."""
        from . import pipeline as PL
        if self._packable:
            try:
                vals = np.asarray(list(values)) if not isinstance(values, np.ndarray) else values
                voc = np.asarray(self.vocabulary)
                kind = lambda a: "i" if a.dtype.kind in "iu" else "S"
                if len(vals) and len(voc) and kind(vals) != kind(voc):
                    raise TypeError("values and vocabulary are of different kinds")      # host dictionary decides
                keys = PL.pack_keys(vals)
                if self._dev is None:
                    self._dev = PL.Vocabulary(device)
                    self._dev.build(PL.pack_keys(voc), offset=2)
                    if self._dev.size != len(self.vocabulary):
                        raise ValueError("StringLookup vocabulary has duplicate entries")
                return self._dev.lookup(torch.from_numpy(keys.view(np.int64)).to(device), oov=1)
            except (ValueError, TypeError) as e:
                if "duplicate" in str(e):
                    raise
                if "different kinds" not in str(e):
                    self._packable = False
        return torch.from_numpy(self(values)).to(device)


class Tower:
    def __init__(self, rows, E, S, rng, device):
        self.E, self.S = E, S
        self.emb = H.Table(torch.from_numpy(H.keras_embedding_init(rows, E, rng)).to(device), slots=1,
                           slot_init=H.Adagrad.INITIAL_ACCUMULATOR)
        self._W0 = None

    def init_dense(self, rng, device):
        lim = np.sqrt(6.0 / (self.E + self.S))
        W = rng.uniform(-lim, lim, size=(self.E, self.S)).astype(np.float32)
        flat = np.concatenate([W.reshape(-1), np.zeros(self.S, np.float32)])
        pad = (-len(flat)) % 4
        self.dense = H.Table(torch.from_numpy(np.pad(flat, (0, pad))).to(device).view(1, -1), slots=1, touched=False,
                             slot_init=H.Adagrad.INITIAL_ACCUMULATOR)

    def c_struct(self):
        return N.brk_tower(self.emb.c_struct(), self.dense.c_struct(), self.E, self.S)

    @property
    def W(self):
        return self.dense.w.view(-1)[:self.E * self.S].view(self.E, self.S)

    @property
    def b(self):
        return self.dense.w.view(-1)[self.E * self.S:self.E * self.S + self.S]


class GlobalNegatives:
    """Global in-batch negatives for data-parallel two-tower training (brk_twotower_step_global): every rank's queries
    are scored against the candidates of the whole global batch, so G GPUs on a global batch compute the one-GPU loss
    and gradients of that batch, up to summation order.

    Holds every rank's candidate block [cap, S], id block [4 + cap] (header {count, S}, then ids) and dc-partial slot
    [n_cap, S]: symmetric (NVLink peer-mapped) buffers with a PeerBarrier between the phases in a multi-GPU run, or G
    local buffers when one process emulates G ranks on one GPU.  Buffers grow on demand; a growth is collective, and
    every rank sees the same split, so all ranks grow at the same step."""

    def __init__(self, G, rank, E, S, device, emulate, barrier=None):
        self.G, self.rank, self.E, self.S, self.device, self.emulate = int(G), int(rank), int(E), int(S), device, bool(emulate)
        self.cap = self.n_cap = 0
        self.err = torch.zeros(1, dtype=torch.int32, device=device)
        self.barrier = barrier
        if not self.emulate and barrier is None:
            from .sharded import PeerBarrier
            self.barrier = PeerBarrier(device)
        self._ws = {}

    def _grow(self, cap, n):
        if cap <= self.cap and n <= self.n_cap:
            return
        cap, n = max(cap, self.cap, 1), max(n, self.n_cap, 1)
        dev, S = self.device, self.S
        sizes = (cap * S, 4 + cap, n * S)
        if self.emulate:
            bufs = [[torch.zeros(k, dtype=dt, device=dev) for k, dt in zip(sizes, (torch.float32, torch.int32, torch.float32))]
                    for _ in range(self.G)]
            self._bufs = bufs
            self.ptrs = [[b[k].data_ptr() for b in bufs] for k in range(3)]
        else:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm_mem
            torch.cuda.synchronize(dev)
            dist.barrier()                                   # no peer still reads the buffers being replaced
            mine = [symm_mem.empty(k, dtype=dt, device=dev) for k, dt in zip(sizes, (torch.float32, torch.int32, torch.float32))]
            hs = [symm_mem.rendezvous(b, dist.group.WORLD.group_name) for b in mine]
            for b in mine:
                b.zero_()
            self._bufs, self._handles = mine, hs
            self.ptrs = [list(h.buffer_ptrs) for h in hs]
            torch.cuda.synchronize(dev)
            dist.barrier()
        self.c_all = torch.empty(n * S, dtype=torch.float32, device=dev)
        self.ids_all = torch.empty(n, dtype=torch.int32, device=dev)
        self.cap, self.n_cap = cap, n

    def _struct(self, r, counts):
        g = N.brk_twotower_global()
        off = 0
        for p in range(self.G):
            g.cand[p], g.ids[p], g.slot[p] = self.ptrs[0][p], self.ptrs[1][p], self.ptrs[2][p]
            g.offset[p], g.count[p] = off, counts[p]
            off += counts[p]
        g.cap, g.n_cap = self.cap, self.n_cap
        g.c_all, g.ids_all, g.err = self.c_all.data_ptr(), self.ids_all.data_ptr(), self.err.data_ptr()
        g.world, g.rank = self.G, r
        return g

    def _workspace(self, r, b, n):
        have = self._ws.get(r)
        if have is None or have[0] < b or have[1] < n:
            dev, E, S = self.device, self.E, self.S
            f = lambda k: torch.empty(max(k, 1), dtype=torch.float32, device=dev)
            bufs = dict(eu=f(b * E), ei=f(b * E), deu=f(b * E), dei=f(b * E), q=f(b * S), dq=f(b * S), dc=f(b * S),
                        scores=f(b * n), acc=torch.zeros(1, dtype=torch.float64, device=dev))
            have = self._ws[r] = (b, n, bufs)
        b_ = have[2]
        return N.brk_twotower_workspace(b_["eu"].data_ptr(), b_["ei"].data_ptr(), b_["q"].data_ptr(), None, b_["dq"].data_ptr(),
                                        b_["dc"].data_ptr(), b_["scores"].data_ptr(), None, b_["acc"].data_ptr(),
                                        b_["deu"].data_ptr(), b_["dei"].data_ptr())

    def step(self, user, item, shards, parts, counts, tensor_cores, loss_out):
        """Forward and backward of one step (no optimizer).  parts: {rank: (u, i)} int32 slices of the ranks this process
        drives (every rank under emulation, else this one); counts: the G slice sizes of the global batch, the same on
        every rank.  shards(r): the brk_twotower_shards of rank r, or None for mirrored tables.  loss_out receives the
        sum of the driven ranks' losses."""
        counts = [int(c) for c in counts]
        if len(counts) != self.G or min(counts) < 0:
            raise ValueError(f"global negatives: split {counts} is not {self.G} slice sizes")
        for r, (u, _) in parts.items():
            if u.numel() != counts[r]:
                raise ValueError(f"global negatives: rank {r} passes {u.numel()} rows, the split says {counts[r]}")
        n = sum(counts)
        self._grow(max(counts), n)
        lib, ctx, st = N.lib(), N.ctx(self.device), N.stream_ptr()
        mode = 0x100 if tensor_cores else 0
        losses = loss_out if len(parts) == 1 else torch.zeros(len(parts), dtype=torch.float32, device=self.device)
        calls = [(r, self._struct(r, counts), self._workspace(r, counts[r], n), shards(r), u, i, losses[k:k + 1])
                 for k, (r, (u, i)) in enumerate(parts.items())]
        for phase in (0, 1, 2):
            for r, g, ws, sh, u, i, lo in calls:
                N.check(lib.brk_twotower_step_global(ctx, phase, C.byref(user), C.byref(item), C.byref(sh) if sh is not None else None,
                                                     C.byref(g), N.ptr(u), N.ptr(i), mode, C.byref(ws), N.ptr(lo), st),
                        "brk_twotower_step_global")
            if phase < 2 and self.barrier is not None:
                self.barrier()                               # every rank's phase is complete before any rank reads it
        if len(parts) != 1:
            torch.sum(losses, 0, keepdim=True, out=loss_out)
        return loss_out

    def check(self):
        if self.barrier is not None:
            self.barrier.check()
        err = int(self.err.item())
        if err:
            self.err.zero_()
            raise RuntimeError(f"global negatives: rank {err - 1}'s published slice differs from the split this rank was "
                               "given (the ranks passed different splits, or a rank skipped a step)")


def check_retrieval_options(rdZero, global_negatives, temperature, streamingFrequency, candidate_probs):
    """The checks of tfrs Retrieval's options that TwoTowerModel and sharded.ShardedTwoTowerNet share (ValueError).
    candidate_probs: the caller also supplies candidate probabilities.  Returns the estimator's alpha (streamingFrequency
    True: 0.01), or None without the estimator."""
    if rdZero:
        raise ValueError("temperature / candidateProbKey / weightKey / streamingFrequency need the in-batch softmax: "
                         "rdZero has no in-batch negatives")
    if global_negatives:
        raise ValueError("temperature / candidateProbKey / weightKey / streamingFrequency are not offered with "
                         "global_negatives: the probabilities would have to be published with the peers' candidate blocks")
    if temperature is not None and not (math.isfinite(float(temperature)) and float(temperature) > 0):
        raise ValueError(f"temperature must be finite and > 0, got {temperature}")
    if temperature is not None and not math.isfinite(1.0 / float(temperature)):
        raise ValueError(f"temperature {temperature} is too small: 1 / temperature is not finite")
    if streamingFrequency is None or streamingFrequency is False:
        return None
    if candidate_probs:
        raise ValueError("candidate probabilities (candidateProbKey, cand_prob) and streamingFrequency both give p: "
                         "pass one")
    alpha = 0.01 if streamingFrequency is True else float(streamingFrequency)
    if not 0.0 < alpha <= 1.0:
        raise ValueError(f"streamingFrequency (the estimator's alpha) must be in (0, 1], got {streamingFrequency}")
    return alpha


def check_sampled_options(sampledNegatives, rdZero, global_negatives, streamingFrequency, candidate_probs):
    """The checks of sampled negatives that TwoTowerModel and sharded.ShardedTwoTowerNet share (ValueError).  Returns M,
    the number of rows drawn per step (0: none).  candidate_probs: the caller also supplies candidate probabilities."""
    if sampledNegatives is None or sampledNegatives is False:
        return 0
    if isinstance(sampledNegatives, bool) or int(sampledNegatives) != sampledNegatives or int(sampledNegatives) < 1:
        raise ValueError(f"sampledNegatives must be an integer >= 1 (rows drawn per step), got {sampledNegatives!r}")
    if rdZero:
        raise ValueError("sampledNegatives needs the in-batch softmax: rdZero has no candidate columns")
    if global_negatives:
        raise ValueError("sampledNegatives is not offered with global_negatives: the draws would have to be published "
                         "with the peers' candidate blocks")
    if streamingFrequency is not None and streamingFrequency is not False:
        raise ValueError("sampledNegatives is not offered with streamingFrequency: the logQ correction of a mixed pool needs "
                         "each sampled column's probability under both routes")
    if candidate_probs:
        raise ValueError("sampledNegatives is not offered with candidate probabilities (candidateProbKey, cand_prob): the "
                         "logQ correction of a mixed pool needs each sampled column's probability under both routes")
    return int(sampledNegatives)


class SampledNegatives:
    """The sampler state of a model with sampledNegatives=M (brk_tt_sampled): the draws of the last training step (ids,
    int32 [M]) and the device counter of training steps (step, int64 [1]).  Rows are drawn from [2, item_rows): never
    StringLookup's mask row 0 or OOV row 1."""

    def __init__(self, M, item_rows, seed, replica, device):
        self.M, self.item_rows, self.seed, self.replica = int(M), int(item_rows), int(seed) & 0xFFFFFFFF, int(replica)
        self.ids = torch.zeros(self.M, dtype=torch.int32, device=device)
        self.step = torch.zeros(1, dtype=torch.int64, device=device)

    def c_struct(self):
        s = N.brk_tt_sampled()
        s.ids, s.step, s.count = self.ids.data_ptr(), self.step.data_ptr(), self.M
        s.lo, s.hi, s.rows = 2, self.item_rows, self.item_rows
        s.seed, s.replica = self.seed, self.replica
        return s


class TwoTowerModel:
    def __init__(self, embedDim, nbrItem, nbrUser, userKey, itemKey, usersId, itemsId, eval_batch_size=8000,
                 loss=None, rdZero=False, resKey=None, semb=100, seed=42, device=None, tensor_cores=False,
                 global_negatives=False, temperature=None, candidateProbKey=None, weightKey=None, streamingFrequency=None,
                 sampledNegatives=None):
        # sampledNegatives=M: mixed negative sampling (Yang et al., WWW 2020) -- every training step draws M item rows
        # uniformly from the catalog on the device and adds them as candidate columns shared by every row
        # (brk_twotower_train_step_sampled); evaluation stays the in-batch loss
        self.sampledNegatives = check_sampled_options(sampledNegatives, rdZero, global_negatives, streamingFrequency,
                                                      candidateProbKey is not None)
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        self.embedDim, self.nbrItem, self.nbrUser = embedDim, nbrItem, nbrUser
        self.userKey, self.itemKey, self.resKey = userKey, itemKey, resKey
        self.eval_batch_size, self.rdZero, self.semb = eval_batch_size, rdZero, semb
        # tensor_cores: Dense / in-batch products on tcgen05 with TF32 operands (csrc/gemm_tc.cu); fp32 FMA otherwise
        self.tensor_cores = bool(tensor_cores)
        # global_negatives: under torch.distributed every rank's queries take the candidates of the whole global batch as
        # negatives (GlobalNegatives) instead of its own slice's (the per-replica loss, MirroredStrategy's default)
        if global_negatives and rdZero:
            raise ValueError("global_negatives needs the in-batch softmax: rdZero has no in-batch negatives")
        self.global_negatives = bool(global_negatives)
        # tfrs.tasks.Retrieval(temperature=...) called with candidate_sampling_probability / sample_weight
        # (brk_twotower_step_retrieval): candidateProbKey / weightKey name columns of the batch info, as resKey does;
        # streamingFrequency=alpha (True: 0.01) estimates the candidate probabilities on the device instead (Yi et al.,
        # RecSys 2019, Algorithm 2), with one slot per item-table row owned by the model
        self._configure_retrieval(temperature, candidateProbKey, weightKey, streamingFrequency, nbrItem + 2)
        self._smp = SampledNegatives(self.sampledNegatives, nbrItem + 2, seed, D.rank(), self.device) \
            if self.sampledNegatives else None
        self.userTowerIn = StringLookup(usersId)
        self.itemTowerIn = StringLookup(itemsId)
        rng = np.random.Generator(np.random.Philox(key=seed))
        # draw order = oracle/twotower.py: Eu, Ei, Wu, Wi
        self.userTower = Tower(nbrUser + 2, embedDim, semb, rng, self.device)
        self.itemTower = Tower(nbrItem + 2, embedDim, semb, rng, self.device)
        self.userTower.init_dense(rng, self.device)
        self.itemTower.init_dense(rng, self.device)
        # mirrored data parallelism: the four gradient accumulators become views of ONE flat arena in NVLink peer-mapped
        # memory, summed over the ranks once per step by brk_allreduce_dense_peer (no NCCL call on the step's path)
        self.grad_arena = self._reducer = None
        if D.world_size() > 1:
            tabs = [self.userTower.emb, self.itemTower.emb, self.userTower.dense, self.itemTower.dense]
            sizes = [t.w.numel() for t in tabs]
            self.grad_arena, self._reducer = D.gradient_arena(sum(sizes), self.device)
            for t, v in zip(tabs, torch.split(self.grad_arena[:sum(sizes)], sizes)):
                t.g = v.view(t.rows, t.d)
        self._global = GlobalNegatives(D.world_size(), D.rank(), embedDim, semb, self.device, emulate=False) \
            if self.global_negatives and D.world_size() > 1 else None
        self.bruteForceLayer = None
        self._candidates = None
        self.optimizer = None
        self.computeLoss = self.computeLossRdZero if rdZero else self.computeLossTfrs
        self._ws_batch = 0
        self.history = {"loss": []}

    def _configure_retrieval(self, temperature, candidateProbKey, weightKey, streamingFrequency, item_rows):
        self.temperature, self.candidateProbKey, self.weightKey = temperature, candidateProbKey, weightKey
        if streamingFrequency is False:
            streamingFrequency = None
        self.streamingFrequency = streamingFrequency
        self._retrieval = any(x is not None for x in (temperature, candidateProbKey, weightKey, streamingFrequency))
        self._freq = None
        if not self._retrieval:
            return
        alpha = check_retrieval_options(self.rdZero, self.global_negatives, temperature, streamingFrequency,
                                        candidateProbKey is not None)
        if alpha is not None:
            if D.world_size() > 1:
                raise ValueError("streamingFrequency is single-process only: the estimator state is not shared across ranks")
            self._alpha = alpha
            dev = self.device
            self._freq = dict(last=torch.zeros(item_rows, dtype=torch.int64, device=dev),
                              gap=torch.zeros(item_rows, dtype=torch.float32, device=dev),
                              step=torch.zeros(1, dtype=torch.int64, device=dev))

    def _extras(self, info):
        """(candidate probabilities, sample weights) of a batch as float32 device tensors (None where not configured)."""
        n = len(info[self.itemKey])
        out = []
        for key in (self.candidateProbKey, self.weightKey):
            if key is None:
                out.append(None)
                continue
            v = torch.as_tensor(np.asarray(info[key], dtype=np.float32)).to(self.device)
            if v.numel() != n:
                raise ValueError(f"column {key!r} has {v.numel()} entries, the batch {n}")
            out.append(v)
        return tuple(out)

    def _rt(self, extras):
        """brk_tt_retrieval of one call, or None when the model has no retrieval options (the option-free kernels)."""
        if not self._retrieval:
            return None
        prob, weight = extras if extras is not None else (None, None)
        rt = N.brk_tt_retrieval()
        rt.cand_prob = prob.data_ptr() if prob is not None else None
        rt.row_weight = weight.data_ptr() if weight is not None else None
        rt.inv_temperature = 1.0 / float(self.temperature) if self.temperature is not None else 1.0
        if self._freq is not None:
            f = self._freq
            rt.last, rt.gap, rt.step, rt.rows = f["last"].data_ptr(), f["gap"].data_ptr(), f["step"].data_ptr(), f["gap"].numel()
            rt.alpha = self._alpha
        return rt

    # ---- Keras-like surface -----------------------------------------------------------------------
    def compile(self, optimizer="Adagrad", loss=None, learningRate=0.1):
        if isinstance(optimizer, str):
            name = optimizer.lower()
            if name == "adagrad":
                optimizer = H.Adagrad(learningRate)
            else:
                raise ValueError(f"two-tower training is built for Adagrad (twoTower.py:278-279), got {optimizer}")
        self.optimizer = optimizer
        return self

    def _workspace(self, B):
        if B > self._ws_batch:
            dev, S = self.device, self.semb
            f = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)
            n = B + self.sampledNegatives                      # item-side rows: the batch's, then the sampled ones
            self._bufs = dict(eu=f(B, self.embedDim), ei=f(n, self.embedDim), deu=f(B, self.embedDim),
                              dei=f(n, self.embedDim), q=f(B, S), c=f(n, S), dq=f(B, S),
                              dc=f(n, S), scores=f(B, n) if not self.rdZero else None,
                              ones=torch.ones(B, dtype=torch.float32, device=dev),
                              acc=torch.zeros(1, dtype=torch.float64, device=dev))
            self._ws_batch = B
        b = self._bufs
        return N.brk_twotower_workspace(*[b[k].data_ptr() if b[k] is not None else None
                                          for k in ("eu", "ei", "q", "c", "dq", "dc", "scores", "ones", "acc", "deu", "dei")])

    def _ids(self, info):
        dev = self.device
        return self.userTowerIn.lookup_device(info[self.userKey], dev), self.itemTowerIn.lookup_device(info[self.itemKey], dev)

    def _step(self, u, i, labels, training, loss_out=None, extras=None):
        B = u.numel()
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
        ws = self._workspace(max(B, 1))
        ut, it = self.userTower.c_struct(), self.itemTower.c_struct()
        rt = self._rt(extras)
        if training and self._smp is not None:               # evaluation draws nothing: the in-batch loss below
            smp = self._smp.c_struct()
            N.check(N.lib().brk_twotower_step_sampled(N.ctx(self.device), C.byref(ut), C.byref(it), N.ptr(u), N.ptr(i), B,
                                                      0x100 if self.tensor_cores else 0, C.byref(ws), N.ptr(loss_out),
                                                      N.stream_ptr(), C.byref(smp), C.byref(rt) if rt is not None else None),
                    "brk_twotower_step_sampled")
            return loss_out
        if rt is not None:
            N.check(N.lib().brk_twotower_step_retrieval(N.ctx(self.device), C.byref(ut), C.byref(it), N.ptr(u), N.ptr(i), N.ptr(i),
                                                        None, B, 0x100 if self.tensor_cores else 0, 1 if training else 0,
                                                        C.byref(ws), N.ptr(loss_out), N.stream_ptr(), C.byref(rt)),
                    "brk_twotower_step_retrieval")
            return loss_out
        N.check(N.lib().brk_twotower_step(N.ctx(self.device), C.byref(ut), C.byref(it), N.ptr(u), N.ptr(i), N.ptr(i),
                                          N.ptr(labels) if labels is not None else None, B,
                                          (1 if self.rdZero else 0) | (0x100 if self.tensor_cores else 0),
                                          1 if training else 0, C.byref(ws), N.ptr(loss_out), N.stream_ptr()),
                "brk_twotower_step")
        return loss_out

    def computeEmb(self, info):
        """(user embeddings [B,S], item embeddings [B,S]) -- twoTower.py:77-80."""
        u, i = self._ids(info)
        return self._tower_forward(self.userTower, u), self._tower_forward(self.itemTower, i)

    def _tower_forward(self, tower, ids):
        n = ids.numel()
        emb = torch.empty(n, tower.E, dtype=torch.float32, device=self.device)
        out = torch.empty(n, tower.S, dtype=torch.float32, device=self.device)
        t = tower.c_struct()
        N.check(N.lib().brk_tower_forward(N.ctx(self.device), C.byref(t), N.ptr(ids), n, N.ptr(emb), N.ptr(out),
                                          N.stream_ptr()), "brk_tower_forward")
        return out

    def computeLossTfrs(self, usersCaracteristics, itemCaracteristics, info):
        """In-batch softmax loss of already computed tower outputs (twoTower.py:82-83), forward only.  With the retrieval
        options, in the order of tfrs Retrieval.call: scores / temperature, minus log(clip(p, 1e-6, 1)) of each column,
        accidental hits masked, loss weighted per row; the estimator's probabilities are read, not updated."""
        scores = usersCaracteristics @ itemCaracteristics.T
        ids = torch.from_numpy(self.itemTowerIn(info[self.itemKey])).to(self.device)
        B = scores.shape[0]
        prob, weight = self._extras(info) if self._retrieval else (None, None)
        if self.temperature is not None:
            scores = scores / float(self.temperature)
        if self._freq is not None:
            gap = self._freq["gap"][ids.long()]
            prob = torch.where(gap >= 1.0, 1.0 / gap, torch.ones_like(gap))
        if prob is not None:
            scores = scores - torch.log(torch.clamp(prob, 1e-6, 1.0))[None, :]
        dup = (ids[:, None] == ids[None, :]).float() - torch.eye(B, device=self.device)
        scores = scores + dup * (float(np.finfo(np.float32).min) / 100.0)
        return torch.nn.functional.cross_entropy(scores, torch.arange(B, device=self.device), weight=weight, reduction="sum")

    def computeLossRdZero(self, usersCaracteristics, itemCaracteristics, info):
        y = torch.as_tensor(np.asarray(info[self.resKey], dtype=np.float32)).to(self.device)
        return torch.nn.functional.binary_cross_entropy_with_logits((usersCaracteristics * itemCaracteristics).sum(1), y)

    def _labels(self, info):
        if not self.rdZero:
            return None
        return torch.as_tensor(np.asarray(info[self.resKey], dtype=np.float32)).to(self.device)

    def train_step(self, info, split=None):
        """One fused forward/backward + Adagrad step; returns {"loss": device scalar} (twoTower.py:89-102).
        Under torch.distributed the replicas' SUM-reduced gradients are summed by one all-reduce per
        tower (MirroredStrategy sums per-replica gradients of a SUM-reduced loss).  With global_negatives, `info` is
        this rank's slice of the global batch and `split` the slice sizes of all ranks (default: equal slices)."""
        u, i = self._ids(info)
        return {"loss": self._train_ids(u, i, self._labels(info), split=split, extras=self._extras(info))}

    def _train_step_native(self, u, i, labels, loss_out=None, extras=None):
        """Step + Keras Adagrad in one library call (brk_twotower_train_step): ONE cooperative launch when the in-batch
        softmax step runs on the tensor cores and the batch fits on chip, the step + optimizer kernels otherwise."""
        B = u.numel()
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
        ws = self._workspace(B)
        ut, it = self.userTower.c_struct(), self.itemTower.c_struct()
        opt = self.optimizer
        rt = self._rt(extras)
        if self._smp is not None:
            smp = self._smp.c_struct()
            N.check(N.lib().brk_twotower_train_step_sampled(
                N.ctx(self.device), C.byref(ut), C.byref(it), N.ptr(u), N.ptr(i), B, 0x100 if self.tensor_cores else 0,
                C.byref(ws), float(opt.lr), float(opt.eps), int(opt.rows_threshold_bytes), N.ptr(loss_out), N.stream_ptr(),
                C.byref(smp), C.byref(rt) if rt is not None else None), "brk_twotower_train_step_sampled")
            return loss_out
        if rt is not None:
            N.check(N.lib().brk_twotower_train_step_retrieval(
                N.ctx(self.device), C.byref(ut), C.byref(it), N.ptr(u), N.ptr(i), N.ptr(i), None, B,
                0x100 if self.tensor_cores else 0, C.byref(ws), float(opt.lr), float(opt.eps), int(opt.rows_threshold_bytes),
                N.ptr(loss_out), N.stream_ptr(), C.byref(rt)), "brk_twotower_train_step_retrieval")
            return loss_out
        N.check(N.lib().brk_twotower_train_step(N.ctx(self.device), C.byref(ut), C.byref(it), N.ptr(u), N.ptr(i), N.ptr(i),
                                                N.ptr(labels) if labels is not None else None, B,
                                                (1 if self.rdZero else 0) | (0x100 if self.tensor_cores else 0), C.byref(ws),
                                                float(opt.lr), float(opt.eps), int(opt.rows_threshold_bytes), N.ptr(loss_out),
                                                N.stream_ptr()), "brk_twotower_train_step")
        return loss_out

    def _train_ids(self, u, i, labels, loss_out=None, split=None, extras=None):
        if self.optimizer is None:
            self.compile()
        if D.world_size() == 1 and u.numel() > 0 and isinstance(self.optimizer, H.Adagrad):
            return self._train_step_native(u, i, labels, loss_out, extras)
        if self._global is not None:                         # every rank calls, an empty slice included
            loss = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
            self._global.step(self.userTower.c_struct(), self.itemTower.c_struct(), lambda r: None,
                              {D.rank(): (u, i)}, split if split is not None else [u.numel()] * D.world_size(),
                              self.tensor_cores, loss)
        elif u.numel() > 0 or self._smp is not None:          # an empty slice still draws: the counters stay in step
            loss = self._step(u, i, labels, True, loss_out, extras)
        else:                                                # this rank's slice of a small global batch is empty
            loss = loss_out if loss_out is not None else torch.zeros(1, dtype=torch.float32, device=self.device)
            loss.zero_()
        if D.world_size() > 1:
            D.all_reduce_sum_(self.grad_arena, self._reducer)
            # the touched-row bitmasks are per rank: after the sum every rank applies the dense pass (rows nobody touched
            # have g == 0 and do not move under Adagrad)
            self.optimizer.apply([self.userTower.emb, self.itemTower.emb], dense=[self.userTower.dense, self.itemTower.dense],
                                 force_dense=True)
            return loss
        self.optimizer.apply([self.userTower.emb, self.itemTower.emb], dense=[self.userTower.dense, self.itemTower.dense])
        return loss

    def test_step(self, info):
        u, i = self._ids(info)
        return {"loss": self._step(u, i, self._labels(info), False, extras=self._extras(info))}

    def fit(self, dataset, epochs=1, verbose=0, graph=True):
        """dataset: iterable of info dicts (batches), replayed every epoch like a cached tf.data set.
        graph=True replays the training step as ONE CUDA graph launch per batch (single process, equal-sized batches
        except a shorter last one): at the reference's batch of 1000 the step is a chain of few-microsecond kernels
        and the per-kernel launch cost is the larger half of it (124 -> 70 us per step on B200)."""
        batches = list(dataset)
        # string -> index lookups and H2D of the ids once per fit, not once per step and epoch (the reference caches
        # its batched dataset too: trainSetCached, twoTower.py:197-198)
        staged = [(self._ids(info), self._labels(info), self._extras(info)) for info in batches]
        if D.world_size() > 1:
            # mirrored data parallelism: a batch of the dataset is the GLOBAL batch (MultiWorkerMirroredStrategy auto-shards
            # it); this rank trains its slice, with its slice's items as in-batch negatives (the per-replica loss) or, with
            # global_negatives, the items of the whole global batch, and the SUM-reduced gradients are summed over the
            # ranks (peer all-reduce in _train_ids)
            def mine(t):
                if t is None:
                    return None
                lo, hi = D.local_slice(t.numel())
                return t[lo:hi].contiguous()
            G = D.world_size()
            splits = [[(lambda s: s[1] - s[0])(D.local_slice(u.numel(), r, G)) for r in range(G)] for (u, _), _, _ in staged]
            staged = [((mine(u), mine(i)), mine(lab), tuple(mine(x) for x in ex)) for (u, i), lab, ex in staged]
            D.barrier()
        sizes = [u.numel() for (u, _), _, _ in staged]
        n_full = 0
        while n_full < len(sizes) and sizes[n_full] == sizes[0]:
            n_full += 1
        use_graph = bool(graph) and D.world_size() == 1 and n_full >= 4 and n_full >= len(sizes) - 1
        replay = None
        for e in range(epochs):
            losses = torch.zeros(max(len(staged), 1), dtype=torch.float32, device=self.device)
            if use_graph:
                # batch 0 runs eagerly (first-use initialisation of the library happens outside the capture), the other
                # full batches replay the graph, a shorter last batch runs eagerly again: same order, same arithmetic
                (u, i), lab, ex = staged[0]
                self._train_ids(u, i, lab, losses[0:1], extras=ex)
                if replay is None:
                    replay = self._capture_fit_graph(staged[:n_full])
                replay(losses, 1, n_full)
                rest = range(n_full, len(staged))
            else:
                rest = range(len(staged))
            for k in rest:
                (u, i), lab, ex = staged[k]
                self._train_ids(u, i, lab, losses[k:k + 1], split=splits[k] if D.world_size() > 1 else None, extras=ex)
            # one host sync per epoch: Keras reports the running mean of the per-batch losses
            self.history["loss"].append(float(losses.double().sum().item()) / max(len(staged), 1))
            if self._reducer is not None:
                self._reducer.check()                        # a peer all-reduce that timed out aborted its step: raise here
            if self._global is not None:
                self._global.check()
            if verbose:
                print(f"epoch {e + 1}: loss {self.history['loss'][-1]:.6f}")
        return self

    def _capture_fit_graph(self, full):
        """Captures `copy batch [pos] into the static id buffers -> fused step -> Adagrad -> store the loss at [pos] ->
        pos += 1` once; returns replay(losses, first, last) that runs batches first..last-1 of `full`."""
        dev = self.device
        all_u = torch.stack([u for (u, _), _, _ in full]); all_i = torch.stack([i for (_, i), _, _ in full])
        all_lab = torch.stack([lab for _, lab, _ in full]) if full[0][1] is not None else None
        # the retrieval columns (candidate probabilities, sample weights) are staged like the ids; the estimator's step
        # counter lives on the device, so every replay is the next step
        all_ex = [torch.stack([ex[k] for _, _, ex in full]) if full[0][2][k] is not None else None for k in range(2)]
        B = all_u.shape[1]
        cur_u, cur_i = torch.empty_like(all_u[0]), torch.empty_like(all_i[0])
        cur_lab = torch.empty_like(all_lab[0]) if all_lab is not None else None
        cur_ex = tuple(torch.empty_like(a[0]) if a is not None else None for a in all_ex)
        cur_loss = torch.zeros(1, dtype=torch.float32, device=dev)
        pos = torch.zeros(1, dtype=torch.int64, device=dev)
        sink = torch.zeros(len(full), dtype=torch.float32, device=dev)
        self._workspace(B)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            cur_u.copy_(all_u.index_select(0, pos)[0]); cur_i.copy_(all_i.index_select(0, pos)[0])
            if cur_lab is not None:
                cur_lab.copy_(all_lab.index_select(0, pos)[0])
            for a, c in zip(all_ex, cur_ex):
                if c is not None:
                    c.copy_(a.index_select(0, pos)[0])
            self._train_ids(cur_u, cur_i, cur_lab, cur_loss, extras=cur_ex)
            sink.index_copy_(0, pos, cur_loss)
            pos.add_(1)

        def replay(losses, first, last):
            pos.fill_(first)
            for _ in range(first, last):
                g.replay()
            losses[first:last].copy_(sink[first:last])
        self._fit_graph_keepalive = (g, all_u, all_i, all_lab, all_ex, cur_u, cur_i, cur_lab, cur_ex, cur_loss, pos, sink)
        return replay

    # ---- retrieval --------------------------------------------------------------------------------------
    def setCandidates(self, items, k):
        """BruteForce(k).index(itemTower(items), identifiers=items) -- twoTower.py:64-69."""
        items = list(items)
        vecs = []
        for s in range(0, len(items), self.eval_batch_size):
            ids = torch.from_numpy(self.itemTowerIn(items[s:s + self.eval_batch_size])).to(self.device)
            vecs.append(self._tower_forward(self.itemTower, ids))
        self._candidates = items
        self.bruteForceLayer = H.BruteForceIndex(k).index(torch.cat(vecs))
        return self

    def call(self, info):
        """userTower(info) -> BruteForce: (scores [U,k], identifiers [U,k] as list of lists) -- :60-62."""
        ids = torch.from_numpy(self.userTowerIn(list(info))).to(self.device)
        vals, idx = self.bruteForceLayer(self._tower_forward(self.userTower, ids))
        return vals, idx

    __call__ = call

    def predict(self, usersId, batch_size=5000, exclude=None):
        """(scores ndarray [U,k], identifiers list-of-lists [U][k]) like model.predict(usersId) at :230.  `exclude`:
        (user, item) pairs in raw ids to leave out of that user's list (items are matched against setCandidates);
        a user left with fewer than k candidates gets a shorter identifier list, its score row ends in -inf."""
        usersId = list(usersId)
        csr = None if exclude is None else exclusion_pairs_csr(exclude, usersId, self._candidates, self.device)
        vs, ixs = [], []
        for s in range(0, len(usersId), batch_size):
            if csr is None:
                v, ix = self.call(usersId[s:s + batch_size])
            else:
                info = usersId[s:s + batch_size]
                q = self._tower_forward(self.userTower, torch.from_numpy(self.userTowerIn(info)).to(self.device))
                v, ix = self.bruteForceLayer.query_with_exclusions(q, (csr[0][s:s + len(info) + 1], csr[1]))
            vs.append(v); ixs.append(ix)
        v = torch.cat(vs).cpu().numpy(); ix = torch.cat(ixs).cpu().numpy()
        idents = [[self._candidates[j] for j in row if j >= 0] for row in ix]
        return v, idents

    def score_vectors(self, usersId, itemsId):
        """(user vectors, item vectors) for topKmetrics.topKRatings."""
        u = torch.from_numpy(self.userTowerIn(list(usersId))).to(self.device)
        i = torch.from_numpy(self.itemTowerIn(list(itemsId))).to(self.device)
        return self._tower_forward(self.userTower, u), self._tower_forward(self.itemTower, i)


def batch_dataset(data, batchSize, keys):
    """tf.data.Dataset.from_tensor_slices(dict(df)).batch(batchSize): list of info dicts."""
    n = len(data[keys[0]])
    return [{k: data[k][s:s + batchSize] for k in keys} for s in range(0, n, batchSize)]


def splitTrainTest(data, ratio, seed=0):
    """Shuffle once, then take/skip (twoTower.py:113-122); data is a dict of equally long columns."""
    keys = list(data)
    n = len(data[keys[0]])
    perm = np.random.Generator(np.random.Philox(key=seed)).permutation(n)
    cut = int(n * ratio)
    take = lambda idx: {k: [data[k][j] for j in idx] for k in keys}
    return take(perm[:cut]), take(perm[cut:])


def crossValidation(dataSets, k, learningRate, optimiser, loss, epoch, embNum, batchSize, randomZero=False,
                    rdZeroDataSets=None, testBatchSize=5000, semb=64, userKey="CUSTOMER_ID", itemKey="MATERIAL",
                    resKey="RATING_TYPE", seed=42, verbose=0, rdZeroFilenames=None, bname=None, excludeTrain=False):
    """k-fold cross-validation of twoTower.py:125-272 on in-memory folds (dicts of columns) or, like the reference,
    on a list of file names read through loadBinaryMovieLens.gfData: train on all folds but one,
    index the whole catalog, top-k for every user, topKMetrics against the held-out fold and against
    the training folds ("full_" keys), averaged over folds.
    excludeTrain=True leaves each user's pairs of the training folds of dataSets out of their list (pairs added by
    rdZeroDataSets are not excluded), the held-out protocol's usual form; the "full_" metrics then count no hits
    by construction."""
    # keyword names of the reference's signature (twoTower.py:125): rdZeroFilenames = the folds with randomly added
    # zeros; bname = directory of its resource-usage logger (benchmarkLogger, out of scope here: accepted, unused)
    if rdZeroDataSets is None and rdZeroFilenames is not None:
        rdZeroDataSets = rdZeroFilenames
    folds = list(dataSets)
    if folds and isinstance(folds[0], str):                    # the reference's call form: file names (twoTower.py:125-139)
        from .loadBinaryMovieLens import gfData
        folds = [gfData(f)["ratings"] for f in folds]
        if randomZero:
            rdZeroDataSets = [gfData(f, rdZero=True)["ratings"] if isinstance(f, str) else f for f in rdZeroDataSets]
    usersId = list(dict.fromkeys(u for f in folds for u in f[userKey]))
    matId = list(dict.fromkeys(m for f in folds for m in f[itemKey]))
    train_folds = list(rdZeroDataSets) if randomZero else folds
    keys = [userKey, itemKey] + ([resKey] if randomZero else [])
    res, fullRes = [], []
    for it in range(len(folds)):
        test = folds[it]
        rest = [f for j, f in enumerate(train_folds) if j != it]
        train = {kk: [x for f in rest for x in f[kk]] for kk in keys}
        perm = np.random.Generator(np.random.Philox(key=seed + it)).permutation(len(train[userKey]))
        train = {kk: [train[kk][j] for j in perm] for kk in keys}          # shuffle once (:196)
        model = TwoTowerModel(embNum, len(matId), len(usersId), userKey, itemKey, usersId, matId,
                              eval_batch_size=batchSize, loss=loss, rdZero=randomZero, resKey=resKey, semb=semb, seed=seed)
        model.compile(optimiser, learningRate=learningRate)
        model.fit(batch_dataset(train, batchSize, keys), epochs=epoch, verbose=verbose)
        model.setCandidates(matId, k)
        others = [f for j, f in enumerate(folds) if j != it]
        seen = [(u, m) for f in others for u, m in zip(f[userKey], f[itemKey])]
        scores, idents = model.predict(usersId, batch_size=testBatchSize, exclude=seen if excludeTrain else None)
        topk = [(u, [(scores[r][j], idents[r][j]) for j in range(len(idents[r]))]) for r, u in enumerate(usersId)]
        res.append(topKMetrics(topk, list(zip(test[userKey], test[itemKey])), usersId, matId))
        fullRes.append(topKMetrics(topk, seen, usersId, matId))
    averageMetrics = {}
    for m in res[0]:
        averageMetrics[m] = sum(r[m] for r in res) / len(folds)
    for m in fullRes[0]:
        averageMetrics["full_" + m] = sum(r[m] for r in fullRes) / len(folds)
    return averageMetrics
