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


class TwoTowerModel:
    def __init__(self, embedDim, nbrItem, nbrUser, userKey, itemKey, usersId, itemsId, eval_batch_size=8000,
                 loss=None, rdZero=False, resKey=None, semb=100, seed=42, device=None, tensor_cores=False):
        self.device = torch.device(device or f"cuda:{torch.cuda.current_device()}")
        self.embedDim, self.nbrItem, self.nbrUser = embedDim, nbrItem, nbrUser
        self.userKey, self.itemKey, self.resKey = userKey, itemKey, resKey
        self.eval_batch_size, self.rdZero, self.semb = eval_batch_size, rdZero, semb
        # tensor_cores: Dense / in-batch products on tcgen05 with TF32 operands (csrc/gemm_tc.cu); fp32 FMA otherwise
        self.tensor_cores = bool(tensor_cores)
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
        self.bruteForceLayer = None
        self._candidates = None
        self.optimizer = None
        self.computeLoss = self.computeLossRdZero if rdZero else self.computeLossTfrs
        self._ws_batch = 0
        self.history = {"loss": []}

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
            self._bufs = dict(eu=f(B, self.embedDim), ei=f(B, self.embedDim), deu=f(B, self.embedDim),
                              dei=f(B, self.embedDim), q=f(B, S), c=f(B, S), dq=f(B, S),
                              dc=f(B, S), scores=f(B, B) if not self.rdZero else None,
                              ones=torch.ones(B, dtype=torch.float32, device=dev),
                              acc=torch.zeros(1, dtype=torch.float64, device=dev))
            self._ws_batch = B
        b = self._bufs
        return N.brk_twotower_workspace(*[b[k].data_ptr() if b[k] is not None else None
                                          for k in ("eu", "ei", "q", "c", "dq", "dc", "scores", "ones", "acc", "deu", "dei")])

    def _ids(self, info):
        dev = self.device
        return self.userTowerIn.lookup_device(info[self.userKey], dev), self.itemTowerIn.lookup_device(info[self.itemKey], dev)

    def _step(self, u, i, labels, training, loss_out=None):
        B = u.numel()
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
        ws = self._workspace(B)
        ut, it = self.userTower.c_struct(), self.itemTower.c_struct()
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
        """In-batch softmax loss of already computed tower outputs (twoTower.py:82-83), forward only."""
        scores = usersCaracteristics @ itemCaracteristics.T
        ids = torch.from_numpy(self.itemTowerIn(info[self.itemKey])).to(self.device)
        B = scores.shape[0]
        dup = (ids[:, None] == ids[None, :]).float() - torch.eye(B, device=self.device)
        scores = scores + dup * (float(np.finfo(np.float32).min) / 100.0)
        return torch.nn.functional.cross_entropy(scores, torch.arange(B, device=self.device), reduction="sum")

    def computeLossRdZero(self, usersCaracteristics, itemCaracteristics, info):
        y = torch.as_tensor(np.asarray(info[self.resKey], dtype=np.float32)).to(self.device)
        return torch.nn.functional.binary_cross_entropy_with_logits((usersCaracteristics * itemCaracteristics).sum(1), y)

    def _labels(self, info):
        if not self.rdZero:
            return None
        return torch.as_tensor(np.asarray(info[self.resKey], dtype=np.float32)).to(self.device)

    def train_step(self, info):
        """One fused forward/backward + Adagrad step; returns {"loss": device scalar} (twoTower.py:89-102).
        Under torch.distributed the replicas' SUM-reduced gradients are summed by one all-reduce per
        tower (MirroredStrategy sums per-replica gradients of a SUM-reduced loss)."""
        u, i = self._ids(info)
        return {"loss": self._train_ids(u, i, self._labels(info))}

    def _train_step_native(self, u, i, labels, loss_out=None):
        """Step + Keras Adagrad in one library call (brk_twotower_train_step): ONE cooperative launch when the in-batch
        softmax step runs on the tensor cores and the batch fits on chip, the step + optimizer kernels otherwise."""
        B = u.numel()
        loss_out = loss_out if loss_out is not None else torch.empty(1, dtype=torch.float32, device=self.device)
        ws = self._workspace(B)
        ut, it = self.userTower.c_struct(), self.itemTower.c_struct()
        opt = self.optimizer
        N.check(N.lib().brk_twotower_train_step(N.ctx(self.device), C.byref(ut), C.byref(it), N.ptr(u), N.ptr(i), N.ptr(i),
                                                N.ptr(labels) if labels is not None else None, B,
                                                (1 if self.rdZero else 0) | (0x100 if self.tensor_cores else 0), C.byref(ws),
                                                float(opt.lr), float(opt.eps), int(opt.rows_threshold_bytes), N.ptr(loss_out),
                                                N.stream_ptr()), "brk_twotower_train_step")
        return loss_out

    def _train_ids(self, u, i, labels, loss_out=None):
        if self.optimizer is None:
            self.compile()
        if D.world_size() == 1 and u.numel() > 0 and isinstance(self.optimizer, H.Adagrad):
            return self._train_step_native(u, i, labels, loss_out)
        if u.numel() > 0:
            loss = self._step(u, i, labels, True, loss_out)
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
        return {"loss": self._step(u, i, self._labels(info), False)}

    def fit(self, dataset, epochs=1, verbose=0, graph=True):
        """dataset: iterable of info dicts (batches), replayed every epoch like a cached tf.data set.
        graph=True replays the training step as ONE CUDA graph launch per batch (single process, equal-sized batches
        except a shorter last one): at the reference's batch of 1000 the step is a chain of few-microsecond kernels
        and the per-kernel launch cost is the larger half of it (124 -> 70 us per step on B200)."""
        batches = list(dataset)
        # string -> index lookups and H2D of the ids once per fit, not once per step and epoch (the reference caches
        # its batched dataset too: trainSetCached, twoTower.py:197-198)
        staged = [(self._ids(info), self._labels(info)) for info in batches]
        if D.world_size() > 1:
            # mirrored data parallelism: a batch of the dataset is the GLOBAL batch (MultiWorkerMirroredStrategy auto-shards
            # it); this rank trains its slice, with its slice's items as in-batch negatives (the per-replica loss), and the
            # SUM-reduced gradients are summed over the ranks (peer all-reduce in _train_ids)
            def mine(t):
                if t is None:
                    return None
                lo, hi = D.local_slice(t.numel())
                return t[lo:hi].contiguous()
            staged = [((mine(u), mine(i)), mine(lab)) for (u, i), lab in staged]
            D.barrier()
        sizes = [u.numel() for (u, _), _ in staged]
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
                (u, i), lab = staged[0]
                self._train_ids(u, i, lab, losses[0:1])
                if replay is None:
                    replay = self._capture_fit_graph(staged[:n_full])
                replay(losses, 1, n_full)
                rest = range(n_full, len(staged))
            else:
                rest = range(len(staged))
            for k in rest:
                (u, i), lab = staged[k]
                self._train_ids(u, i, lab, losses[k:k + 1])
            # one host sync per epoch: Keras reports the running mean of the per-batch losses
            self.history["loss"].append(float(losses.double().sum().item()) / max(len(staged), 1))
            if self._reducer is not None:
                self._reducer.check()                        # a peer all-reduce that timed out aborted its step: raise here
            if verbose:
                print(f"epoch {e + 1}: loss {self.history['loss'][-1]:.6f}")
        return self

    def _capture_fit_graph(self, full):
        """Captures `copy batch [pos] into the static id buffers -> fused step -> Adagrad -> store the loss at [pos] ->
        pos += 1` once; returns replay(losses, first, last) that runs batches first..last-1 of `full`."""
        dev = self.device
        all_u = torch.stack([u for (u, _), _ in full]); all_i = torch.stack([i for (_, i), _ in full])
        all_lab = torch.stack([lab for _, lab in full]) if full[0][1] is not None else None
        B = all_u.shape[1]
        cur_u, cur_i = torch.empty_like(all_u[0]), torch.empty_like(all_i[0])
        cur_lab = torch.empty_like(all_lab[0]) if all_lab is not None else None
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
            self._train_ids(cur_u, cur_i, cur_lab, cur_loss)
            sink.index_copy_(0, pos, cur_loss)
            pos.add_(1)

        def replay(losses, first, last):
            pos.fill_(first)
            for _ in range(first, last):
                g.replay()
            losses[first:last].copy_(sink[first:last])
        self._fit_graph_keepalive = (g, all_u, all_i, all_lab, cur_u, cur_i, cur_lab, cur_loss, pos, sink)
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
