"""Multi-GPU plumbing: one process per GPU over torch.distributed (NCCL on the GPU box, gloo in the
CPU tests).  Replaces the reference's tf.distribute.experimental.MultiWorkerMirroredStrategy
(/root/reference/src/models/RModel.py:119-121; cluster from TF_CONFIG,
test/NeuMFModelWorker01.py:9): synchronous data parallelism.

Three pieces:
  * mirrored training (what the reference does): every rank holds the full tables, trains its slice
    of the global batch, the flat gradient arena is summed with ONE all-reduce per step and every rank
    applies the identical optimizer step.  The fused kernels scale gradients by 1/global_batch so
    the sum is the gradient of the global mean loss.  Right for tables that fit one GPU many times
    over (ML-1M shape: 2.5 MB).
  * row-sharded tables (owner = id mod G, local row = id div G) with an all-to-all of ids, rows and
    row gradients -- for tables too large to mirror (BASELINE.json configs[3]); the routing helpers
    here are pure index arithmetic and run on CPU or GPU tensors alike.
  * top-K over item-range shards: every rank scores all queries against its item range, the [U, k]
    lists are all-gathered and merged (score desc, id asc) -- identical to an unsharded scan.
"""
import os

import torch
import torch.distributed as dist


def is_dist():
    return dist.is_available() and dist.is_initialized()


def world_size():
    return dist.get_world_size() if is_dist() else 1


def rank():
    return dist.get_rank() if is_dist() else 0


def init_from_env(backend=None):
    """RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT as torchrun sets them (the reference reads
    TF_CONFIG instead)."""
    if is_dist() or int(os.environ.get("WORLD_SIZE", "1")) == 1:
        return
    backend = backend or ("nccl" if torch.cuda.is_available() else "gloo")
    if backend == "nccl":
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    else:
        dist.init_process_group(backend)


def barrier():
    """Host-side rendezvous of all ranks (no-op in a single process)."""
    if is_dist() and world_size() > 1:
        dist.barrier()


def all_reduce_sum_(flat, reducer=None):
    """In-place sum over ranks of the flat gradient arena: over NVLink peer memory when the arena came from
    gradient_arena() (brk_allreduce_dense_peer: no NCCL call on the step's path), else one NCCL all-reduce."""
    if reducer is not None:
        reducer.all_reduce_()
    elif is_dist() and world_size() > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    return flat


class PeerBuffer:
    """A flat fp32 arena in NVLink peer-mapped (symmetric) memory with the flag block of brk_allreduce_dense_peer."""

    def __init__(self, n_floats, device):
        import torch.distributed._symmetric_memory as symm_mem
        from . import _native as N
        self.n = (int(n_floats) + 3) // 4 * 4
        self.device = device
        group = dist.group.WORLD.group_name
        self.buf = symm_mem.empty(self.n, dtype=torch.float32, device=device)
        self.flags = symm_mem.empty(2 * 64, dtype=torch.int32, device=device)
        hb = symm_mem.rendezvous(self.buf, group)
        hf = symm_mem.rendezvous(self.flags, group)
        self.buf.zero_(); self.flags.zero_()
        self._ptrs = [torch.tensor(list(h.buffer_ptrs), dtype=torch.int64, device=device) for h in (hb, hf)]
        self.local_sync = torch.zeros(8, dtype=torch.int32, device=device)
        self._handles = (hb, hf)
        torch.cuda.synchronize(device)
        dist.barrier()                       # nobody posts a flag before everyone has zeroed its block

    def all_reduce_(self):
        from . import _native as N
        N.check(N.lib().brk_allreduce_dense_peer(N.ctx(self.device), self._ptrs[0].data_ptr(), self._ptrs[1].data_ptr(),
                                                 N.ptr(self.local_sync), self.n, rank(), world_size(), N.stream_ptr()),
                "brk_allreduce_dense_peer")

    def check(self):
        if int(self.local_sync[4].item()) != 0:
            raise RuntimeError("peer all-reduce: a cross-GPU barrier timed out (a rank did not reach the step); the step was "
                               "aborted on this rank (BRK_PEER_SPIN_MS sets the wait budget, default 30 s)")


def gradient_arena(n_floats, device):
    """(flat fp32 tensor of >= n_floats zeros, reducer or None): under torch.distributed with peer access the arena is
    symmetric memory and `reducer` sums it over the ranks through NVLink peer memory; otherwise a plain tensor (and
    all_reduce_sum_ falls back to NCCL when there is more than one rank)."""
    if is_dist() and world_size() > 1 and os.environ.get("BRK_DP", "peer") != "nccl":
        try:
            pb = PeerBuffer(n_floats, device)
            return pb.buf, pb
        except Exception as e:                # pragma: no cover - depends on the box
            if rank() == 0:
                print(f"[binrec_b200] symmetric memory unavailable ({e!r}); using NCCL all-reduce", flush=True)
    return torch.zeros((int(n_floats) + 3) // 4 * 4, dtype=torch.float32, device=device), None


def broadcast_(t, src=0):
    if is_dist() and world_size() > 1:
        dist.broadcast(t, src)
    return t


# ---- symmetric (peer-mapped) arenas for the fused data-parallel optimizer ---------------------------------
class PeerArena:
    """Weight and gradient arenas in NVLink peer-mapped memory plus the flag block of
    brk_dp_adam_peer.  The allocation / pointer exchange is torch's symmetric-memory plumbing; the
    reduce + Adam + broadcast + barriers are ours (csrc/dp_peer.cu)."""

    def __init__(self, n_floats, device):
        import torch.distributed._symmetric_memory as symm_mem
        from . import _native as N
        self.n = (int(n_floats) + 3) // 4 * 4
        self.device = device
        G, r = world_size(), rank()
        group = dist.group.WORLD.group_name
        self.w = symm_mem.empty(self.n, dtype=torch.float32, device=device)
        self.g = symm_mem.empty(self.n, dtype=torch.float32, device=device)
        self.flags = symm_mem.empty(2 * 64, dtype=torch.int32, device=device)
        hw = symm_mem.rendezvous(self.w, group)
        hg = symm_mem.rendezvous(self.g, group)
        hf = symm_mem.rendezvous(self.flags, group)
        self.w.zero_(); self.g.zero_(); self.flags.zero_()
        self._ptrs = [torch.tensor(list(h.buffer_ptrs), dtype=torch.int64, device=device) for h in (hw, hg, hf)]
        n4 = self.n // 4
        self.slice_lo, self.slice_hi = 4 * (n4 * r // G), 4 * (n4 * (r + 1) // G)
        sl = max(self.slice_hi - self.slice_lo, 4)
        self.m = torch.zeros(sl, dtype=torch.float32, device=device)
        self.v = torch.zeros(sl, dtype=torch.float32, device=device)
        self.local_sync = torch.zeros(8, dtype=torch.int32, device=device)
        self._handles = (hw, hg, hf)
        torch.cuda.synchronize(device)
        dist.barrier()                       # nobody posts a flag before everyone has zeroed its block
        self.desc = N.brk_dp_peer(self._ptrs[0].data_ptr(), self._ptrs[1].data_ptr(), self._ptrs[2].data_ptr(),
                                  self.m.data_ptr(), self.v.data_ptr(), self.local_sync.data_ptr(), self.n, r, G)

    def adam_step(self, hyper, state):
        """One fused reduce-scatter + Adam + all-gather step (all ranks must call it)."""
        import ctypes as C
        from . import _native as N
        N.check(N.lib().brk_dp_adam_peer(N.ctx(self.device), C.byref(self.desc), hyper, N.ptr(state), N.stream_ptr()),
                "brk_dp_adam_peer")

    def check(self):
        """Raises when a cross-GPU wait of the fused exchange timed out (a rank never reached the step; the kernels
        abort that step without touching the weights -- csrc/dp_peer.cu, csrc/bpr.cu).  One 4-byte device read: called
        at epoch ends and before checkpoints, not per step."""
        if int(self.local_sync[4].item()) != 0:
            raise RuntimeError("mirrored data parallelism: a cross-GPU barrier timed out (a rank did not reach the step); "
                               "the step was aborted on this rank and the replicas can no longer be trusted to be identical "
                               "(BRK_PEER_SPIN_MS sets the wait budget, default 30 s)")

    def full_moments(self):
        """Adam moments of the whole arena on every rank (they are sharded: rank r holds float4 slice r): for checkpoints."""
        m = torch.zeros(self.n, dtype=torch.float32, device=self.device); v = torch.zeros_like(m)
        k = self.slice_hi - self.slice_lo
        m[self.slice_lo:self.slice_hi] = self.m[:k]; v[self.slice_lo:self.slice_hi] = self.v[:k]
        dist.all_reduce(m); dist.all_reduce(v)
        return m, v

    def load_moments(self, m, v):
        k = self.slice_hi - self.slice_lo
        self.m[:k].copy_(m.reshape(-1)[self.slice_lo:self.slice_hi]); self.v[:k].copy_(v.reshape(-1)[self.slice_lo:self.slice_hi])


def peer_arena_or_none(n_floats, device):
    """PeerArena when running multi-rank on CUDA with peer access (and BRK_DP != 'nccl'), else None --
    the caller then falls back to one NCCL all-reduce per step."""
    if not is_dist() or world_size() == 1 or os.environ.get("BRK_DP", "peer") == "nccl":
        return None
    try:
        return PeerArena(n_floats, device)
    except Exception as e:                    # pragma: no cover - depends on the box
        if rank() == 0:
            print(f"[binrec_b200] symmetric memory unavailable ({e!r}); using NCCL all-reduce", flush=True)
        return None


# ---- batch slicing ------------------------------------------------------------------------------------
def local_slice(n, r=None, w=None):
    """Contiguous slice [lo, hi) of n items owned by rank r of w (remainder to the low ranks)."""
    r = rank() if r is None else r
    w = world_size() if w is None else w
    base, rem = divmod(n, w)
    lo = r * base + min(r, rem)
    return lo, lo + base + (1 if r < rem else 0)


# ---- row-shard routing (owner = id mod G) -----------------------------------------------------------------
def owner_of(ids, G):
    return ids % G


def local_row(ids, G):
    return torch.div(ids, G, rounding_mode="floor")


def shard_rows(num_rows, r, G):
    """Number of rows rank r owns under owner = id mod G."""
    return (num_rows - r + G - 1) // G


def bucket_by_owner(ids, G):
    """Stable partition of `ids` by owner.  Returns (perm, counts): ids[perm] is grouped by owner
    0..G-1 (original order kept inside a bucket), counts[g] = bucket size.  inverse: out[perm] = x."""
    own = owner_of(ids.long(), G)
    perm = torch.sort(own, stable=True).indices
    counts = torch.bincount(own, minlength=G)
    return perm, counts


def exchange_counts(counts):
    """all-to-all of the per-peer counts: returns how many ids each peer will send to this rank."""
    out = torch.empty_like(counts)
    dist.all_to_all_single(out, counts)
    return out


def exchange_rows(send, send_counts, recv_counts):
    """Variable-size all-to-all of rows ([n, ...] tensors); counts are host lists."""
    recv = send.new_empty((int(sum(recv_counts)),) + tuple(send.shape[1:]))
    dist.all_to_all_single(recv, send, output_split_sizes=[int(c) for c in recv_counts],
                           input_split_sizes=[int(c) for c in send_counts])
    return recv


class ShardedLookup:
    """Routing of one batch of ids to the owners of a row-sharded table and back.
    forward : ids -> (all-to-all ids) -> owners gather rows -> (all-to-all rows) -> rows in batch order
    backward: row gradients in batch order -> (all-to-all) -> owners scatter-add into their shard.
    `gather` and `scatter_add` are callables so that the CPU tests can run the same routing with
    NumPy-style indexing while the GPU path passes the C-ABI kernels."""

    def __init__(self, ids, G):
        self.G = G
        self.perm, counts = bucket_by_owner(ids, G)
        self.send_counts = counts.tolist()
        self.recv_counts = exchange_counts(counts).tolist()
        sorted_ids = ids[self.perm]
        self.owner_local_ids = local_row(exchange_rows(sorted_ids.contiguous(), self.send_counts, self.recv_counts), G)

    def forward(self, gather):
        rows_for_peers = gather(self.owner_local_ids)                       # [n_recv, d] from my shard
        got = exchange_rows(rows_for_peers.contiguous(), self.recv_counts, self.send_counts)
        out = torch.empty_like(got)
        out[self.perm] = got                                                 # back to batch order
        return out

    def backward(self, grads, scatter_add):
        send = grads[self.perm].contiguous()
        got = exchange_rows(send, self.send_counts, self.recv_counts)
        scatter_add(self.owner_local_ids, got)


# ---- top-K over item-range shards ----------------------------------------------------------------------------
def gather_topk_parts(vals, ids):
    """all-gather of the per-shard [U, k] lists -> ([G, U, k], [G, U, k])."""
    if not is_dist() or world_size() == 1:
        return vals.unsqueeze(0), ids.unsqueeze(0)
    G = world_size()
    pv = [torch.empty_like(vals) for _ in range(G)]
    pi = [torch.empty_like(ids) for _ in range(G)]
    dist.all_gather(pv, vals.contiguous())
    dist.all_gather(pi, ids.contiguous())
    return torch.stack(pv), torch.stack(pi)


def sharded_topk(queries, item_vectors_local, item_lo, k, merge=None, local_topk=None, exclude=None):
    """Top-k of `queries` against an item catalog range-sharded over the ranks: this rank holds rows
    [item_lo, item_lo + len(item_vectors_local)).  Result identical on every rank and identical to
    the unsharded scan (same tie rule).  `exclude`: one (indptr, ids) CSR of GLOBAL item ids per query row, the
    same on every rank (each rank's scorer ignores ids outside its range); it applies to the default local scorer."""
    from . import hotpath as H
    if exclude is not None and local_topk is not None:
        raise ValueError("sharded_topk: exclude applies to the default local scorer, not to a custom local_topk")
    if exclude is not None:
        local_topk = lambda q, c, off: H.BruteForceIndex(k).index(c, id_offset=off).query_with_exclusions(q, exclude)
    local_topk = local_topk or (lambda q, c, off: H.BruteForceIndex(k).index(c, id_offset=off)(q))
    merge = merge or H.topk_merge
    v, i = local_topk(queries, item_vectors_local, item_lo)
    pv, pi = gather_topk_parts(v, i)
    return merge(pv, pi)
