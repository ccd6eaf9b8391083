"""Multi-GPU plumbing for the link-prediction path (SURVEY.md section 8e).  One process per GPU,
``torch.distributed`` (NCCL on the GPUs; the host logic below is backend-agnostic and is tested
with gloo, world_size 2, on CPU tensors).

The reference is single-process (kgvae/link_predict.py:113-115); everything here is new:

* small graphs (FB15k-237 / WN18 shapes): **replicas** - each rank samples its own subgraph with
  the reference's sampler, gradients are averaged with one all-reduce of the flattened gradient;
* evaluation: **entity-sharded** - every rank scores all queries against its slice of the
  candidates and the per-shard rank counts are summed;
* large graphs (wikikg2 shape): **destination-node ownership** - rank p owns a contiguous block
  of nodes and every edge whose destination is in it; layer inputs are all-gathered.
"""
import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L


def world():
    """(rank, world_size) of the default process group, (0, 1) when not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


class _exposed:
    """Context manager: when bench.py has switched per-op profiling on (_lib.profile is a dict), record CUDA
    events on the CURRENT stream around a collective (or around the wait for an asynchronous one).  The
    compute stream idles while it waits for NCCL's stream, so the elapsed time is the communication time that
    was NOT hidden behind compute - what bench.py reports as comm_ms."""

    def __init__(self, tag):
        self.tag = "nccl_exposed[" + tag + "]"

    def __enter__(self):
        if L.profile is not None:
            self.ev0 = torch.cuda.Event(enable_timing=True)
            self.ev0.record()
        return self

    def __exit__(self, *exc):
        if L.profile is not None and hasattr(self, "ev0"):
            ev1 = torch.cuda.Event(enable_timing=True)
            ev1.record()
            L.profile.setdefault(self.tag, []).append((self.ev0, ev1))
        return False


def agree_scalar(value, op, group=None):
    """All-reduce of one integer over the group (on the backend's device type): the ranks leave with the
    same number, so decisions derived from it are taken identically everywhere."""
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = torch.tensor([int(value)], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=op, group=group)
    return int(t.item())


def block_range(n, rank, world_size):
    """Contiguous block [lo, hi) of ``n`` items owned by ``rank``; sizes differ by at most one."""
    return (n * rank) // world_size, (n * (rank + 1)) // world_size


entity_shard = block_range


def uniform_block_range(n, rank, world_size):
    """Contiguous blocks of ONE size, ceil(n / world_size) (the last ranks may own fewer rows or none):
    the owner of row r is r // blk, which is what a kernel can compute per edge (PeerRows)."""
    blk = (n + world_size - 1) // world_size
    lo = min(n, rank * blk)
    return lo, min(n, lo + blk)


def allreduce_mean_grads(params, group=None):
    """Average ``p.grad`` over the group with ONE all-reduce of the flattened gradient (replicas).
    Parameters without a gradient contribute zeros so that every rank sends the same layout."""
    params = [p for p in params if p.requires_grad]
    if not params:
        return
    ws = dist.get_world_size(group)
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat /= ws
    off = 0
    for p in params:
        n = p.numel()
        if p.grad is None:
            p.grad = flat[off:off + n].view_as(p).clone()
        else:
            p.grad.copy_(flat[off:off + n].view_as(p.grad))
        off += n


class GradBuckets:
    """Replica training: gradients live in ONE persistent flat buffer (``p.grad`` is a view of it) cut into
    buckets, and a bucket is all-reduced (NCCL, asynchronously, on the communicator's stream) the moment the
    last of its parameters has received its gradient - from autograd's post-accumulate hooks, i.e. while
    the rest of the backward pass is still running.  Replaces the post-backward ``torch.cat`` + one
    all-reduce + copy-back of allreduce_mean_grads: no flatten, no copy back, and only the bucket that
    becomes ready last (the entity embedding, whose gradient backward produces at the very end) is exposed.

    ``buckets``: list of parameter lists in the order their gradients become ready (decoder / prior first,
    embedding last); parameters not listed form a final bucket.  Call ``zero()`` instead of
    ``optimizer.zero_grad()`` (one memset; the views must stay in place) and ``finish()`` after
    ``loss.backward()``; ``average``: divide by the world size (replicas) or keep the sum (partitioned)."""

    def __init__(self, params, buckets=None, group=None, average=True):
        params = [p for p in params if p.requires_grad]
        listed = {id(p) for b in (buckets or []) for p in b}
        groups = [[p for p in b if p.requires_grad] for b in (buckets or [])]
        rest = [p for p in params if id(p) not in listed]
        if rest:
            groups.append(rest)
        self.groups = [g for g in groups if g]
        self.group, self.average = group, average
        self.world_size = dist.get_world_size(group) if dist.is_initialized() else 1
        total = sum(p.numel() for g in self.groups for p in g)
        dev = self.groups[0][0].device
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.slices, self._bucket_of, self._pending, self._handles, self._hooks = [], {}, [], [], []
        self._views = {}
        off = 0
        for b, g in enumerate(self.groups):
            start = off
            for p in g:
                n = p.numel()
                p.grad = self.flat[off:off + n].view_as(p)
                self._views[id(p)] = p.grad
                self._bucket_of[id(p)] = b
                self._hooks.append(p.register_post_accumulate_grad_hook(self._hook))
                off += n
            self.slices.append(self.flat[start:off])
        self._reset()

    def close(self):
        """Detach from the parameters: remove the hooks and give every parameter a gradient tensor of its own."""
        for h in self._hooks:
            h.remove()
        self._hooks = []
        for g in self.groups:
            for p in g:
                if p.grad is not None:
                    p.grad = p.grad.clone()

    def _reset(self):
        self._pending = [len(g) for g in self.groups]
        self._handles = []

    def _hook(self, p):
        view = self._views[id(p)]
        if p.grad is not view and (p.grad is None or p.grad.data_ptr() != view.data_ptr()):
            # someone dropped the view (optimizer.zero_grad(set_to_none=True), p.grad = None): autograd then made a
            # fresh gradient tensor - move it into the flat buffer so that the bucket all-reduce sees it
            if p.grad is not None:
                view.copy_(p.grad)
            p.grad = view
        b = self._bucket_of[id(p)]
        self._pending[b] -= 1
        if self._pending[b] == 0 and self.world_size > 1:
            self._launch(b)

    def _launch(self, b):
        op = dist.ReduceOp.AVG if (self.average and dist.get_backend(self.group) == "nccl") else dist.ReduceOp.SUM
        h = dist.all_reduce(self.slices[b], op=op, group=self.group, async_op=True)
        self._handles.append((h, b, op))

    def zero(self):
        self.flat.zero_()
        self._reset()

    def clip_(self, max_norm):
        """torch.nn.utils.clip_grad_norm_ over all bucketed gradients (kgvae/link_predict.py:227) on the flat
        buffer: one norm, one scale, no per-parameter launches and no host sync."""
        total = torch.linalg.vector_norm(self.flat)
        self.flat.mul_(torch.clamp(max_norm / (total + 1e-6), max=1.0))
        return total

    def finish(self):
        """Wait for the bucket all-reduces (stream-ordered: the current stream waits, the host does not block
        beyond NCCL's own enqueue) and launch any bucket whose parameters received no gradient this step."""
        if self.world_size > 1:
            for b, n in enumerate(self._pending):
                if n > 0:                     # unused parameters: zeros on this rank, still part of the layout
                    self._launch(b)
            with _exposed("gradient buckets"):
                for h, b, op in self._handles:
                    h.wait()
                    if self.average and op == dist.ReduceOp.SUM:
                        self.slices[b].div_(self.world_size)
        self._reset()


def sharded_rank_counts(count_fn, num_entities, group=None):
    """Entity-sharded evaluation: ``count_fn(lo, hi)`` returns, for every query, the number of
    candidates in [lo, hi) ranked ahead of the target (an integer tensor); the shards' counts add
    up to the 0-indexed rank.  The sum is exact because every (query, candidate) decision is made
    on the same score on whichever rank holds the candidate."""
    rank, ws = (dist.get_rank(group), dist.get_world_size(group)) if dist.is_initialized() else (0, 1)
    lo, hi = block_range(num_entities, rank, ws)
    counts = count_fn(lo, hi)
    if ws > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    return counts


def merge_topk(idx, score, k, group=None):
    """Entity-sharded generation: every rank holds the ``[M, k]`` top-k lists (``idx`` global entity ids, -1 for
    none; ``score``) of the same M queries over its own slice of the candidates.  All-gathers them and keeps, per
    query, the ``k`` best by (score descending, id ascending); -1 entries are dropped and the result is padded with
    -1 / -inf.  Exact: the shards are disjoint, every score is the same canonical value whichever rank computes it,
    and the union of the shards' top-k lists contains the global top-k.  Collective; every rank returns the same
    ``(idx, score)`` (dtypes and device of the inputs)."""
    ws = dist.get_world_size(group) if dist.is_initialized() else 1
    idx, score = idx.contiguous(), score.contiguous()
    if ws > 1:
        parts_i = [torch.empty_like(idx) for _ in range(ws)]
        parts_s = [torch.empty_like(score) for _ in range(ws)]
        dist.all_gather(parts_i, idx, group=group)
        dist.all_gather(parts_s, score, group=group)
        idx, score = torch.cat(parts_i, dim=1), torch.cat(parts_s, dim=1)
    valid = idx >= 0
    big = torch.iinfo(idx.dtype).max
    ids = torch.where(valid, idx, torch.full_like(idx, big))
    sc = torch.where(valid, score, torch.full_like(score, float("-inf")))
    # (score desc, id asc): sort by id, then stably by score
    order = torch.sort(ids, dim=1, stable=True)[1]
    ids, sc = ids.gather(1, order), sc.gather(1, order)
    order = torch.sort(sc, dim=1, descending=True, stable=True)[1][:, :k]
    ids, sc = ids.gather(1, order), sc.gather(1, order)
    if ids.shape[1] < k:
        pad = k - ids.shape[1]
        ids = torch.cat([ids, ids.new_full((ids.shape[0], pad), big)], dim=1)
        sc = torch.cat([sc, sc.new_full((sc.shape[0], pad), float("-inf"))], dim=1)
    kept = ids != big
    return torch.where(kept, ids, torch.full_like(ids, -1)), torch.where(kept, sc, torch.full_like(sc, float("-inf")))


def partition_by_destination(src, dst, etype, norm, num_nodes, world_size, uniform=False):
    """Destination-node ownership: returns a list (one entry per rank) of dicts with the owned node
    block ``[lo, hi)``, the rank's edges (every edge with dst in the block, original relative
    order kept - so per-destination summation order equals the single-GPU order) and
    ``needed_src``: the sorted unique source ids the rank must receive features for.
    ``uniform``: blocks of one size (uniform_block_range), required by the peer-memory gather."""
    src, dst, etype = (np.asarray(a) for a in (src, dst, etype))
    norm = None if norm is None else np.asarray(norm).reshape(-1)
    # owner of an edge: the rank p with lo_p <= dst < hi_p
    rng = uniform_block_range if uniform else block_range
    bounds = np.array([rng(num_nodes, p, world_size)[0] for p in range(world_size)] + [num_nodes])
    owner = np.searchsorted(bounds, dst, side="right") - 1
    parts = []
    for p in range(world_size):
        sel = np.nonzero(owner == p)[0]
        lo, hi = int(bounds[p]), int(bounds[p + 1])
        parts.append({"lo": lo, "hi": hi, "edge_ids": sel, "src": src[sel], "dst": dst[sel], "etype": etype[sel],
                      "norm": None if norm is None else norm[sel], "needed_src": np.unique(src[sel])})
    return parts


def allgather_rows(local_rows, num_rows, group=None, uniform=False):
    """All-gather of node features for destination-partitioned message passing: every rank holds
    rows [lo, hi) of a [num_rows, d] matrix and receives the full matrix.  Blocks may differ in
    size (block_range: by one row; uniform_block_range: the last ones are shorter), so the gather
    is padded to the largest block."""
    rank, ws = dist.get_rank(group), dist.get_world_size(group)
    rng = uniform_block_range if uniform else block_range
    sizes = [rng(num_rows, p, ws)[1] - rng(num_rows, p, ws)[0] for p in range(ws)]
    pad = max(sizes)
    buf = local_rows.new_zeros((pad,) + tuple(local_rows.shape[1:]))
    buf[:local_rows.shape[0]] = local_rows
    out = local_rows.new_empty((ws * pad,) + tuple(local_rows.shape[1:]))
    if hasattr(dist, "all_gather_into_tensor") and dist.get_backend(group) != "gloo":
        dist.all_gather_into_tensor(out, buf, group=group)
        parts = out.view((ws, pad) + tuple(local_rows.shape[1:]))
    else:
        lst = [torch.empty_like(buf) for _ in range(ws)]
        dist.all_gather(lst, buf, group=group)
        parts = lst
    if all(n == pad for n in sizes):
        return out if not isinstance(parts, list) else torch.cat(parts, dim=0)
    return torch.cat([parts[p][:n] for p, n in enumerate(sizes)], dim=0)


# ---------------------------------------------------------------------------------------------
# destination-partitioned training: differentiable collectives and the partition descriptor
# ---------------------------------------------------------------------------------------------
class Partition:
    """Rank-local view of a destination-partitioned graph: this rank owns nodes [lo, hi) of
    ``n_global`` and every edge whose destination is in that block (edge sources keep global ids,
    destinations are local: dst - lo).  Attach to the graph object as ``g.partition``; RelGraphConv,
    KGVAE and LinkPredict then insert the all-gathers / reductions below."""

    def __init__(self, lo, hi, n_global, group=None, peer_gather=None, col_chunks=None):
        self.lo, self.hi, self.n_global, self.group = int(lo), int(hi), int(n_global), group
        # all-gather mode: layer inputs travel (and source gradients return) in this many COLUMN chunks, each
        # pipelined against the message passing of the previous / next chunk (ops.BddConvFn); 1 = one collective
        # Measured on the wikikg2 shape: 2 chunks hide 6 ms of NCCL time at 8 ranks (106.0 vs 107.4 ms/step) but cost
        # more in smaller kernels than they hide at 2 ranks (328.5 vs 318.8 ms/step) - default by world size.
        self.col_chunks = int(col_chunks) if col_chunks else (2 if dist.get_world_size(group) >= 4 else 1)
        self.n_local = self.hi - self.lo
        self.world_size = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        # uniform blocks (uniform_block_range) allow the fused peer-memory gather: the kernel finds
        # the owner of a source row as row // blk.  Whether the blocks are uniform is a property of the
        # whole partition, so it is AGREED across the ranks (one MIN all-reduce), not inferred per rank:
        # ranks that disagreed would pad their all-gathers differently or issue mismatched collectives.
        blk = (self.n_global + self.world_size - 1) // self.world_size
        mine = (self.lo, self.hi) == uniform_block_range(self.n_global, self.rank, self.world_size)
        uniform = bool(agree_scalar(1 if mine else 0, dist.ReduceOp.MIN, group))
        self.blk = blk if uniform else None
        # None: decide per graph (use_peer_gather); True/False: forced (True still needs uniform blocks)
        self.peer_gather = None if peer_gather is None else (bool(peer_gather) and uniform)
        self._peer_decision = None
        self._noise_gen = None
        self._peer_rows = {}

    def use_peer_gather(self, n_local_edges):
        """Fused peer-memory gather or NCCL all-gather for a layer input?  Peer loads bypass the local
        L2, so the gather moves one row per EDGE whose source is remote, the all-gather one row per
        remote NODE: gather from peers when a rank has, on average, fewer edges than the graph has nodes.
        The decision is collective (one SUM all-reduce of the local edge counts on first use, then
        cached): every rank of the job takes the same branch, whatever its own share of the edges."""
        if self.blk is None:
            return False
        if self.peer_gather is not None:
            return self.peer_gather
        if self._peer_decision is None:
            total = agree_scalar(int(n_local_edges), dist.ReduceOp.SUM, self.group)
            self._peer_decision = total < self.n_global * self.world_size
        return self._peer_decision

    def noise_generator(self, device):
        """Device generator seeded ``torch.initial_seed() + 1 + rank``: the reparameterisation noise and the
        dropout masks of a rank's node block must be independent of the other ranks' (replicated parameters
        require the SAME default seed everywhere, which would give every block identical draws)."""
        if self._noise_gen is None:
            self._noise_gen = torch.Generator(device=device)
            self._noise_gen.manual_seed((torch.initial_seed() + 1 + self.rank) % (1 << 62))
        return self._noise_gen

    def peer_rows(self, key, width, device):
        """The PeerRows buffer of one layer (created collectively on first use, then reused)."""
        k = (key, int(width))
        if k not in self._peer_rows:
            self._peer_rows[k] = PeerRows(self.blk, width, device, self.group)
        return self._peer_rows[k]


class _DeviceMemory:
    """Exposes raw device memory through __cuda_array_interface__ so torch can alias it (no copy)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (int(ptr), False),
                                         "version": 3, "strides": None}


def _wrap_device_memory(ptr, shape, device):
    return torch.as_tensor(_DeviceMemory(ptr, shape), device=device)


class PeerRows:
    """One [blk, width] fp32 row block per rank, each in its owner's HBM and mapped into every
    process of the node with CUDA IPC, so that a kernel on any rank can read any rank's rows over
    NVLink.  ``publish(x)`` copies this rank's rows in between two stream-ordered barriers: the
    first keeps peers that still read the previous contents (their backward pass) safe, the second
    makes the new rows visible before anyone gathers from them.  ``ptrs`` is the device-resident
    table of the P block base pointers that kg_bdd_rel_fwd / kg_bdd_rel_bwd take as ``x_parts``."""

    def __init__(self, blk_rows, width, device, group=None):
        import ctypes
        self.group = group
        self.rank, self.world_size = dist.get_rank(group), dist.get_world_size(group)
        self.blk, self.width = int(blk_rows), int(width)
        self.device = torch.device(device)
        nbytes = self.blk * self.width * 4
        with torch.cuda.device(self.device):
            ptr, handle = ctypes.c_void_p(), (ctypes.c_ubyte * 64)()
            L.call("kg_peer_alloc", nbytes, ctypes.byref(ptr), handle)
            self._own_ptr = ptr.value
            handles = [None] * self.world_size
            dist.all_gather_object(handles, bytes(handle), group=group)
            self._peer_ptrs, base = [], []
            for r, h in enumerate(handles):
                if r == self.rank:
                    base.append(self._own_ptr)
                    continue
                p, buf = ctypes.c_void_p(), (ctypes.c_ubyte * 64).from_buffer_copy(h)
                L.call("kg_peer_open", buf, ctypes.byref(p))      # mapped on MY device, peer access enabled
                self._peer_ptrs.append(p.value)
                base.append(p.value)
        self.local = _wrap_device_memory(self._own_ptr, (self.blk, self.width), self.device)
        self.views = [self.local if r == self.rank else _wrap_device_memory(b, (self.blk, self.width), self.device)
                      for r, b in enumerate(base)]
        self.ptrs = torch.tensor(base, dtype=torch.int64, device=self.device)
        self._sync = torch.zeros(1, device=self.device)

    def close(self):
        """Unmap the peers' blocks and free this rank's (collective: every rank must be done reading)."""
        if self._own_ptr is None:
            return
        torch.cuda.synchronize(self.device)
        self.barrier()
        torch.cuda.synchronize(self.device)
        with torch.cuda.device(self.device):
            for p in self._peer_ptrs:
                L.call("kg_peer_close", p)
            self.barrier()
            torch.cuda.synchronize(self.device)
            L.call("kg_peer_free", self._own_ptr)
        self._own_ptr, self._peer_ptrs, self.views, self.local = None, [], [], None

    def barrier(self):
        with _exposed("peer barrier"):
            dist.all_reduce(self._sync, group=self.group)       # stream-ordered on every rank

    def publish(self, x):
        if x.shape[0] > self.blk or x.shape[1] != self.width:
            raise RuntimeError(f"PeerRows: {tuple(x.shape)} rows do not fit a [{self.blk}, {self.width}] block")
        self.barrier()
        self.local[:x.shape[0]].copy_(x)
        self.barrier()


class _Pending:
    """An asynchronous collective and what turns its raw output into the result; ``wait()`` makes the current
    stream wait for it (the host does not block) and returns the result."""

    def __init__(self, work, finish, tag="collective"):
        self.work, self.finish, self.tag = work, finish, tag

    def wait(self):
        if self.work is not None:
            with _exposed(self.tag):
                self.work.wait()
        return self.finish()


def allgather_rows_start(x_local, part):
    """allgather_rows as an asynchronous NCCL collective (uniform or near-uniform blocks): returns a _Pending
    whose ``wait()`` yields the [n_global, d] matrix.  Work enqueued between the call and ``wait()`` overlaps
    the transfer."""
    group = part.group
    ws, n_global = part.world_size, part.n_global
    uniform = part.blk is not None
    rng = uniform_block_range if uniform else block_range
    sizes = [rng(n_global, p, ws)[1] - rng(n_global, p, ws)[0] for p in range(ws)]
    pad = max(sizes)
    x_local = x_local.contiguous()
    if x_local.shape[0] == pad:
        buf = x_local
    else:
        buf = x_local.new_zeros((pad,) + tuple(x_local.shape[1:]))
        buf[:x_local.shape[0]] = x_local
    out = x_local.new_empty((ws * pad,) + tuple(x_local.shape[1:]))
    if dist.get_backend(group) == "gloo":
        lst = [torch.empty_like(buf) for _ in range(ws)]
        work = dist.all_gather(lst, buf, group=group, async_op=True)

        def finish():
            return torch.cat([lst[p][:n] for p, n in enumerate(sizes)], dim=0)
    else:
        work = dist.all_gather_into_tensor(out, buf, group=group, async_op=True)

        def finish():
            if all(n == pad for n in sizes):
                return out
            if uniform:               # only the last blocks are short: the first n_global rows are the matrix
                return out[:n_global]
            parts = out.view((ws, pad) + tuple(x_local.shape[1:]))
            return torch.cat([parts[p][:n] for p, n in enumerate(sizes)], dim=0)
    return _Pending(work, finish, "all-gather rows")


def reduce_scatter_rows_start(g_full, part):
    """reduce_scatter_rows as an asynchronous collective: ``wait()`` yields this rank's rows of the sum."""
    if part.blk is not None and hasattr(dist, "reduce_scatter_tensor") and dist.get_backend(part.group) != "gloo":
        rows = part.blk * part.world_size
        if g_full.shape[0] < rows:
            pad = g_full.new_zeros((rows,) + tuple(g_full.shape[1:]))
            pad[:g_full.shape[0]] = g_full
            g_full = pad
        out = g_full.new_empty((part.blk,) + tuple(g_full.shape[1:]))
        work = dist.reduce_scatter_tensor(out, g_full[:rows], op=dist.ReduceOp.SUM, group=part.group, async_op=True)
        return _Pending(work, lambda: out[:part.n_local], "reduce-scatter rows")
    work = dist.all_reduce(g_full, op=dist.ReduceOp.SUM, group=part.group, async_op=True)
    return _Pending(work, lambda: g_full[part.lo:part.hi].clone(), "reduce-scatter rows")


class AllGatherRowsFn(torch.autograd.Function):
    """x_local [n_local, d] -> x_full [n_global, d]; backward: reduce-scatter(sum) of the gradient -
    every rank's loss depends on every row it gathered."""

    @staticmethod
    def forward(ctx, x_local, part):
        ctx.part = part
        with _exposed("all-gather rows"):
            return allgather_rows(x_local.contiguous(), part.n_global, part.group, uniform=part.blk is not None)

    @staticmethod
    def backward(ctx, g_full):
        part = ctx.part
        with _exposed("reduce-scatter rows"):
            return reduce_scatter_rows(g_full.contiguous(), part), None


def reduce_scatter_rows(g_full, part):
    """Sum over ranks of a [n_global (or more), d] matrix of per-row contributions; every rank keeps
    its own rows [lo, hi).  Uniform blocks: one reduce-scatter (each rank receives 1/P of the
    bytes); otherwise all-reduce and slice."""
    if part.blk is not None and hasattr(dist, "reduce_scatter_tensor") and dist.get_backend(part.group) != "gloo":
        rows = part.blk * part.world_size
        if g_full.shape[0] < rows:
            pad = g_full.new_zeros((rows,) + tuple(g_full.shape[1:]))
            pad[:g_full.shape[0]] = g_full
            g_full = pad
        out = g_full.new_empty((part.blk,) + tuple(g_full.shape[1:]))
        dist.reduce_scatter_tensor(out, g_full[:rows], op=dist.ReduceOp.SUM, group=part.group)
        return out[:part.n_local]
    dist.all_reduce(g_full, op=dist.ReduceOp.SUM, group=part.group)
    return g_full[part.lo:part.hi].clone()


class AllReduceSumFn(torch.autograd.Function):
    """sum over ranks of a tensor every rank then uses in its own loss; backward sums the upstream
    gradients of all ranks."""

    @staticmethod
    def forward(ctx, x, group):
        ctx.group = group
        y = x.clone()
        dist.all_reduce(y, op=dist.ReduceOp.SUM, group=group)
        return y

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous().clone()
        dist.all_reduce(g, op=dist.ReduceOp.SUM, group=ctx.group)
        return g, None


def allreduce_sum_grads(params, group=None):
    """Partitioned training: every rank holds a partial gradient of the replicated parameters;
    the total is their SUM (one flattened all-reduce)."""
    params = [p for p in params if p.requires_grad]
    if not params:
        return
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    off = 0
    for p in params:
        n = p.numel()
        if p.grad is None:
            p.grad = flat[off:off + n].view_as(p).clone()
        else:
            p.grad.copy_(flat[off:off + n].view_as(p.grad))
        off += n
