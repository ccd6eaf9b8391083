"""torch.autograd.Function wrappers over the C ABI (include/kgvae_b200.h).

Each Function is one fused operator of the link-prediction path and names the reference
code it replaces.  All tensors are CUDA, fp32 / int32, contiguous; PyTorch supplies device
memory, the stream and autograd bookkeeping only.
"""
import ctypes
import os

import torch

from . import _lib as L


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


class tensor_core_terms:
    """Context manager: run the tensor-core products (kg_gemm_f32, kg_distmult_rank) with ``terms`` split
    terms - 3 is the fp32-accurate default, 1 the single-product mode that north_star asks to be reported
    separately (operands rounded to 11 significant bits)."""

    def __init__(self, terms):
        self.terms = int(terms)

    def __enter__(self):
        self.old = L.lib().kg_set_tc_terms(self.terms)
        return self

    def __exit__(self, *exc):
        L.lib().kg_set_tc_terms(self.old)
        return False


def as_i32(t, device=None):
    """int32 contiguous view/copy of an index tensor (reference tensors are int64)."""
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(t)
    if device is not None and t.device != torch.device(device):
        t = t.to(device, non_blocking=True)
    if t.dtype != torch.int32:
        t = t.to(torch.int32)
    return _c(t)


# ---------------------------------------------------------------------------------------------
# graph index (a1)
# ---------------------------------------------------------------------------------------------
class GraphIndex:
    """Device-resident edge orderings for one (graph, etypes, norm) triple."""

    __slots__ = ("n_nodes", "n_edges", "n_etypes", "row_ptr", "fwd_pack", "col_ptr", "bwd_pack",
                 "rel_ptr", "rel_pack", "e_src", "e_dst", "e_type", "node_norm", "e_norm", "_tiled")

    def __init__(self, n_nodes, n_edges, n_etypes, device):
        self.n_nodes, self.n_edges, self.n_etypes = int(n_nodes), int(n_edges), int(n_etypes)
        i32 = dict(dtype=torch.int32, device=device)
        self.row_ptr = torch.empty(n_nodes + 1, **i32)
        self.col_ptr = torch.empty(n_nodes + 1, **i32)
        self.rel_ptr = torch.empty(n_etypes + 1, **i32)
        self.fwd_pack = self.bwd_pack = None      # dst-major / src-major lists: built on request only
        self.rel_pack = torch.empty((max(n_edges, 1), 4), **i32)
        self.e_src = self.e_dst = self.e_type = self.node_norm = self.e_norm = None
        self._tiled = {}

    def ensure_node_major(self):
        """Build the dst-major (fwd_pack + row_ptr) and src-major (bwd_pack + col_ptr) lists as well
        (the basis id-feature kernel walks destinations; message passing itself only needs rel_pack)."""
        if self.fwd_pack is None:
            full = graph_index(self.e_src, self.e_dst, self.e_type, self._norm_per_edge(), self.n_nodes,
                               self.n_etypes, node_major=True)
            self.fwd_pack, self.bwd_pack, self.row_ptr, self.col_ptr = full.fwd_pack, full.bwd_pack, full.row_ptr, full.col_ptr
        return self

    def _norm_per_edge(self):
        if self.e_norm is None and self.node_norm is not None:
            self.e_norm = self.node_norm[self.e_dst.long()].contiguous()
        return self.e_norm

    def tiled_rel_pack(self, by_src, tile_nodes):
        """kg_graph_rel_tiled: relation-major records grouped by node tile (built once, cached)."""
        key = (int(bool(by_src)), int(tile_nodes))
        if key not in self._tiled:
            self._norm_per_edge()
            pack = torch.empty_like(self.rel_pack)
            ws = L.workspace(L.lib().kg_graph_rel_tiled_workspace_bytes(self.n_edges), pack.device)
            L.call("kg_graph_rel_tiled", L.i32(self.e_src), L.i32(self.e_dst), L.i32(self.e_type),
                   L.f32(self.e_norm), self.n_edges, self.n_nodes, self.n_etypes, key[1], key[0],
                   L.i32(pack), L.ptr(ws), ws.numel(), L.stream())
            self._tiled[key] = pack
        return self._tiled[key]


# Rows that message passing reduces into (agg[dst] forward, x[src] + dx[src] backward) are kept
# L2-resident: graphs whose reduced matrix exceeds this budget are walked tile by tile.
L2_TILE_BYTES = int(os.environ.get("KG_L2_TILE_MB", "32")) << 20   # reduced rows of one node tile (tuning knob)
L2_RESIDENT_BYTES = 96 << 20        # a reduced matrix up to this size is left untiled (126 MB L2)
L2_STREAM_BYTES = 64 << 20          # a gathered matrix larger than this is read with evict-first
HINT_STREAM_X, HINT_STREAM_D, HINT_TILE_RESIDENT = 1, 2, 4


TILE_MIN_EDGES_PER_ROW = 4           # below this, a tile's rows are touched too rarely for L2 residency to pay


def _rel_order(gi, by_src, n_rows, row_bytes):
    """the relation-major record list to walk for a reduction into ``n_rows`` rows of ``row_bytes``.  Node tiling
    trades relation-run length (block weights reloaded, weight gradients flushed once per (tile, relation) group)
    for L2 residency of the reduced rows; with few edges per reduced row - the backward pass of a destination-
    partitioned rank spreads its 1/P of the edges over ALL source rows (1.6 edges per row at P = 8) - there is
    nothing to keep resident and the groups shrink to a dozen edges, so the plain relation-major list is walked."""
    if n_rows * row_bytes <= max(L2_TILE_BYTES, L2_RESIDENT_BYTES) or gi.n_edges < TILE_MIN_EDGES_PER_ROW * n_rows:
        return gi.rel_pack
    return gi.tiled_rel_pack(by_src, max(L2_TILE_BYTES // row_bytes, 256))


def graph_index(e_src, e_dst, e_type, e_norm, n_nodes, n_etypes, node_major=False):
    """kg_graph_index: relation-major edge records (and, with ``node_major``, the dst-major and
    src-major lists) for an edge list given in the reference's order (DGLGraph.add_edges + etypes +
    norm, kgvae/utils.py:141-148)."""
    dev = e_src.device
    E = int(e_src.numel())
    gi = GraphIndex(n_nodes, E, n_etypes, dev)
    if node_major:
        gi.fwd_pack = torch.empty((max(E, 1), 4), dtype=torch.int32, device=dev)
        gi.bwd_pack = torch.empty((max(E, 1), 4), dtype=torch.int32, device=dev)
    gi.e_src, gi.e_dst, gi.e_type = e_src, e_dst, e_type
    ws = L.workspace(L.lib().kg_graph_index_workspace_bytes(E), dev)
    norm = None if e_norm is None else _c(e_norm.reshape(-1).to(torch.float32))
    gi.e_norm = norm
    L.call("kg_graph_index", L.i32(e_src), L.i32(e_dst), L.i32(e_type), L.f32(norm), E, n_nodes,
           n_etypes, L.i32(gi.row_ptr), L.i32(gi.fwd_pack), L.i32(gi.col_ptr), L.i32(gi.bwd_pack),
           L.i32(gi.rel_ptr), L.i32(gi.rel_pack), L.ptr(ws), ws.numel(), L.stream())
    return gi


def graph_build(src, rel, dst, n_nodes, n_rels, node_major=False):
    """kg_graph_build: the whole of utils.build_graph_from_triplets + node_norm_to_edge_norm
    (kgvae/utils.py:127-150, kgvae/link_predict.py:95-100) on the device."""
    dev = src.device
    T = int(src.numel())
    gi = GraphIndex(n_nodes, 2 * T, 2 * n_rels, dev)
    i32 = dict(dtype=torch.int32, device=dev)
    if node_major:
        gi.fwd_pack = torch.empty((max(2 * T, 1), 4), **i32)
        gi.bwd_pack = torch.empty((max(2 * T, 1), 4), **i32)
    gi.e_src, gi.e_dst, gi.e_type = (torch.empty(max(2 * T, 1), **i32) for _ in range(3))
    gi.node_norm = torch.empty(n_nodes, dtype=torch.float32, device=dev)
    ws = L.workspace(L.lib().kg_graph_build_workspace_bytes(T), dev)
    L.call("kg_graph_build", L.i32(src), L.i32(rel), L.i32(dst), T, n_nodes, n_rels,
           L.i32(gi.e_src), L.i32(gi.e_dst), L.i32(gi.e_type), L.i32(gi.row_ptr), L.f32(gi.node_norm),
           L.i32(gi.fwd_pack), L.i32(gi.col_ptr), L.i32(gi.bwd_pack), L.i32(gi.rel_ptr),
           L.i32(gi.rel_pack), L.ptr(ws), ws.numel(), L.stream())
    gi.e_src, gi.e_dst, gi.e_type = gi.e_src[:2 * T], gi.e_dst[:2 * T], gi.e_type[:2 * T]
    return gi


def sample_relabel(picked, num_nodes, cap):
    """kg_sample_relabel: np.unique((src, dst), return_inverse=True) of B sampled triples (kgvae/utils.py:85-124)
    with a fixed node budget ``cap``.  ``picked``: int32 [B, 3] on the device.  Returns (node_id int32 [cap],
    src, rel, dst int32 [B], n_valid int32 [1]): rows 0 .. n_valid-1 of node_id are the distinct ids in ascending
    order, row i >= n_valid holds entity i (padding).  No host read-back: capturable."""
    picked = _c(picked)
    dev = picked.device
    B = int(picked.shape[0])
    i32 = dict(dtype=torch.int32, device=dev)
    node_id = torch.empty(int(cap), **i32)
    src, rel, dst = (torch.empty(B, **i32) for _ in range(3))
    n_valid = torch.empty(1, **i32)
    ws = L.workspace(L.lib().kg_sample_relabel_workspace_bytes(B), dev)
    L.call("kg_sample_relabel", L.i32(picked), B, int(num_nodes), int(cap), L.i32(node_id), L.i32(src), L.i32(rel),
           L.i32(dst), L.i32(n_valid), L.ptr(ws), ws.numel(), L.stream())
    return node_id, src, rel, dst, n_valid


NEIGHBOR_WORDS, NEIGHBOR_TRIES = 8, 6         # KG_NEIGHBOR_WORDS / KG_NEIGHBOR_TRIES of include/kgvae_b200.h


def neighbor_adjacency(triplets, num_nodes):
    """The adjacency lists of utils.get_adj_and_degrees as a device CSR, built by one stable sort of the 2T ends:
    ``adj_ptr`` int32 [N+1] and ``adj`` int32 [2T, 2] rows (edge id, other end), per entity in ascending edge id with
    the subject end first for a self-loop.  ``triplets``: int tensor [T, 3] on the device."""
    tri = _c(triplets).long()
    ends = tri[:, [0, 2]].reshape(-1)                   # s0, o0, s1, o1, ...: edge order, subject end first
    order = torch.sort(ends, stable=True).indices
    other = tri[:, [2, 0]].reshape(-1)[order]
    adj = torch.stack([order // 2, other], dim=1).to(torch.int32).contiguous()
    adj_ptr = torch.zeros(int(num_nodes) + 1, dtype=torch.int32, device=tri.device)
    adj_ptr[1:] = torch.cumsum(torch.bincount(ends, minlength=int(num_nodes)), 0)
    return adj_ptr, adj


def neighbor_sample_plan(num_nodes, n_triples, sample_size):
    """(samples drawn per launch, workspace bytes) of kg_neighbor_sample on the current device."""
    k, ws = ctypes.c_int(), ctypes.c_size_t()
    L.call("kg_neighbor_sample_plan", int(num_nodes), int(n_triples), int(sample_size), ctypes.byref(k),
           ctypes.byref(ws))
    return k.value, ws.value


def neighbor_sample(adj_ptr, adj, num_nodes, sample_size, words, out=None, fallbacks=None, workspace=None):
    """kg_neighbor_sample: one neighbourhood-expansion sample (kgvae/utils.py:33-76) of ``sample_size`` distinct
    triples per row of ``words`` (int32 [K, B, NEIGHBOR_WORDS], read as uniform 32-bit words).  Returns picks int32
    [K, B] (edge ids).  ``fallbacks``: optional int32 [K] that receives, per sample, the picks that needed the scan
    over unpicked entries.  Same procedure as the host sampler, not numpy's random stream; tests/neighbor_mirror.py is
    its specification.  No host read-back: capturable."""
    words = _c(words)
    K, B = int(words.shape[0]), int(sample_size)
    if words.shape[1:] != (B, NEIGHBOR_WORDS):
        raise ValueError(f"neighbor_sample: words must be [K, {B}, {NEIGHBOR_WORDS}], got {tuple(words.shape)}")
    dev = words.device
    if out is None:
        out = torch.empty(K, B, dtype=torch.int32, device=dev)
    if workspace is None:
        workspace = L.workspace(neighbor_sample_plan(num_nodes, adj.shape[0] // 2, B)[1], dev)
    L.call("kg_neighbor_sample", L.i32(adj_ptr), L.i32(adj), int(num_nodes), int(adj.shape[0]) // 2, B, K,
           L.i32(words), L.i32(out), L.i32(fallbacks), L.ptr(workspace), workspace.numel(), L.stream())
    return out


def valid_rows(n_rows, n_valid, device):
    """bool [n_rows]: row < n_valid (device scalar), for masked means over a padded node set."""
    return torch.arange(n_rows, device=device) < n_valid.reshape(())


# ---------------------------------------------------------------------------------------------
# dense GEMM helper
# ---------------------------------------------------------------------------------------------
class Prepared:
    """A matrix in the tensor-core GEMM's operand form (kg_gemm_prepare): split once, then usable by every product
    it takes part in, in either orientation.  Keeps the fp32 source for products too small for the tensor cores."""
    __slots__ = ("src", "buf", "shape", "device")

    def __init__(self, src):
        rows, cols = src.shape
        self.src, self.shape, self.device = src, src.shape, src.device
        nbytes = L.lib().kg_gemm_prep_bytes(rows, cols)
        self.buf = L.workspace(nbytes, src.device)
        L.call("kg_gemm_prepare", L.f32(src), src.stride(0), rows, cols, L.ptr(self.buf), nbytes, L.stream())


def uses_tensor_cores(M, N, K):
    return bool(L.lib().kg_gemm_f32_uses_tensor_cores(M, N, K))


def prepare(t, other_dim):
    """Prepared form of the 2-D fp32 matrix ``t`` when its products with a matrix whose free dimension is
    ``other_dim`` run on the tensor cores (all three extents >= 64 and a large enough volume); else ``t``."""
    if isinstance(t, Prepared):
        return t
    r, c = t.shape
    if min(r, c, other_dim) >= 64 and uses_tensor_cores(r, c, other_dim):
        return Prepared(t)
    return t


def gemm(a, b, out, trans_a=False, trans_b=False, bias=None, addend=None, relu=False, mask=None,
         accumulate=False):
    """out[M,N] (+)= epilogue(op(a) @ op(b)); a, b 2-D fp32 with contiguous rows or ``Prepared``, out 2-D fp32."""
    M, N = out.shape
    K = a.shape[0] if trans_a else a.shape[1]
    tag = f"kg_gemm_f32[{M}x{N}x{K},{'T' if trans_a else 'N'}{'T' if trans_b else 'N'}]"
    if uses_tensor_cores(M, N, K):
        pa = a if isinstance(a, Prepared) else Prepared(a)
        pb = b if isinstance(b, Prepared) else Prepared(b)
        nbytes = L.lib().kg_gemm_f32_prepared_workspace_bytes(M, N, K)
        ws = L.workspace(nbytes, out.device)
        L.call("kg_gemm_f32_prepared", L.ptr(pa.buf), int(trans_a), L.ptr(pb.buf), int(trans_b), L.f32(out),
               out.stride(0), M, N, K, L.f32(bias), L.f32(addend), int(relu), L.f32(mask), int(accumulate),
               L.ptr(ws), nbytes, L.stream(), tag=tag)
        return out
    a = a.src if isinstance(a, Prepared) else a
    b = b.src if isinstance(b, Prepared) else b
    L.call("kg_gemm_f32", L.f32(a), a.stride(0), int(trans_a), L.f32(b), b.stride(0), int(trans_b),
           L.f32(out), out.stride(0), M, N, K, L.f32(bias), L.f32(addend), int(relu), L.f32(mask),
           int(accumulate), None, 0, L.stream(), tag=tag)
    return out


def epilogue_only(out, bias=None, addend=None, relu=False, mask=None):
    """out = mask * act(addend + bias): the GEMM epilogue with an empty product (K = 0)."""
    M, N = out.shape
    L.call("kg_gemm_f32", None, 0, 0, None, 0, 0, L.f32(out), N, M, N, 0, L.f32(bias), L.f32(addend),
           int(relu), L.f32(mask), 0, None, 0, L.stream())
    return out


def colsum(x):
    rows, cols = x.shape
    out = torch.empty(cols, dtype=torch.float32, device=x.device)
    ws = L.workspace(L.lib().kg_colsum_workspace_bytes(rows, cols), x.device)
    L.call("kg_colsum", L.f32(x), rows, cols, L.f32(out), L.ptr(ws), ws.numel(), L.stream())
    return out


def act_dropout_bwd(g, out, mask, act, want_colsum=False):
    """grad wrt the pre-activation of out = dropout(act(pre)); with ``want_colsum`` also its column sums
    (the bias gradient) from the same pass."""
    gpre = torch.empty_like(out)
    if not want_colsum:
        L.call("kg_act_dropout_bwd", L.f32(g), L.f32(out), L.f32(mask), act, out.numel(), L.f32(gpre), L.stream())
        return gpre, None
    rows, cols = out.shape
    dbias = torch.empty(cols, dtype=torch.float32, device=out.device)
    ws = L.workspace(L.lib().kg_colsum_workspace_bytes(rows, cols), out.device)
    L.call("kg_act_dropout_bwd_colsum", L.f32(g), L.f32(out), L.f32(mask), act, rows, cols, L.f32(gpre), L.f32(dbias),
           L.ptr(ws), ws.numel(), L.stream())
    return gpre, dbias


def _sum_squares_rows(x, n_valid):
    """sum of squares over the first n_valid (device) rows of x [n, h] (kg_sum_squares_rows)."""
    out = torch.empty((), dtype=torch.float32, device=x.device)
    ws = L.workspace(L.lib().kg_reduce_workspace_bytes(x.numel()), x.device)
    L.call("kg_sum_squares_rows", L.f32(x), x.shape[0], x.shape[1], L.i32(n_valid), L.f32(out), L.ptr(ws), ws.numel(),
           L.stream())
    return out


def _reduce(name, x):
    out = torch.empty((), dtype=torch.float32, device=x.device)
    ws = L.workspace(L.lib().kg_reduce_workspace_bytes(x.numel()), x.device)
    L.call(name, L.f32(x), x.numel(), L.f32(out), L.ptr(ws), ws.numel(), L.stream())
    return out


# ---------------------------------------------------------------------------------------------
# a2  embedding
# ---------------------------------------------------------------------------------------------
class EmbeddingFn(torch.autograd.Function):
    """EmbeddingLayer.forward (kgvae/model.py:185-191)."""

    @staticmethod
    def forward(ctx, table, ids):
        table = _c(table)
        out = torch.empty((ids.numel(), table.shape[1]), dtype=torch.float32, device=table.device)
        L.call("kg_embedding_fwd", L.f32(table), L.i32(ids), ids.numel(), table.shape[1], L.f32(out),
               L.stream())
        ctx.save_for_backward(ids)
        ctx.shape = table.shape
        return out

    @staticmethod
    def backward(ctx, g):
        (ids,) = ctx.saved_tensors
        g = _c(g)
        grad = torch.zeros(ctx.shape, dtype=torch.float32, device=g.device)
        L.call("kg_embedding_bwd", L.f32(g), L.i32(ids), ids.numel(), ctx.shape[1], L.f32(grad),
               L.stream())
        return grad, None


# ---------------------------------------------------------------------------------------------
# a3  RelGraphConv("bdd") layer
# ---------------------------------------------------------------------------------------------
def _block_chunks(num_bases, si, so, n_chunks):
    """Split the diagonal blocks of a bdd layer into ``n_chunks`` contiguous ranges the column-chunk kernels accept
    (5x5 / 5x10 blocks, an even number of blocks per chunk, at most 64, chunk offsets 16-byte aligned); [] when the
    shape has no chunked kernels."""
    if n_chunks <= 1 or L.lib().kg_bdd_layouts_needed(num_bases, si, so) or num_bases % 4:
        return []
    units = num_bases // 4                  # cut at multiples of 4 blocks: 20 / 40 floats of x / agg -> 16-byte aligned
    if units < n_chunks:
        return []
    cuts = [0] + [4 * ((units * (c + 1)) // n_chunks) for c in range(n_chunks)]
    out = [(cuts[c], cuts[c + 1]) for c in range(n_chunks) if cuts[c + 1] > cuts[c]]
    return out if all(b1 - b0 <= 64 for b0, b1 in out) else []


class BddConvFn(torch.autograd.Function):
    """One RelGraphConv(bdd) layer: out = dropout(act(sum_e norm_e W_{r_e} x_src + h_bias +
    x @ loop_weight)) - DGL RelGraphConv.forward as constructed at kgvae/model.py:54-59.

    Order of work: the self-loop product (+ bias) is written FIRST, straight into the buffer the messages are
    then reduced into (so there is no zero-fill pass), and activation + dropout mask are applied in place at
    the end.  That order is what lets the destination-partitioned forms overlap their collective with the
    GEMM, which only needs the rows this rank owns:

    * ``part`` + ``gather``: ``x`` holds this rank's rows; the NCCL all-gather of all nodes' rows is started
      asynchronously, the self-loop GEMM runs meanwhile, message passing waits for the gather.  Backward:
      the reduce-scatter of the source gradients runs while the weight-gradient GEMM of the self-loop does.
    * ``peer`` (parallel.PeerRows) + ``part``: ``x`` holds only this rank's rows; they are published in the
      rank's peer-visible block and every rank's kernel gathers the source rows it needs straight from the
      owners' HBM over NVLink (no all-gather); the gradient wrt the sources is accumulated for all nodes and
      reduce-scattered to the owners.
    Edge sources are global ids, destinations local ids; the layer produces the rows of the owned nodes."""

    @staticmethod
    def forward(ctx, x, weight, loop_weight, h_bias, gi, num_bases, act, drop_mask, gather=False,
                peer=None, part=None):
        x, weight = _c(x), _c(weight)
        dev = x.device
        n_own, in_feat = x.shape
        R = weight.shape[0]
        si = in_feat // num_bases
        so = weight.shape[1] // (num_bases * si)
        out_feat = num_bases * so
        needs_layouts = bool(L.lib().kg_bdd_layouts_needed(num_bases, si, so))
        pending = None
        if peer is not None:
            if needs_layouts:
                raise RuntimeError("RelGraphConv: the peer-memory gather needs 5x5 / 5x10 blocks")
            peer.publish(x)
            n_src_rows = peer.blk * peer.world_size
        elif gather:
            from . import parallel
            chunks = _block_chunks(num_bases, si, so, getattr(part, "col_chunks", 1))
            if chunks:          # one asynchronous all-gather per COLUMN chunk, queued in order on NCCL's stream
                pending = [parallel.allgather_rows_start(x[:, b0 * si:b1 * si].contiguous(), part) for b0, b1 in chunks]
            else:
                pending = parallel.allgather_rows_start(x, part)      # NCCL, asynchronous
            n_src_rows = part.n_global
        else:
            if n_own != gi.n_nodes:
                raise RuntimeError(f"RelGraphConv: {n_own} feature rows for a graph of {gi.n_nodes} nodes")
            n_src_rows = n_own
        w_fwd = w_bwd = None
        if needs_layouts:
            w_fwd = torch.empty((R, si, out_feat), dtype=torch.float32, device=dev)
            w_bwd = torch.empty((R, so, in_feat), dtype=torch.float32, device=dev)
            L.call("kg_bdd_weight_layouts", L.f32(weight), R, num_bases, si, so, L.f32(w_fwd),
                   L.f32(w_bwd), L.stream())
        bias = None if h_bias is None else _c(h_bias)
        mask = None if drop_mask is None else _c(drop_mask)
        out = torch.empty((n_own, out_feat), dtype=torch.float32, device=dev)
        if loop_weight is not None:                   # out = x_own @ loop_weight + bias   (only local rows)
            loop_weight = _c(loop_weight)
            xp, lwp = prepare(x, out_feat), prepare(loop_weight, n_own)
            gemm(xp, lwp, out, bias=bias)
            ctx.prepared = (xp, lwp)   # reused by the backward products  g W_loop^T  and  x^T g
        else:
            epilogue_only(out, bias=bias) if bias is not None else out.zero_()
        pack = _rel_order(gi, 0, n_own, 4 * out_feat)
        x_chunks = []
        if isinstance(pending, list):
            # chunk c runs as soon as ITS columns of every node's row have arrived; the later chunks' gathers
            # proceed meanwhile (block-diagonal weights: a chunk of blocks reads only its own columns)
            for (b0, b1), pend in zip(chunks, pending):
                xc = pend.wait()
                x_chunks.append(xc)
                hints = (HINT_STREAM_X if xc.numel() * 4 > L2_STREAM_BYTES else 0) | \
                        (HINT_TILE_RESIDENT if pack is not gi.rel_pack else 0)
                L.call("kg_bdd_rel_fwd_cols", L.f32(xc), L.i32(pack), gi.n_edges, L.f32(weight), b0, b1 - b0, num_bases,
                       si, so, L.f32(out), hints, L.stream(), tag=f"kg_bdd_rel_fwd[{si}x{so}]")
            x_src = x
        else:
            x_src = x
            if pending is not None:
                x_src = pending.wait()                # [n_global, in] on this stream from here on
            src_args = (None, L.ptr(peer.ptrs), peer.blk) if peer is not None else (L.f32(x_src), None, 0)
            hints = (HINT_STREAM_X if n_src_rows * in_feat * 4 > L2_STREAM_BYTES else 0) | \
                    (HINT_TILE_RESIDENT if pack is not gi.rel_pack else 0)
            L.call("kg_bdd_rel_fwd", *src_args, L.i32(pack), gi.n_edges, L.f32(weight),
                   L.f32(w_fwd), num_bases, si, so, L.f32(out), hints, L.stream(), tag=f"kg_bdd_rel_fwd[{si}x{so}]")
        if act == 1 or mask is not None:              # activation + dropout mask, in place
            epilogue_only(out, addend=out, relu=(act == 1), mask=mask)
        ctx.x_chunks, ctx.chunks = x_chunks, (chunks if x_chunks else [])
        ctx.save_for_backward(x_src, weight, loop_weight, out, mask, w_bwd)
        ctx.gi, ctx.num_bases, ctx.act, ctx.si, ctx.so = gi, num_bases, act, si, so
        ctx.has_bias = h_bias is not None
        ctx.gather, ctx.n_own, ctx.peer, ctx.part = bool(gather), n_own, peer, part
        return out

    @staticmethod
    def backward(ctx, g):
        x, weight, loop_weight, out, mask, w_bwd = ctx.saved_tensors
        gi, B, si, so, peer, part = ctx.gi, ctx.num_bases, ctx.si, ctx.so, ctx.peer, ctx.part
        g = _c(g)
        chunked = bool(ctx.x_chunks)
        lo = part.lo if (ctx.gather and not chunked) else 0
        gpre, dbias_fused = act_dropout_bwd(g, out, mask, ctx.act, want_colsum=ctx.has_bias)
        dx = dw = dloop = dbias = None
        xp = lwp = None
        if loop_weight is not None:
            xp, lwp = ctx.prepared
        gp = prepare(gpre, x.shape[1]) if loop_weight is not None else gpre
        pending = None
        if chunked and (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]):
            from . import parallel
            want_dx = ctx.needs_input_grad[0]
            dw = torch.zeros_like(weight)
            own_dx = None
            if want_dx and loop_weight is not None:     # self-loop part of the input gradient (local rows only)
                own_dx = torch.empty((ctx.n_own, x.shape[1]), dtype=torch.float32, device=x.device)
                gemm(gp, lwp, own_dx, trans_b=True)
            pending = []
            for (b0, b1), xc in zip(ctx.chunks, ctx.x_chunks):
                dxc = torch.zeros_like(xc) if want_dx else None
                pack = _rel_order(gi, 1, xc.shape[0], (8 if want_dx else 4) * xc.shape[1])
                hints = (HINT_STREAM_D if gpre.numel() * 4 > L2_STREAM_BYTES else 0) | \
                        (HINT_TILE_RESIDENT if pack is not gi.rel_pack else 0)
                L.call("kg_bdd_rel_bwd_cols", L.f32(xc), L.f32(gpre), L.i32(pack), gi.n_edges, L.f32(weight), b0, b1 - b0,
                       B, si, so, L.f32(dxc), L.f32(dw), hints, L.stream(), tag=f"kg_bdd_rel_bwd[{si}x{so}]")
                if want_dx:
                    if own_dx is not None:
                        dxc[part.lo:part.lo + ctx.n_own] += own_dx[:, b0 * si:b1 * si]
                    # this chunk's source gradients travel while the next chunk computes
                    pending.append(parallel.reduce_scatter_rows_start(dxc, part))
            if not ctx.needs_input_grad[1]:
                dw = None
        elif ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            if peer is not None:       # source rows are still in the peers' blocks (published in forward)
                n_src_rows = peer.blk * peer.world_size
                src_args = (None, L.ptr(peer.ptrs), peer.blk)
            else:
                n_src_rows, src_args = x.shape[0], (L.f32(x), None, 0)
            dx = torch.zeros((n_src_rows, x.shape[1]), dtype=torch.float32, device=x.device) \
                if ctx.needs_input_grad[0] else None
            dw = torch.zeros_like(weight)
            # walked by source tile: x[src] and dx[src] stay L2-resident, dagg[dst] is the gathered row
            pack = _rel_order(gi, 1, n_src_rows, (8 if dx is not None else 4) * x.shape[1])
            hints = (HINT_STREAM_D if gpre.numel() * 4 > L2_STREAM_BYTES else 0) | \
                    (HINT_TILE_RESIDENT if pack is not gi.rel_pack and peer is None else 0)
            L.call("kg_bdd_rel_bwd", *src_args, L.f32(gpre), L.i32(pack), gi.n_edges, L.f32(weight), L.f32(w_bwd),
                   B, si, so, L.f32(dx), L.f32(dw), hints, L.stream(), tag=f"kg_bdd_rel_bwd[{si}x{so}]")
            if dx is not None and loop_weight is not None:
                own_lo = peer.rank * peer.blk if peer is not None else lo
                gemm(gp, lwp, dx[own_lo:own_lo + ctx.n_own], trans_b=True, accumulate=True)
            if dx is not None and (peer is not None or ctx.gather):
                # every rank holds partial sums for all nodes: reduce-scatter to the owners, asynchronously -
                # the weight-gradient GEMM below does not depend on it
                from . import parallel
                pending = parallel.reduce_scatter_rows_start(dx, part)
            if not ctx.needs_input_grad[1]:
                dw = None
        if loop_weight is not None and ctx.needs_input_grad[2]:
            dloop = torch.empty_like(loop_weight)
            gemm(xp, gp, dloop, trans_a=True)
        if ctx.has_bias and ctx.needs_input_grad[3]:
            dbias = dbias_fused
        if isinstance(pending, list):
            dx = torch.cat([p_.wait() for p_ in pending], dim=1) if pending else None
        elif pending is not None:
            dx = pending.wait()
        return dx, dw, dloop, dbias, None, None, None, None, None, None, None


# ---------------------------------------------------------------------------------------------
# a5  heads + reparameterised sample
# ---------------------------------------------------------------------------------------------
class ReparamFn(torch.autograd.Function):
    """gaussian_parameters + sample_gaussian (kgvae/utils.py:323-361): returns (mean, var, z)."""

    @staticmethod
    def forward(ctx, h2, eps):
        h2, eps = _c(h2), _c(eps)
        n, h = eps.shape
        zm, zv, z = (torch.empty_like(eps) for _ in range(3))
        L.call("kg_reparam_fwd", L.f32(h2), L.f32(eps), n, h, L.f32(zm), L.f32(zv), L.f32(z), L.stream())
        ctx.save_for_backward(h2, eps, zv)
        return zm, zv, z

    @staticmethod
    def backward(ctx, gm, gv, gz):
        h2, eps, zv = ctx.saved_tensors
        n, h = eps.shape
        gm = None if gm is None else _c(gm)
        gv = None if gv is None else _c(gv)
        gz = None if gz is None else _c(gz)
        dh2 = torch.empty_like(h2)
        L.call("kg_reparam_bwd", L.f32(h2), L.f32(eps), L.f32(zv), L.f32(gz), L.f32(gm), L.f32(gv),
               n, h, L.f32(dh2), L.stream())
        return dh2, None


# ---------------------------------------------------------------------------------------------
# a7  KL against the MoG prior
# ---------------------------------------------------------------------------------------------
class KlMogFn(torch.autograd.Function):
    """mean_n[log N(z; m, v) - log MoG(z)] (kgvae/model.py:82-87 without the scalar flow term,
    which the caller adds)."""

    @staticmethod
    def forward(ctx, z, z_mean, z_var, z_pre):
        z, z_mean, z_var = _c(z), _c(z_mean), _c(z_var)
        zp = _c(z_pre.reshape(-1, z_pre.shape[-1]))
        n, h = z.shape
        k = zp.shape[0] // 2
        dev = z.device
        ws = torch.empty((3, k, h), dtype=torch.float32, device=dev)
        rows = torch.empty(n, dtype=torch.float32, device=dev)
        resp = torch.empty((n, k), dtype=torch.float32, device=dev)
        L.call("kg_kl_mog_fwd", L.f32(z), L.f32(z_mean), L.f32(z_var), L.f32(zp), n, h, k, L.f32(ws),
               L.f32(rows), L.f32(resp), L.stream())
        ctx.save_for_backward(z, z_mean, z_var, zp, ws, resp)
        ctx.pre_shape = z_pre.shape
        return _reduce("kg_sum", rows) / n

    @staticmethod
    def backward(ctx, g):
        z, z_mean, z_var, zp, ws, resp = ctx.saved_tensors
        n, h = z.shape
        k = zp.shape[0] // 2
        dz, dm, dv = (torch.empty_like(z) for _ in range(3))
        dzp = torch.zeros_like(zp)
        # the upstream gradient is a device scalar: apply it with a broadcast multiply below
        L.call("kg_kl_mog_bwd", L.f32(z), L.f32(z_mean), L.f32(z_var), L.f32(zp), L.f32(ws),
               L.f32(resp), 1.0 / n, n, h, k, L.f32(dz), L.f32(dm), L.f32(dv), L.f32(dzp), L.stream())
        return dz * g, dm * g, dv * g, (dzp * g).view(ctx.pre_shape)


# ---------------------------------------------------------------------------------------------
# a6  IAF pieces
# ---------------------------------------------------------------------------------------------
class LinearFn(torch.autograd.Function):
    """y = [relu](x @ w^T + b): MaskedLinear (+ the in-place ReLU after it) with the masked
    weight precomputed - and, as ``wp``, split for the tensor cores - once per MADE call
    (kgvae/flow_network.py:15,53-63)."""

    @staticmethod
    def forward(ctx, x, w, b, relu, wp=None):
        x, w = _c(x), _c(w)
        if not isinstance(wp, Prepared) or wp.src.data_ptr() != w.data_ptr():
            wp = prepare(w, x.shape[0])
        xp = prepare(x, w.shape[0])
        y = torch.empty((x.shape[0], w.shape[0]), dtype=torch.float32, device=x.device)
        gemm(xp, wp, y, trans_b=True, bias=None if b is None else _c(b), relu=relu)
        ctx.save_for_backward(x, w, y if relu else None)
        ctx.prepared = (xp, wp)        # the split operands serve the two backward products as they are
        ctx.relu, ctx.has_bias = relu, b is not None
        return y

    @staticmethod
    def backward(ctx, g):
        x, w, y = ctx.saved_tensors
        g = _c(g)
        db_fused = None
        if ctx.relu:                 # ReLU backward and the bias gradient in one pass over g
            g, db_fused = act_dropout_bwd(g, y, None, 1, want_colsum=ctx.has_bias and ctx.needs_input_grad[2])
        dx = dw = db = None
        xp, wp = ctx.prepared
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = db_fused if db_fused is not None else colsum(g)
        gp = prepare(g, x.shape[1])
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            gemm(gp, wp, dx)
        if ctx.needs_input_grad[1]:
            dw = torch.empty_like(w)
            gemm(gp, xp, dw, trans_a=True)
        return dx, dw, db, None, None


class IafUpdateFn(torch.autograd.Function):
    """One pass of MADE.forward's update x[:, idx] = z[:, idx] * exp(alpha + mu) and, on request,
    log_det = sum_j alpha_j (kgvae/flow_network.py:93-96).  ``col_mult`` [d] int32 counts how often
    each column occurs in ``idx`` (0: column keeps ``x_old``; see kg_iaf_update_bwd)."""

    @staticmethod
    def forward(ctx, z, net_out, x_old, col_mult, want_log_det):
        z, net_out, x_old = _c(z), _c(net_out), _c(x_old)
        n, d = z.shape
        x_new = torch.empty_like(z)
        log_det = torch.empty(n, dtype=torch.float32, device=z.device) if want_log_det else None
        L.call("kg_iaf_update_fwd", L.f32(z), L.f32(net_out), L.f32(x_old), L.i32(col_mult), n, d,
               L.f32(x_new), L.f32(log_det), L.stream())
        ctx.save_for_backward(z, net_out, col_mult)
        return x_new, log_det

    @staticmethod
    def backward(ctx, gx, gl):
        z, net_out, col_mult = ctx.saved_tensors
        n, d = z.shape
        gx = torch.zeros_like(z) if gx is None else _c(gx)
        gl = None if gl is None else _c(gl)
        dz, dxo = torch.empty_like(z), torch.empty_like(z)
        dnet = torch.empty_like(net_out)
        L.call("kg_iaf_update_bwd", L.f32(z), L.f32(net_out), L.f32(gx), L.f32(gl), L.i32(col_mult),
               n, d, L.f32(dz), L.f32(dnet), L.f32(dxo), L.stream())
        return dz, dnet, dxo, None, None


class ReverseColumnsFn(torch.autograd.Function):
    """PermuteLayer (kgvae/flow_network.py:18-34): column reversal, its own inverse."""

    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        out = torch.empty_like(x)
        L.call("kg_reverse_columns", L.f32(x), x.shape[0], x.shape[1], L.f32(out), L.stream())
        return out

    @staticmethod
    def backward(ctx, g):
        return ReverseColumnsFn.apply(g)


# ---------------------------------------------------------------------------------------------
# a9  DistMult + BCE + regulariser
# ---------------------------------------------------------------------------------------------
class TripletIndex:
    """(r, s)-ordered and, on request, (entity, r)-ordered views of one batch of triplets.  ``trailing``: the entity
    index covers only the TRAILING end of every triplet (S entries) - what the two-pass decoder gathers over."""

    def __init__(self, triplets, n_nodes, n_rels, entity_index=True, trailing=False):
        dev = triplets.device
        S = triplets.shape[0]
        i32 = dict(dtype=torch.int32, device=dev)
        self.n = S
        self.rs_rec = torch.empty((max(S, 1), 4), **i32)
        want = entity_index or trailing
        self.ent_ptr = torch.empty(n_nodes + 1, **i32) if want else None
        self.ent_pack = torch.empty((max(S if trailing else 2 * S, 1), 4), **i32) if want else None
        ws = L.workspace(L.lib().kg_triplet_index_workspace_bytes(S), dev)
        L.call("kg_triplet_index_trailing" if trailing else "kg_triplet_index", L.i32(triplets), S, n_nodes, n_rels,
               L.i32(self.rs_rec), L.i32(self.ent_ptr), L.i32(self.ent_pack), L.ptr(ws), ws.numel(), L.stream(),
               tag="kg_triplet_index")


# None: two passes when z is far larger than L2 (a reduction into a random row of z's gradient is then a DRAM
# read-modify-write: 6 KB of compulsory traffic per scored triplet instead of 4 KB; while z is L2-resident the fused
# single pass is faster - 1.63 ms against 2.1 ms at the FB15k-237 shape); True / False force one form (tests)
DECODER_TWO_PASS = None
DECODER_TWO_PASS_BYTES = 256 << 20


def distmult_bce_pass(z, w, triplets, labels, shift, want_dz):
    """DistMult score + BCE-with-logits (mean) over ``triplets`` and its whole backward in the forward pass
    (kgvae/link_predict.py:57-63,74-77): returns (out [2] = loss, sum of dloss/dscore; dw; dz or None).
    One fused pass when z is L2-resident; for a larger z the gradient of the trailing entity of every triplet is
    gathered over a (trailing entity, r) index instead of reduced (kg_distmult_bce_fwd_lead +
    kg_distmult_bwd_dz_trailing)."""
    S, (n, h) = triplets.shape[0], z.shape
    dev = z.device
    two_pass = DECODER_TWO_PASS
    if two_pass is None:
        two_pass = z.numel() * 4 > DECODER_TWO_PASS_BYTES
    two_pass = bool(two_pass) and want_dz and h % 4 == 0 and h <= 1024 and S > 0
    idx = TripletIndex(triplets, n, w.shape[0], entity_index=False, trailing=two_pass)
    g = torch.empty(max(S, 1), dtype=torch.float32, device=dev)
    dw = torch.zeros_like(w)
    dz = torch.zeros_like(z) if want_dz else None
    out = torch.empty(2, dtype=torch.float32, device=dev)             # loss, sum of g
    sh = None if shift is None else _c(shift.reshape(1).to(torch.float32))
    ws = L.workspace(L.lib().kg_distmult_bce_workspace_bytes(S), dev)
    L.call("kg_distmult_bce_fwd_lead" if two_pass else "kg_distmult_bce_fwd", L.f32(z), L.f32(w), L.i32(idx.rs_rec),
           L.f32(labels), S, h, L.f32(sh), None, L.f32(g), L.f32(dw), L.f32(dz), L.ptr(out[0:1]), L.ptr(out[1:2]),
           L.ptr(ws), ws.numel(), L.stream(), tag="kg_distmult_bce_fwd")
    if two_pass:
        L.call("kg_distmult_bwd_dz_trailing", L.f32(z), L.f32(w), L.f32(g), L.i32(idx.ent_ptr), L.i32(idx.ent_pack),
               n, h, L.f32(dz), L.stream())
    return out, dw, dz


class DistMultScoreFn(torch.autograd.Function):
    """score_i = sum_d z[s,d] w[r,d] z[o,d] (+ shift): LinkPredict.calc_score and the
    flow_log_prob shift of get_loss (kgvae/link_predict.py:57-63,75-76)."""

    @staticmethod
    def forward(ctx, z, w, triplets, shift):
        z, w = _c(z), _c(w)
        S = triplets.shape[0]
        score = torch.empty(S, dtype=torch.float32, device=z.device)
        sh = None if shift is None else _c(shift.reshape(1).to(torch.float32))
        L.call("kg_distmult_score", L.f32(z), L.f32(w), L.i32(triplets), S, z.shape[1], L.f32(sh),
               L.f32(score), L.stream())
        ctx.save_for_backward(z, w, triplets)
        ctx.shift_shape = None if shift is None else shift.shape
        return score

    @staticmethod
    def backward(ctx, g):
        z, w, triplets = ctx.saved_tensors
        g = _c(g)
        S, h = triplets.shape[0], z.shape[1]
        dz = dw = dshift = None
        idx = TripletIndex(triplets, z.shape[0], w.shape[0])
        if ctx.needs_input_grad[0]:
            dz = torch.empty_like(z)
            L.call("kg_distmult_bwd_dz", L.f32(z), L.f32(w), L.f32(g), L.i32(idx.ent_ptr),
                   L.i32(idx.ent_pack), z.shape[0], h, L.f32(dz), L.stream())
        if ctx.needs_input_grad[1]:
            dw = torch.zeros_like(w)
            L.call("kg_distmult_bwd_dw", L.f32(z), L.f32(g), L.i32(idx.rs_rec), S, h, L.f32(dw), L.stream())
        if ctx.shift_shape is not None and ctx.needs_input_grad[3]:
            dshift = _reduce("kg_sum", g).reshape(ctx.shift_shape)
        return dz, dw, None, dshift


class DistMultBceFn(torch.autograd.Function):
    """mean BCE-with-logits of the DistMult scores (+ shift) in one pass: the prediction term of
    LinkPredict.get_loss (kgvae/link_predict.py:74-77).  The forward kernel also produces
    dloss/dscore and the gradients wrt w_relation and (when z needs one) wrt z: each triplet's
    rows are in registers once, for the score and for all three gradients."""

    @staticmethod
    def forward(ctx, z, w, triplets, labels, shift):
        z, w, labels = _c(z), _c(w), _c(labels)
        out, dw, dz = distmult_bce_pass(z, w, triplets, labels, shift, ctx.needs_input_grad[0])
        ctx.save_for_backward(dw, dz, out)
        ctx.shift_shape = None if shift is None else shift.shape
        return out[0].clone()

    @staticmethod
    def backward(ctx, go):
        dw, dz, out = ctx.saved_tensors
        dzo = dwo = dshift = None
        if ctx.needs_input_grad[0]:
            dzo = dz * go
        if ctx.needs_input_grad[1]:
            dwo = dw * go
        if ctx.shift_shape is not None and ctx.needs_input_grad[4]:
            dshift = (out[1] * go).reshape(ctx.shift_shape)
        return dzo, dwo, None, None, dshift


class PartitionedDistMultBceFn(torch.autograd.Function):
    """DistMultBceFn for destination-partitioned training: this rank's rows of z go in, its share of the triplets
    (global entity ids) is scored against the all-gathered z.  Both collectives are taken off the critical path:
    ``pending_z`` is the asynchronous all-gather the caller started before its local loss terms (KL, regulariser),
    and the reduce-scatter of dz - which the fused kernel already produced in the FORWARD pass - is started right
    after the kernel and only waited for when backward needs the rows (the upstream scalar is applied afterwards:
    the reduction is linear)."""

    @staticmethod
    def forward(ctx, z_local, w, triplets, labels, shift, part, pending_z):
        from . import parallel
        z = pending_z.wait()                                  # [n_global, h]
        w, labels = _c(w), _c(labels)
        out, dw, dz = distmult_bce_pass(z, w, triplets, labels, shift, True)
        ctx.pending_dz = parallel.reduce_scatter_rows_start(dz, part) if ctx.needs_input_grad[0] else None
        ctx.save_for_backward(dw, out)
        ctx.shift_shape = None if shift is None else shift.shape
        return out[0].clone()

    @staticmethod
    def backward(ctx, go):
        dw, out = ctx.saved_tensors
        dzo = dwo = dshift = None
        if ctx.pending_dz is not None:
            dzo = ctx.pending_dz.wait() * go
            ctx.pending_dz = None
        if ctx.needs_input_grad[1]:
            dwo = dw * go
        if ctx.shift_shape is not None and ctx.needs_input_grad[4]:
            dshift = (out[1] * go).reshape(ctx.shift_shape)
        return dzo, dwo, None, None, dshift, None, None


class LossHeadFn(torch.autograd.Function):
    """The loss head of LinkPredict.get_loss in one autograd node (kgvae/link_predict.py:74-91):

        pred = mean BCE-with-logits(DistMult(z, w, triplets) + shift, labels)      (kg_distmult_bce_fwd)
        reg  = mean(z^2) + mean(w^2)                                               (kg_sum_squares)
        kl   = mean_n[log N(z; m, v) - log MoG(z)]                                 (kg_kl_mog_fwd)
        loss = pred + reg_param * reg + kl_param * kl

    Returns (loss, pred, reg, kl).  As separate Functions these three terms each produced their own [n, h]
    gradient wrt z, scaled it by the upstream scalar with an elementwise multiply, and autograd added the three
    up: ten elementwise passes over 29 MB matrices.  Here backward forms the total in the KL backward pass
    (kg_kl_mog_bwd_fused): dz = c_kl dKL/dz + c_pred dz_pred + c_reg (2 / n h) z, coefficients on the device.
    The scalar flow terms (flow_log_prob in the scores' shift and in the KL) stay with the caller.

    ``n_valid`` (int32 device [1], optional): only the first n_valid rows of z are nodes, the rest pad a sampled
    subgraph to a fixed node budget (utils.SampledDeviceSampler).  KL and regulariser are then means over the valid
    rows (kg_kl_mog_fwd_rows, kg_sum_squares_rows, kg_kl_mog_bwd_fused_rows) and the gradient rows of the padding
    are exactly zero; the triplets must only reference valid rows."""

    @staticmethod
    def forward(ctx, z, z_mean, z_var, z_pre, w, triplets, labels, shift, reg_param, kl_param, n_valid=None):
        z, w, labels = _c(z), _c(w), _c(labels)
        S, (n, h) = triplets.shape[0], z.shape
        dev = z.device
        out, dw, dz_pred = distmult_bce_pass(z, w, triplets, labels, shift, True)       # out: pred loss, sum of g
        pred = out[0].clone()
        if n_valid is None:
            reg = _reduce("kg_sum_squares", z) / z.numel() + _reduce("kg_sum_squares", w) / w.numel()
        else:
            n_valid = _c(n_valid.reshape(1).to(torch.int32))
            nv_f = n_valid.reshape(()).to(torch.float32)
            reg = _sum_squares_rows(z, n_valid) / (nv_f * h) + _reduce("kg_sum_squares", w) / w.numel()
        use_kl = kl_param > 0 and z_mean is not None
        if use_kl:
            z_mean, z_var = _c(z_mean), _c(z_var)
            zp = _c(z_pre.reshape(-1, z_pre.shape[-1]))
            k = zp.shape[0] // 2
            pws = torch.empty((3, k, h), dtype=torch.float32, device=dev)
            rows = torch.empty(n, dtype=torch.float32, device=dev)
            resp = torch.empty((n, k), dtype=torch.float32, device=dev)
            if n_valid is None:
                L.call("kg_kl_mog_fwd", L.f32(z), L.f32(z_mean), L.f32(z_var), L.f32(zp), n, h, k, L.f32(pws),
                       L.f32(rows), L.f32(resp), L.stream())
                kl = _reduce("kg_sum", rows) / n
            else:                                           # padding rows: kl_rows = 0
                L.call("kg_kl_mog_fwd_rows", L.f32(z), L.f32(z_mean), L.f32(z_var), L.f32(zp), n, h, k,
                       L.i32(n_valid), L.f32(pws), L.f32(rows), L.f32(resp), L.stream())
                kl = _reduce("kg_sum", rows) / nv_f
            ctx.save_for_backward(z, w, dz_pred, dw, out, z_mean, z_var, zp, pws, resp)
            loss = pred + reg_param * reg + kl_param * kl
        else:
            kl = torch.zeros((), dtype=torch.float32, device=dev)
            ctx.save_for_backward(z, w, dz_pred, dw, out)
            loss = pred + reg_param * reg
        ctx.n_valid = n_valid
        ctx.use_kl, ctx.reg_param, ctx.kl_param = use_kl, float(reg_param), float(kl_param)
        ctx.shift_shape = None if shift is None else shift.shape
        ctx.pre_shape = None if z_pre is None else z_pre.shape
        return loss, pred, reg, kl

    @staticmethod
    def backward(ctx, g_loss, g_pred, g_reg, g_kl):
        saved = ctx.saved_tensors
        z, w, dz_pred, dw, out = saved[:5]
        n, h = z.shape
        zero = torch.zeros((), dtype=torch.float32, device=z.device)
        g_loss, g_pred, g_reg, g_kl = ((zero if t is None else t.reshape(()).to(torch.float32))
                                       for t in (g_loss, g_pred, g_reg, g_kl))
        c_pred = g_loss + g_pred
        c_reg = g_loss * ctx.reg_param + g_reg
        c_kl = g_loss * ctx.kl_param + g_kl
        nv = ctx.n_valid
        # the regulariser's d mean(z^2) / dz = 2 z / (rows h): rows = n, or the valid rows of a padded node set
        c_z = c_reg * (2.0 / z.numel()) if nv is None else c_reg * 2.0 / (nv.reshape(()).to(torch.float32) * h)
        dm = dv = dzp = None
        if ctx.use_kl:
            z_mean, z_var, zp, pws, resp = saved[5:]
            k = zp.shape[0] // 2
            coefs = torch.stack([c_kl, c_pred, c_z]).contiguous()
            dz, dm, dv = (torch.empty_like(z) for _ in range(3))
            dzp = torch.zeros_like(zp)
            if nv is None:
                L.call("kg_kl_mog_bwd_fused", L.f32(z), L.f32(z_mean), L.f32(z_var), L.f32(zp), L.f32(pws),
                       L.f32(resp), 1.0 / n, n, h, k, L.f32(coefs), L.f32(dz_pred), L.f32(dz), L.f32(dm), L.f32(dv),
                       L.f32(dzp), L.stream(), tag="kg_kl_mog_bwd")
            else:                                           # padding rows: exact zeros, nothing into dz_pre
                L.call("kg_kl_mog_bwd_fused_rows", L.f32(z), L.f32(z_mean), L.f32(z_var), L.f32(zp), L.f32(pws),
                       L.f32(resp), n, h, k, L.i32(nv), L.f32(coefs), L.f32(dz_pred), L.f32(dz), L.f32(dm), L.f32(dv),
                       L.f32(dzp), L.stream(), tag="kg_kl_mog_bwd")
            dzp = dzp.view(ctx.pre_shape)
        else:
            dz = torch.addcmul(dz_pred * c_pred, z, c_z)
            if nv is not None:                              # padding rows of z must not reach the encoder
                dz = torch.where(valid_rows(n, nv, z.device).view(-1, 1), dz, 0.0)
        dwo = torch.addcmul(dw * c_pred, w, c_reg * (2.0 / w.numel()))
        dshift = (out[1] * c_pred).reshape(ctx.shift_shape) if ctx.shift_shape is not None else None
        return dz, dm, dv, dzp, dwo, None, None, dshift, None, None, None


class BceLogitsFn(torch.autograd.Function):
    """F.binary_cross_entropy_with_logits(score, labels), mean reduction (kgvae/link_predict.py:77)."""

    @staticmethod
    def forward(ctx, score, labels):
        score, labels = _c(score), _c(labels)
        n = score.numel()
        loss = torch.empty((), dtype=torch.float32, device=score.device)
        dscore = torch.empty_like(score)
        ws = L.workspace(L.lib().kg_reduce_workspace_bytes(n), score.device)
        L.call("kg_bce_logits_fwd", L.f32(score), L.f32(labels), n, L.f32(loss), L.f32(dscore),
               L.ptr(ws), ws.numel(), L.stream())
        ctx.save_for_backward(dscore)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dscore,) = ctx.saved_tensors
        return dscore * g, None


class MeanSquareFn(torch.autograd.Function):
    """torch.mean(x.pow(2)) (kgvae/link_predict.py:68-69).  ``n_valid`` (int32 device [1], optional): the mean over
    the first n_valid rows of x [n, h] only (a node set padded to a fixed budget); padding rows get zero gradient."""

    @staticmethod
    def forward(ctx, x, n_valid=None):
        x = _c(x)
        ctx.save_for_backward(x)
        if n_valid is None:
            ctx.n_valid = None
            return _reduce("kg_sum_squares", x) / x.numel()
        ctx.n_valid = _c(n_valid.reshape(1).to(torch.int32))
        return _sum_squares_rows(x, ctx.n_valid) / (ctx.n_valid.reshape(()).to(torch.float32) * x.shape[1])

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        nv = ctx.n_valid
        if nv is None:
            return x * (g * (2.0 / x.numel())), None
        dx = x * (g * 2.0 / (nv.reshape(()).to(torch.float32) * x.shape[1]))
        return torch.where(valid_rows(x.shape[0], nv, x.device).view(-1, 1), dx, 0.0), None


# ---------------------------------------------------------------------------------------------
# a10  ranks
# ---------------------------------------------------------------------------------------------
def distmult_rank(emb, w, a, r, b, shift=None, cand_range=None, filt_ptr=None, filt_idx=None, tc_scores=None):
    """0-indexed raw (or filtered) rank of b_i among all entities for queries (a_i, r_i):
    utils.perturb_and_get_rank + sort_and_rank (kgvae/utils.py:180-221) without the score matrix.
    ``tc_scores`` (tests only): [M, hi - lo] fp32 tensor that receives the tensor-core scores."""
    emb, w = _c(emb.detach()), _c(w.detach())
    M, (V, h) = a.numel(), emb.shape
    dev = emb.device
    lo, hi = (0, V) if cand_range is None else cand_range
    ranks = torch.empty(max(M, 1), dtype=torch.int32, device=dev)
    ws = L.workspace(L.lib().kg_distmult_rank_workspace_bytes(M, int(hi) - int(lo), h), dev)
    sh = None if shift is None else _c(torch.as_tensor(shift, dtype=torch.float32, device=dev).reshape(1))
    L.call("kg_distmult_rank", L.f32(emb), L.f32(w), L.i32(a), L.i32(r), L.i32(b), M, V, h, L.f32(sh),
           int(lo), int(hi), L.i32(filt_ptr), L.i32(filt_idx), L.ptr(ws), ws.numel(), L.i32(ranks),
           L.f32(tc_scores), L.stream())
    return ranks[:M]


def distmult_topk(emb, w, a, r, k=1, shift=None, filt_ptr=None, filt_idx=None, cand_range=None):
    """The ``k`` highest-scored tails of each query (a_i, r_i) among all entities, best first (ties by ascending
    entity id): utils.generate's ``score.argmax`` (kgvae/utils.py:245-288) generalised to top-k, without the
    score matrix.  ``filt_ptr`` / ``filt_idx``: per-query CSR of entities to leave out (ascending, duplicate-free;
    ``filter_lists``); a query with fewer than k other entities gets trailing -1.
    ``cand_range=(lo, hi)``: only entities [lo, hi) are candidates (one shard of a multi-GPU generation; the ids
    returned are global and the scores the same bits the unsharded call gives, so ``parallel.merge_topk`` of the
    shards' lists is exact).  Returns (idx int32 [M, k], score fp32 [M, k]), -1 / -inf past the eligible ones."""
    if (filt_ptr is None) != (filt_idx is None):
        raise ValueError("distmult_topk: a filter needs both filt_ptr and filt_idx")
    emb, w = _c(emb.detach()), _c(w.detach())
    M, (V, h) = a.numel(), emb.shape
    dev = emb.device
    idx = torch.empty((max(M, 1), k), dtype=torch.int32, device=dev)
    score = torch.empty((max(M, 1), k), dtype=torch.float32, device=dev)
    lo, hi = (0, V) if cand_range is None else (int(cand_range[0]), int(cand_range[1]))
    ws = L.workspace(L.lib().kg_distmult_topk_workspace_bytes(M, hi - lo, h, k), dev)
    sh = None if shift is None else _c(torch.as_tensor(shift, dtype=torch.float32, device=dev).reshape(1))
    L.call("kg_distmult_topk_shard", L.f32(emb), L.f32(w), L.i32(a), L.i32(r), M, V, h, L.f32(sh), int(k), lo, hi,
           L.i32(filt_ptr), L.i32(filt_idx), L.ptr(ws), ws.numel(), L.i32(idx), L.f32(score), L.stream())
    return idx[:M], score[:M]


# ---------------------------------------------------------------------------------------------
# filter lists (device counterpart of utils.build_filter)
# ---------------------------------------------------------------------------------------------
FILTER_DIRECTIONS = {"object": 0, "subject": 1}     # KG_FILTER_OBJECT / KG_FILTER_SUBJECT of include/kgvae_b200.h


def filter_table(triplets, num_nodes, num_rels, direction):
    """kg_filter_table: the sorted, duplicate-free keys (a R + r) N + c of the known ``triplets`` (int tensor [T, 3]
    (s, r, o) on the device), a = s and c = o for ``direction="object"``, the other way round for "subject".
    Returns (table int64 [max(T, 1)], table_len int32 [1]) on the device."""
    tri = as_i32(triplets)
    dev, T = tri.device, int(tri.shape[0])
    table = torch.empty(max(T, 1), dtype=torch.int64, device=dev)
    n = torch.empty(1, dtype=torch.int32, device=dev)
    ws = L.workspace(L.lib().kg_filter_table_workspace_bytes(T), dev)
    L.call("kg_filter_table", L.i32(tri), T, int(num_nodes), int(num_rels), FILTER_DIRECTIONS[direction],
           L.ptr(table, torch.int64), L.i32(n), L.ptr(ws), ws.numel(), L.stream())
    return table, n


def filter_lists(table, table_len, num_nodes, num_rels, a, r):
    """kg_filter_count + kg_filter_gather: for queries (a_i, r_i) (int32 device tensors) the CSR (ptr int32 [M+1],
    idx int32 [ptr[M]]) of the entities their runs of ``table`` list - what utils.build_filter returns.  Reads the
    total back once to size idx."""
    a, r = as_i32(a), as_i32(r)
    dev, M = a.device, int(a.numel())
    ptr = torch.empty(M + 1, dtype=torch.int32, device=dev)
    total = ctypes.c_longlong()
    ws = L.workspace(L.lib().kg_filter_count_workspace_bytes(M), dev)
    L.call("kg_filter_count", L.ptr(table, torch.int64), L.i32(table_len), int(num_nodes), int(num_rels),
           L.i32(a), L.i32(r), M, L.i32(ptr), ctypes.byref(total), L.ptr(ws), ws.numel(), L.stream())
    idx = torch.empty(max(total.value, 1), dtype=torch.int32, device=dev)
    L.call("kg_filter_gather", L.ptr(table, torch.int64), L.i32(table_len), int(num_nodes), int(num_rels),
           L.i32(a), L.i32(r), M, L.i32(ptr), L.i32(idx), L.stream())
    return ptr, idx[:total.value]
