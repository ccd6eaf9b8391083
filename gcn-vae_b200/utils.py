"""Host-side helpers with the reference's names and behaviour (kgvae/utils.py).

* graph construction and sampling stay on the host and follow the reference's legacy global
  ``np.random`` call order, so sampled indices are bit-identical (SURVEY a11);
* evaluation (``calc_mrr`` / ``perturb_and_get_rank``) runs on the GPU through the fused
  score-and-count kernel - the reference moves the model to the CPU for this step;
* the probability helpers are kept for the cold paths (``get_mmd``, ``sample_z``); the hot path
  uses the fused kernels in ``ops``.
"""
import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F

from . import ops, parallel
from .graph import Graph


# --------------------------------------------------------------------------------------------
# graph construction (kgvae/utils.py:20-30,127-155)
# --------------------------------------------------------------------------------------------
def get_adj_and_degrees(num_nodes, triplets):
    """Adjacency lists [[edge id, neighbour], ...] per node and their lengths (utils.py:20-30),
    built with one stable sort instead of a Python loop over triplets."""
    triplets = np.asarray(triplets)
    n = len(triplets)
    ends = np.concatenate((triplets[:, 0], triplets[:, 2]))
    other = np.concatenate((triplets[:, 2], triplets[:, 0]))
    eid = np.concatenate((np.arange(n), np.arange(n)))
    # the reference appends (i, o) to s's list and (i, s) to o's list for i = 0..n-1 in turn
    order = np.lexsort((np.concatenate((np.zeros(n), np.ones(n))), eid, ends))
    degrees = np.bincount(ends, minlength=num_nodes)
    pairs = np.stack((eid[order], other[order]), axis=1)
    bounds = np.concatenate(([0], np.cumsum(degrees)))
    adj_list = [pairs[bounds[v]:bounds[v + 1]] for v in range(num_nodes)]
    return adj_list, degrees


def comp_deg_norm(g):
    in_deg = g.in_degrees(range(g.number_of_nodes())).float().numpy()
    with np.errstate(divide="ignore"):
        norm = 1.0 / in_deg
    norm[np.isinf(norm)] = 0
    return norm


def build_graph_from_triplets(num_nodes, num_rels, triplets):
    """Bidirectional graph with reverse relations ``rel + num_rels``, edges in ascending
    (dst, src, rel) order, and 1/in-degree node norms (utils.py:135-150).  ``np.lexsort``
    yields the same order as the reference's ``sorted(zip(dst, src, rel))``."""
    src, rel, dst = (np.asarray(a) for a in triplets)
    src, dst = np.concatenate((src, dst)), np.concatenate((dst, src))
    rel = np.concatenate((rel, rel + num_rels))
    order = np.lexsort((rel, src, dst))
    src, dst, rel = src[order], dst[order], rel[order]
    g = Graph()
    g.add_nodes(num_nodes)
    g.add_edges(src, dst)
    return g, rel, comp_deg_norm(g)


def build_test_graph(num_nodes, num_rels, edges):
    src, rel, dst = np.asarray(edges).transpose()
    return build_graph_from_triplets(num_nodes, num_rels, (src, rel, dst))


# --------------------------------------------------------------------------------------------
# sampling (kgvae/utils.py:33-124,158-171) - global np.random, reference call order
# --------------------------------------------------------------------------------------------
def sample_edge_uniform(adj_list, degrees, n_triplets, sample_size):
    return np.random.choice(np.arange(n_triplets), sample_size, replace=False)


def sample_edge_neighborhood(adj_list, degrees, n_triplets, sample_size):
    """Neighbourhood-expansion sampler (utils.py:33-76): same RNG calls, same picks."""
    edges = np.zeros(sample_size, dtype=np.int32)
    sample_counts = np.array(degrees).copy()
    picked = np.zeros(n_triplets, dtype=bool)
    seen = np.zeros(len(degrees), dtype=bool)
    node_ids = np.arange(len(degrees))
    for i in range(sample_size):
        weights = sample_counts * seen
        if np.sum(weights) == 0:
            weights = np.ones_like(weights)
            weights[np.where(sample_counts == 0)] = 0
        chosen_vertex = np.random.choice(node_ids, p=weights / np.sum(weights))
        chosen_adj = adj_list[chosen_vertex]
        seen[chosen_vertex] = True
        while True:
            edge_number, other_vertex = chosen_adj[np.random.choice(np.arange(chosen_adj.shape[0]))]
            if not picked[edge_number]:
                break
        edges[i] = edge_number
        picked[edge_number] = True
        sample_counts[chosen_vertex] -= 1
        sample_counts[other_vertex] -= 1
        seen[other_vertex] = True
    return edges


def negative_sampling(pos_samples, num_entity, negative_rate):
    """Corrupt the subject where u > 0.5, else the object (utils.py:158-171)."""
    n = len(pos_samples)
    total = n * negative_rate
    neg = np.tile(pos_samples, (negative_rate, 1))
    labels = np.zeros(n * (negative_rate + 1), dtype=np.float32)
    labels[:n] = 1
    values = np.random.randint(num_entity, size=total)
    coin = np.random.uniform(size=total)
    head = coin > 0.5
    neg[head, 0] = values[head]
    neg[~head, 2] = values[~head]
    return np.concatenate((pos_samples, neg)), labels


def generate_sampled_graph_and_labels(triplets, sample_size, split_size, num_rels, adj_list,
                                      degrees, negative_rate, sampler="uniform"):
    """Sample edges, relabel nodes, draw negatives, keep ``split_size`` of the edges as graph
    structure (utils.py:85-124).  Returns (g, uniq_v, rel, norm, samples, labels)."""
    if sampler == "uniform":
        picked = sample_edge_uniform(adj_list, degrees, len(triplets), sample_size)
    elif sampler == "neighbor":
        picked = sample_edge_neighborhood(adj_list, degrees, len(triplets), sample_size)
    else:
        raise ValueError("Sampler type must be either 'uniform' or 'neighbor'.")
    src, rel, dst = np.asarray(triplets)[picked].transpose()
    uniq_v, relabeled = np.unique((src, dst), return_inverse=True)
    src, dst = np.reshape(relabeled, (2, -1))
    samples, labels = negative_sampling(np.stack((src, rel, dst)).transpose(), len(uniq_v),
                                        negative_rate)
    keep = np.random.choice(np.arange(sample_size), size=int(sample_size * split_size), replace=False)
    g, rel, norm = build_graph_from_triplets(len(uniq_v), num_rels, (src[keep], rel[keep], dst[keep]))
    return g, uniq_v, rel, norm, samples, labels


def generate_sampled_graph_and_labels_device(triplets, sample_size, split_size, num_rels, negative_rate,
                                             generator=None, picked=None):
    """Opt-in DEVICE form of ``generate_sampled_graph_and_labels`` with the uniform edge sampler
    (kgvae/utils.py:79-124,158-171): ``sample_size`` training triples without replacement, nodes
    relabelled to 0..n-1 in ascending id order, ``negative_rate`` corruptions per positive (subject
    where u > 0.5, else object, replacement drawn among the n sampled nodes), ``split_size`` of the
    sampled edges kept as graph structure, bidirectional graph with 1 / in-degree norms.

    Everything stays on the GPU (torch's device generator + ``kg_graph_build``), so the step needs
    neither the host sampler nor the ~50 MB of host -> device copies.  The draws follow the same
    procedure but NOT numpy's random stream: use the host function when sampled indices must match
    the reference bit for bit.  ``triplets``: int tensor [T, 3] on the device.  ``picked``: optional precomputed
    edge sample (int tensor [sample_size] of distinct triple ids, e.g. ``NeighborEdgeBank.next()`` for the
    neighbourhood sampler) used instead of the uniform draw.

    Returns (g, node_id [n, 1] int64, edge_type int32 [E], edge_norm f32 [E, 1], samples int32
    [S, 3], labels f32 [S]) - the arguments of ``model(g, node_id, edge_type, edge_norm)`` and
    ``model.get_loss(g, embed, samples, labels)``."""
    if not triplets.is_cuda:
        raise RuntimeError("generate_sampled_graph_and_labels_device needs the triples on a CUDA device")
    dev = triplets.device
    B, rate = int(sample_size), int(negative_rate)
    if picked is None:
        picked = torch.randperm(triplets.shape[0], device=dev, generator=generator)[:B]
    tri = triplets[picked.long()].long()
    uniq_v, inv = torch.unique(torch.cat([tri[:, 0], tri[:, 2]]), return_inverse=True)
    n = int(uniq_v.numel())
    src, rel, dst = inv[:B], tri[:, 1], inv[B:]
    pos = torch.stack([src, rel, dst], dim=1)
    neg = pos.repeat(rate, 1)
    values = torch.randint(n, (B * rate,), device=dev, generator=generator)
    head = torch.rand(B * rate, device=dev, generator=generator) > 0.5
    neg[:, 0] = torch.where(head, values, neg[:, 0])
    neg[:, 2] = torch.where(head, neg[:, 2], values)
    samples = torch.cat([pos, neg]).to(torch.int32).contiguous()
    labels = torch.zeros(B * (rate + 1), dtype=torch.float32, device=dev)
    labels[:B] = 1
    keep = torch.randperm(B, device=dev, generator=generator)[:int(B * split_size)]
    i32 = lambda t: t.to(torch.int32).contiguous()
    gi = ops.graph_build(i32(src[keep]), i32(rel[keep]), i32(dst[keep]), n, int(num_rels))
    g = Graph()
    g._n = n
    g._dev_edges[dev] = (gi.e_src, gi.e_dst)
    edge_type = gi.e_type
    edge_norm = gi.node_norm[gi.e_dst.long()].view(-1, 1).contiguous()
    g.adopt_index(gi, edge_type, edge_norm, 2 * int(num_rels))
    return g, uniq_v.view(-1, 1), edge_type, edge_norm, samples, labels


class FullBatchDeviceSampler:
    """``generate_sampled_graph_and_labels_device`` for the case ``sample_size == len(triplets)`` (full-graph
    training: every step scores ALL training triples with fresh negatives and builds the graph from a fresh random
    ``split_size`` of them, kgvae/utils.py:79-124,158-171).  The sampled edge set is then always the whole training
    set, so the node relabelling is fixed and is computed once; a call to ``sample()`` draws the negatives and the
    graph split and returns tensors of FIXED shapes - ``node_id [n, 1]``, ``src`` / ``dst`` / ``etype [E]`` (int32,
    both directions), ``norm [E, 1]`` (1 / in-degree), ``samples [S, 3]`` (int32), ``labels [S]`` - with no host
    read-back, using only stream-ordered tensor ops: it can run inside a CUDA-graph capture
    (``link_predict.CapturedTrainStep(..., sampler=...)``), which makes a training step - sampler included - one
    replay.  Same procedure as the host sampler, not numpy's random stream."""

    def __init__(self, triplets, num_rels, negative_rate, split_size=0.5):
        if not triplets.is_cuda:
            raise RuntimeError("FullBatchDeviceSampler needs the triples on a CUDA device (no CPU fallback)")
        tri = triplets.long()
        B = tri.shape[0]
        uniq_v, inv = torch.unique(torch.cat([tri[:, 0], tri[:, 2]]), return_inverse=True)
        self.n = int(uniq_v.numel())                                  # the only host read-back, once
        self.num_rels, self.rate, self.B = int(num_rels), int(negative_rate), B
        self.keep_n = int(B * split_size)
        self.node_id = uniq_v.view(-1, 1)
        self.src, self.rel, self.dst = inv[:B].contiguous(), tri[:, 1].contiguous(), inv[B:].contiguous()
        self.pos = torch.stack([self.src, self.rel, self.dst], dim=1).to(torch.int32)
        self.neg_s, self.neg_r, self.neg_o = (t.repeat(self.rate) for t in (self.src, self.rel, self.dst))
        self.labels = torch.zeros(B * (self.rate + 1), dtype=torch.float32, device=tri.device)
        self.labels[:B] = 1
        self.n_edges, self.n_samples = 2 * self.keep_n, B * (self.rate + 1)

    def sample(self):
        dev = self.src.device
        m = self.B * self.rate
        values = torch.randint(self.n, (m,), device=dev)
        samples = _with_negatives(self.pos, self.neg_s, self.neg_r, self.neg_o, values)
        graph = _split_graph(self.src, self.rel, self.dst, self.keep_n, self.num_rels, self.n)
        return {"node_id": self.node_id, **graph, "samples": samples, "labels": self.labels}


def _with_negatives(pos, neg_s, neg_r, neg_o, values):
    """The positives followed by their corruptions (kgvae/utils.py:158-171): one draw decides per negative whether
    ``values`` replaces the subject (u > 0.5) or the object.  ``neg_*``: the positives' columns repeated."""
    head = torch.rand(values.shape[0], device=values.device) > 0.5
    neg = torch.stack([torch.where(head, values, neg_s), neg_r, torch.where(head, neg_o, values)], dim=1)
    return torch.cat([pos, neg.to(torch.int32)])


def _split_graph(src, rel, dst, keep_n, num_rels, n_nodes):
    """A uniform random ``keep_n`` of the positives as graph structure, in both directions with reverse relation ids,
    and 1 / in-degree norms over ``n_nodes`` nodes (0 edges: norm 1, unused) - kgvae/utils.py:115-150."""
    dev = src.device
    keep = torch.argsort(torch.rand(src.shape[0], device=dev))[:keep_n]       # a uniform random subset
    s, r, d = src[keep], rel[keep], dst[keep]
    src2, dst2 = torch.cat([s, d]), torch.cat([d, s])
    etype = torch.cat([r, r + num_rels]).to(torch.int32)
    deg = torch.zeros(n_nodes, dtype=torch.float32, device=dev).index_add_(
        0, dst2, torch.ones(dst2.shape[0], dtype=torch.float32, device=dev))
    norm = (1.0 / deg.clamp_(min=1.0))[dst2].view(-1, 1)
    return {"src": src2.to(torch.int32), "dst": dst2.to(torch.int32), "etype": etype, "norm": norm}


class NeighborEdgeBank:
    """Neighbourhood-expansion edge samples (kgvae/utils.py:33-76, ``--edge-sampler neighbor``) drawn on the GPU a
    bank at a time.  The picks of one sample are sequential, but samples are independent of each other and of the
    model, so one ``kg_neighbor_sample`` launch draws K samples (K = what one wave of the device holds, chosen by the
    library) into a persistent ``bank [K, B]`` and the training steps consume it one row at a time.

    ``next()`` returns ``bank[cursor]`` and advances the device ``cursor`` with stream-ordered device ops, so it can
    be captured in a CUDA graph.  The host keeps ``consumed``, the number of rows taken since the last refill, equal
    to the device cursor: outside a capture ``next()`` counts its row itself (refilling first when the bank is used
    up); a captured ``next()`` runs at every replay, and the caller calls ``before_replay()`` before each one, which
    counts the row and refills eagerly between replays once all K rows are consumed.

    ``refill()`` draws K x B x 8 uniform 32-bit words with torch's device generator and launches the kernel.  Same
    procedure as the host sampler up to the 2^-32 granularity of the integer mapping, not numpy's random stream."""

    def __init__(self, triplets, num_nodes, sample_size):
        if not triplets.is_cuda:
            raise RuntimeError("NeighborEdgeBank needs the triples on a CUDA device (no CPU fallback)")
        dev = triplets.device
        self.num_nodes, self.n_triples, self.B = int(num_nodes), int(triplets.shape[0]), int(sample_size)
        self.adj_ptr, self.adj = ops.neighbor_adjacency(triplets, self.num_nodes)
        self.K, ws = ops.neighbor_sample_plan(self.num_nodes, self.n_triples, self.B)
        self.workspace = torch.empty(max(ws, 16), dtype=torch.uint8, device=dev)
        self.words = torch.empty(self.K, self.B, ops.NEIGHBOR_WORDS, dtype=torch.int32, device=dev)
        self.bank = torch.empty(self.K, self.B, dtype=torch.int32, device=dev)
        self.cursor = torch.zeros(1, dtype=torch.int64, device=dev)
        self.consumed = self.K                   # empty: the first next() refills
        self.refills = 0

    def refill(self):
        self.words.random_(-2 ** 31, 2 ** 31)
        ops.neighbor_sample(self.adj_ptr, self.adj, self.num_nodes, self.B, self.words, out=self.bank,
                            workspace=self.workspace)
        self.cursor.zero_()
        self.consumed = 0
        self.refills += 1

    def next(self):
        """int32 [B]: the next row of the bank."""
        if not torch.cuda.is_current_stream_capturing():
            if self.consumed >= self.K:
                self.refill()
            self.consumed += 1
        # the remainder only guards the gather; before_replay() keeps the cursor below K
        row = self.bank.index_select(0, torch.remainder(self.cursor, self.K)).view(-1)
        self.cursor.add_(1)
        return row

    def before_replay(self):
        """Call before each replay of a graph that captured one ``next()``."""
        if self.consumed >= self.K:
            self.refill()
        self.consumed += 1


class SampledDeviceSampler:
    """``generate_sampled_graph_and_labels_device`` with ``sample_size`` < len(triplets) in FIXED shapes, so that the
    draw can be captured with the train step (``link_predict.CapturedTrainStep(..., sampler=...)``): every replay
    then draws a fresh uniform edge sample, relabels it, draws negatives and a graph split, and trains on it.

    Only the number of distinct entities among the B sampled triples varies from draw to draw.  The node set is
    therefore padded to a fixed budget ``n = cap = min(2 B, distinct entities of the training triples)``, which no
    draw can exceed: rows 0 .. n_valid-1 are the sampled nodes in ascending id order (as the eager device sampler
    orders them), row i >= n_valid looks up entity i and has no edges.  ``n_valid`` stays on the device (int32
    [1]); the model masks the padding out of every loss term through ``Graph.n_valid``.

    ``sample()`` returns FullBatchDeviceSampler's dict plus ``n_valid``: ``node_id [cap, 1]`` (int32), ``src`` /
    ``dst`` / ``etype [2 split B]`` (int32), ``norm [2 split B, 1]``, ``samples [B (1 + rate), 3]`` (int32),
    ``labels``.  The B distinct picks are the first B of a sort of T uniforms (a uniform random B-subset), the
    relabelling is kg_sample_relabel, negatives replace one end with floor(u n_valid).  Same procedure as the host
    sampler (kgvae/utils.py:79-124,158-171), not numpy's random stream.

    ``edge_sampler="neighbor"``: the B picks are the next row of a ``NeighborEdgeBank`` (the reference's
    neighbourhood-expansion sampler) instead; everything downstream is the same.  Call ``before_replay()`` before each
    replay of a captured ``sample()`` (``CapturedTrainStep.step`` does)."""

    def __init__(self, triplets, sample_size, split_size, num_rels, negative_rate, edge_sampler="uniform"):
        if not triplets.is_cuda:
            raise RuntimeError("SampledDeviceSampler needs the triples on a CUDA device (no CPU fallback)")
        self.triplets = triplets.to(torch.int32).contiguous()
        T = self.triplets.shape[0]
        self.B = int(sample_size)
        if not 0 < self.B <= T:
            raise ValueError(f"SampledDeviceSampler: sample_size must be in 1 .. {T}, got {sample_size}")
        ends = torch.cat([self.triplets[:, 0], self.triplets[:, 2]])
        # the only host read-backs, once: the entity-id range and the number of distinct entities
        self.num_nodes = int(ends.max()) + 1
        self.n = min(2 * self.B, int(torch.unique(ends).numel()))
        self.num_rels, self.rate = int(num_rels), int(negative_rate)
        self.keep_n = int(self.B * split_size)
        dev = self.triplets.device
        self.labels = torch.zeros(self.B * (self.rate + 1), dtype=torch.float32, device=dev)
        self.labels[:self.B] = 1
        self.n_edges, self.n_samples = 2 * self.keep_n, self.B * (self.rate + 1)
        if edge_sampler not in ("uniform", "neighbor"):
            raise ValueError("Sampler type must be either 'uniform' or 'neighbor'.")
        self.bank = NeighborEdgeBank(self.triplets, self.num_nodes, self.B) if edge_sampler == "neighbor" else None

    def before_replay(self):
        if self.bank is not None:
            self.bank.before_replay()

    def sample(self):
        dev = self.triplets.device
        if self.bank is not None:
            picked = self.bank.next()
        else:
            picked = torch.argsort(torch.rand(self.triplets.shape[0], device=dev))[:self.B]
        node_id, src, rel, dst, n_valid = ops.sample_relabel(self.triplets.index_select(0, picked), self.num_nodes,
                                                              self.n)
        pos = torch.stack([src, rel, dst], dim=1)
        m = self.B * self.rate
        # floor(u n_valid) with u in [0, 1) drawn in double: below n_valid for any n_valid < 2^24
        values = (torch.rand(m, dtype=torch.float64, device=dev) * n_valid.to(torch.float64)).to(torch.int32)
        samples = _with_negatives(pos, src.repeat(self.rate), rel.repeat(self.rate), dst.repeat(self.rate), values)
        graph = _split_graph(src, rel, dst, self.keep_n, self.num_rels, self.n)
        return {"node_id": node_id.view(-1, 1), **graph, "samples": samples, "labels": self.labels, "n_valid": n_valid}


# --------------------------------------------------------------------------------------------
# evaluation (kgvae/utils.py:180-221,293-314)
# --------------------------------------------------------------------------------------------
def sort_and_rank(score, target):
    """0-indexed rank of ``target`` in each row of ``score`` (descending).  Same result as the
    reference's sort + nonzero when scores are distinct; ties go to the lower entity id."""
    t = target.view(-1, 1)
    st = score.gather(1, t)
    col = torch.arange(score.shape[1], device=score.device).view(1, -1)
    return ((score > st).sum(1) + ((score == st) & (col < t)).sum(1)).view(-1)


def perturb_and_get_rank(embedding, w, a, r, b, test_size, batch_size=100, all_batches=True,
                         flow_log_prob=None, verbose=True, filt=None, cand_range=None):
    """Rank of ``b`` among all entities for the queries (a, r) (utils.py:187-221).

    The reference scores ``batch_size`` queries at a time through a D x E x V tensor; here all
    queries go through one fused score-and-count launch (``batch_size`` only bounds the work
    when ``all_batches`` is False, as in the reference's periodic validation)."""
    n = int(test_size) if all_batches else min(int(test_size), int(batch_size))
    dev = embedding.device
    a32, r32, b32 = (ops.as_i32(t[:n], dev) for t in (a, r, b))
    fp, fi = (None, None) if filt is None else filt
    ranks = ops.distmult_rank(embedding, w, a32, r32, b32, shift=flow_log_prob,
                              cand_range=cand_range, filt_ptr=fp, filt_idx=fi).long()
    if verbose:
        _print_rank_line(ranks)
    return ranks


def _print_rank_line(ranks):
    rr = ranks.float() + 1.0
    print("ranked {} queries: MR : {:.6f} |  MRR : {:.6f} | Hit1: {:.6f} | Hit5: {:.6f} | Hit10: {:.6f}".format(
        ranks.numel(), rr.mean().item(), (1.0 / rr).mean().item(), (rr <= 1).float().mean().item(),
        (rr <= 5).float().mean().item(), (rr <= 10).float().mean().item()))


def calc_mrr(embedding, w, test_triplets, hits=[], eval_bz=100, all_batches=True, flow_log_prob=None,
             verbose=True, return_ranks=False, filter_index=None, sharded=False, group=None):
    """Raw MRR / Hits@k over both perturbation directions (utils.py:293-314).  With ``filter_index`` (a
    ``FilterIndex``) the metrics are filtered instead (an extension; the reference is raw-only): every other
    entity that forms a known triple with a query is left out of its rank.

    ``sharded=True`` (multi-GPU; collective over ``group``): each rank counts the candidates of its own entity
    shard (``parallel.entity_shard``) and the counts are summed with ``parallel.sharded_rank_counts``, so every
    rank returns the same ranks and MRR as one GPU would.  Every rank must pass the same ``embedding``, ``w``,
    ``flow_log_prob`` and ``test_triplets``; only rank 0 prints."""
    with torch.no_grad():
        s, r, o = test_triplets[:, 0], test_triplets[:, 1], test_triplets[:, 2]
        n = test_triplets.shape[0]
        filt_s = filt_o = None
        if filter_index is not None:
            m = n if all_batches else min(int(n), int(eval_bz))       # the queries perturb_and_get_rank ranks
            filt_s = filter_index.lists(o[:m], r[:m], "subject")      # (c, r, o) known
            filt_o = filter_index.lists(s[:m], r[:m], "object")       # (s, r, c) known
        if sharded:
            verbose = verbose and dist.get_rank(group) == 0
            V = embedding.shape[0]

            def direction(a, b, filt):
                count = lambda lo, hi: perturb_and_get_rank(embedding, w, a, r, b, n, eval_bz, all_batches,
                                                            flow_log_prob, False, filt=filt, cand_range=(lo, hi))
                ranks = parallel.sharded_rank_counts(count, V, group)
                if verbose:
                    _print_rank_line(ranks)
                return ranks
            ranks_s, ranks_o = direction(o, s, filt_s), direction(s, o, filt_o)
        else:
            ranks_s = perturb_and_get_rank(embedding, w, o, r, s, n, eval_bz, all_batches, flow_log_prob, verbose,
                                           filt=filt_s)
            ranks_o = perturb_and_get_rank(embedding, w, s, r, o, n, eval_bz, all_batches, flow_log_prob, verbose,
                                           filt=filt_o)
        ranks = torch.cat([ranks_s, ranks_o]) + 1
        mrr = torch.mean(1.0 / ranks.float())
        if verbose:
            kind = "raw" if filter_index is None else "filtered"
            print("MRR ({}): {:.6f}".format(kind, mrr.item()))
            for hit in hits:
                print("Hits ({}) @ {}: {:.6f}".format(kind, hit, torch.mean((ranks <= hit).float()).item()))
    return (mrr.item(), ranks) if return_ranks else mrr.item()


def generate(embedding, w, test_triplets, eval_bz=200, topk=1, flow_log_prob=None, entity_names=None,
             relation_names=None, out_path=None, max_lines=None, filter_index=None, sharded=False, group=None):
    """Tail generation (kgvae/utils.py:245-288): for every test triple (a, r, b) the highest-scored tail(s) among
    all entities.  The reference scores 200 queries at a time through the D x E x V tensor, takes
    ``score.argmax`` and prints the triples around one hard-coded entity using name files from the author's home
    directory; here all queries go through one tcgen05 score pass with a top-k epilogue (``eval_bz`` is accepted
    and ignored), and the triples are written as ids - or names, when ``entity_names`` / ``relation_names``
    (sequences or dicts indexed by id) are given - to ``out_path`` (default: nothing is written).

    ``filter_index`` (a ``FilterIndex``; an extension): only tails c for which (a, r, c) is not a known triple are
    returned - generation proposes new facts.  A query with fewer than ``topk`` such tails gets trailing -1.

    ``sharded=True`` (multi-GPU; collective over ``group``): each rank generates from its own entity shard
    (``parallel.entity_shard``) and the shards' lists are merged with ``parallel.merge_topk``, which is exact, so
    every rank returns what one GPU would.  Every rank must pass the same ``embedding``, ``w``, ``flow_log_prob``
    and ``test_triplets``; only rank 0 writes ``out_path``.

    Returns (tails int64 [T, topk], scores fp32 [T, topk]) on the embedding's device; ``tails[:, 0]`` is the
    reference's ``highest_scored``."""
    with torch.no_grad():
        dev = embedding.device
        t = torch.as_tensor(test_triplets)
        a, r = ops.as_i32(t[:, 0], dev), ops.as_i32(t[:, 1], dev)
        fp, fi = (None, None) if filter_index is None else filter_index.lists(a, r, "object")
        if sharded:
            rank = dist.get_rank(group)
            lo, hi = parallel.entity_shard(embedding.shape[0], rank, dist.get_world_size(group))
            idx, score = ops.distmult_topk(embedding, w, a, r, k=topk, shift=flow_log_prob, filt_ptr=fp,
                                           filt_idx=fi, cand_range=(lo, hi))
            idx, score = parallel.merge_topk(idx, score, topk, group)
            if rank != 0:
                out_path = None
        else:
            idx, score = ops.distmult_topk(embedding, w, a, r, k=topk, shift=flow_log_prob, filt_ptr=fp,
                                           filt_idx=fi)
        tails = idx.long()
    if out_path is not None:
        ent = (lambda i: str(entity_names[i])) if entity_names is not None else (lambda i: f"e{i}")
        rel = (lambda i: str(relation_names[i])) if relation_names is not None else (lambda i: f"r{i}")
        a_h, r_h, b_h, c_h = (x.cpu().tolist() for x in (t[:, 0], t[:, 1], t[:, 2], tails))
        with open(out_path, "w") as f:
            for i in range(len(a_h) if max_lines is None else min(len(a_h), max_lines)):
                f.write(" - ".join([ent(a_h[i]), rel(r_h[i]), ent(b_h[i])]) + "\n")      # the known triple
                for c in c_h[i]:
                    if c != b_h[i] and c >= 0:
                        f.write(" = ".join([ent(a_h[i]), rel(r_h[i]), ent(c)]) + "\n")   # a generated one
    return tails, score


def build_filter(all_triplets, queries_a, queries_r, num_rels, direction, device):
    """CSR of known-true candidates per query for filtered ranking (extension; the reference is
    raw-only).  direction "object": candidates c with (a, r, c) known; "subject": (c, r, a).
    Host reference of ``FilterIndex.lists``, which builds the same CSR on the GPU."""
    t = np.asarray(all_triplets)
    key_col, val_col = (0, 2) if direction == "object" else (2, 0)
    keys = t[:, key_col].astype(np.int64) * num_rels + t[:, 1]
    order = np.argsort(keys, kind="stable")
    keys_sorted, vals_sorted = keys[order], t[order, val_col]
    q = np.asarray(queries_a).astype(np.int64) * num_rels + np.asarray(queries_r)
    lo = np.searchsorted(keys_sorted, q, side="left")
    hi = np.searchsorted(keys_sorted, q, side="right")
    # the kernel subtracts one count per listed candidate, so each list must be duplicate-free
    lists = [np.unique(vals_sorted[l:h]) for l, h in zip(lo, hi)]
    ptr = np.concatenate(([0], np.cumsum([len(x) for x in lists]))).astype(np.int32)
    idx = (np.concatenate(lists) if lists else np.zeros(0)).astype(np.int32)
    return torch.from_numpy(ptr).to(device), torch.from_numpy(idx).to(device)


class FilterIndex:
    """The known triples of a graph (train + valid + test, usually) indexed once per direction on the GPU, for
    filtered ranks (``calc_mrr(..., filter_index=...)``) and filtered generation (``generate(..., filter_index=...)``).
    An extension: the reference reports raw ranks only (kgvae/link_predict.py:7).

    ``lists(a, r, direction)`` returns the CSR ``(ptr int32 [M+1], idx int32 [nnz])`` of every entity c with
    (a_i, r_i, c) known (``direction="object"``) or (c, r_i, a_i) known ("subject"), ascending and duplicate-free:
    exactly what ``build_filter`` computes on the host, built by the kg_filter_* kernels with one host read-back
    (the list total).  Ids must lie in [0, num_nodes) / [0, num_rels)."""

    def __init__(self, known_triplets, num_nodes, num_rels, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("FilterIndex needs a CUDA device (no CPU fallback)")
        tri = ops.as_i32(known_triplets, device)
        self.num_nodes, self.num_rels = int(num_nodes), int(num_rels)
        self.tables = {d: ops.filter_table(tri, self.num_nodes, self.num_rels, d) for d in ops.FILTER_DIRECTIONS}

    def lists(self, a, r, direction):
        table, n = self.tables[direction]
        dev = table.device
        return ops.filter_lists(table, n, self.num_nodes, self.num_rels, ops.as_i32(a, dev), ops.as_i32(r, dev))


# --------------------------------------------------------------------------------------------
# probability helpers (kgvae/utils.py:323-428)
# --------------------------------------------------------------------------------------------
def gaussian_parameters(h, dim=-1):
    m, raw = torch.split(h, h.size(dim) // 2, dim=dim)
    return m, F.softplus(raw) + 1e-8


def sample_gaussian(m, v, repeat=1):
    if repeat > 1:
        sd = torch.cat([torch.sqrt(v.squeeze())] * repeat, dim=0)
        m = torch.cat([m.squeeze()] * repeat, dim=0)
    else:
        sd = torch.sqrt(v)
    return m + torch.randn_like(sd) * sd


def log_normal(x, m, v):
    lp = -(x - m).pow(2) / (2 * v) - v.sqrt().log() - np.log(np.sqrt(2 * np.pi))
    return lp.sum(-1)


def log_sum_exp(x, dim=0):
    mx = torch.max(x, dim)[0]
    return mx + (x - mx.unsqueeze(dim).expand_as(x)).exp().sum(dim).log()


def log_mean_exp(x, dim):
    return log_sum_exp(x, dim) - np.log(x.size(dim))


def log_normal_mixture(z, m, v):
    return log_mean_exp(log_normal(z.unsqueeze(1), m, v), dim=-1)


class DevicePrefetcher:
    """Double-buffered host -> device staging of step inputs (the ``.cuda()`` copies of
    kgvae/link_predict.py:217-220) on a side stream: ``submit`` starts the copies of a dict of
    pinned host tensors into one of ``depth`` persistent device buffer sets, ``take`` hands that
    set to the current stream once the copies have landed.  Call order per step: ``take()`` (set i),
    ``submit()`` (set i + 1), then run step i - the copy of step i + 1 overlaps step i's kernels.  Any
    other order is still safe (a set is only overwritten after everything the consumer stream had enqueued
    at ``submit`` time), it merely overlaps less."""

    def __init__(self, device, depth=2):
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(self.device)
        self._slots = [None] * depth
        self._used = [False] * depth       # the set has been handed to the consumer stream at least once
        self._count = 0
        self._pending = []

    def submit(self, host_tensors):
        slot = self._count % len(self._slots)
        self._count += 1
        cur = torch.cuda.current_stream(self.device)
        if self._used[slot]:
            # the set being overwritten was handed out before: everything the consumer stream has enqueued up
            # to NOW may still read it (whatever order take / submit / run were called in), so the copies wait
            # for that point.  In the intended order - take(i), submit(i + 1), run step i - this is the end of
            # step i - 1, the set's last reader; step i is not enqueued yet and overlaps the copy.
            ev = torch.cuda.Event()
            ev.record(cur)
            self.stream.wait_event(ev)
        with torch.cuda.stream(self.stream):
            bufs = self._slots[slot]
            if bufs is None or any(k not in bufs or bufs[k].shape != v.shape or bufs[k].dtype != v.dtype
                                   for k, v in host_tensors.items()):
                bufs = {k: torch.empty(v.shape, dtype=v.dtype, device=self.device) for k, v in host_tensors.items()}
                self._slots[slot] = bufs
            for k, v in host_tensors.items():
                bufs[k].copy_(v, non_blocking=True)
            done = torch.cuda.Event()
            done.record(self.stream)
        self._pending.append((slot, done))

    def take(self):
        slot, done = self._pending.pop(0)
        cur = torch.cuda.current_stream(self.device)
        self._used[slot] = True
        cur.wait_event(done)
        out = {k: self._slots[slot][k] for k in self._slots[slot]}
        for t in out.values():             # allocated on the side stream, read on this one
            t.record_stream(cur)
        return out
