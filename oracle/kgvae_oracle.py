"""CPU oracle: a functional restatement of the reference's link-prediction path.

TEST INFRASTRUCTURE ONLY.  Nothing on the product path (``gcn-vae_b200/``) may
import this module; only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` do, as the checker
or as the timed CPU baseline.

Parity status: PINNED against the reference itself.  ``tests/golden/make_golden.py``
imports ``/root/reference/kgvae/{model,utils,link_predict,flow_network}.py``
*verbatim* (over ``oracle/dgl_shim``, a restatement of the DGL 0.4.x calls they
make - DGL is an un-vendored, un-pinned dependency) and stores their outputs on
seeded inputs under ``tests/golden/``; ``tests/test_oracle_golden.py`` checks
every function below against those vectors.  The reference ships no tests or
known-answer vectors of its own (SURVEY.md section 4), so those generated
vectors are the pin.  Deviations allowed (SURVEY.md section 8c): a ``None``
``flow_log_prob`` is treated as ``0.0``; ranks are reported with an explicit
stable tie policy (the reference's is implementation-defined).

Every function cites the reference lines it follows.  The op sequence is kept
the same as the reference's (per-edge weight materialisation, tiny ``bmm``s,
``index_add``, the ``D x E x V`` evaluation tensor) because this module is
also what ``bench.py`` times as the CPU baseline.

Parameters travel in a flat dict keyed by the reference's state-dict names:
``encoder.input_layer.embedding.weight``, ``encoder.rconv_layer_{1,2}.{weight,
h_bias,loop_weight}``, ``encoder.z_pre``, ``encoder.nf.{0,2,4}.net.{0,2,4,6,8}.
{weight,bias}``, ``w_relation``.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

LOG_SQRT_2PI = float(np.log(np.sqrt(2 * np.pi)))


# ---------------------------------------------------------------------------
# a1  graph construction            reference kgvae/utils.py:127-155,
#                                   kgvae/link_predict.py:95-100
# ---------------------------------------------------------------------------
def build_graph_from_triplets(num_nodes, num_rels, src, rel, dst):
    """Add reverse edges (``rel + num_rels``), order edges by ascending
    (dst, src, rel), ``norm_v = 1/in_deg(v)`` (0 for isolated nodes),
    ``edge_norm_e = norm[dst_e]``.  Integer outputs are int64 numpy arrays.
    """
    src, rel, dst = (np.asarray(a, dtype=np.int64) for a in (src, rel, dst))
    s2 = np.concatenate((src, dst))
    d2 = np.concatenate((dst, src))
    r2 = np.concatenate((rel, rel + num_rels))
    order = np.lexsort((r2, s2, d2))          # == sorted(zip(dst, src, rel))
    s2, d2, r2 = s2[order], d2[order], r2[order]
    in_deg = np.bincount(d2, minlength=num_nodes).astype(np.float32)
    with np.errstate(divide="ignore"):
        norm = (1.0 / in_deg).astype(np.float32)
    norm[np.isinf(norm)] = 0
    return {"num_nodes": int(num_nodes), "src": s2, "dst": d2, "etype": r2,
            "norm": norm, "edge_norm": norm[d2].reshape(-1, 1)}


# ---------------------------------------------------------------------------
# a11 sampling (host)               reference kgvae/utils.py:79-124,158-171
# ---------------------------------------------------------------------------
def negative_sampling(pos_samples, num_entity, negative_rate, rng=np.random):
    """Corrupt subject where u > 0.5 else object; legacy global RNG call order
    ``randint`` then ``uniform`` (kgvae/utils.py:164-165)."""
    n = len(pos_samples)
    total = n * negative_rate
    neg = np.tile(pos_samples, (negative_rate, 1))
    labels = np.zeros(n * (negative_rate + 1), dtype=np.float32)
    labels[:n] = 1
    values = rng.randint(num_entity, size=total)
    u = rng.uniform(size=total)
    neg[u > 0.5, 0] = values[u > 0.5]
    neg[u <= 0.5, 2] = values[u <= 0.5]
    return np.concatenate((pos_samples, neg)), labels


def generate_sampled_graph_and_labels(triplets, sample_size, split_size, num_rels,
                                      negative_rate, rng=np.random):
    """Uniform edge sampler path of kgvae/utils.py:85-124.  RNG call order:
    choice(T, B) -> randint -> uniform -> choice(B, B*split)."""
    picked = rng.choice(np.arange(len(triplets)), sample_size, replace=False)
    src, rel, dst = triplets[picked].transpose()
    uniq_v, inv = np.unique((src, dst), return_inverse=True)
    src, dst = np.reshape(inv, (2, -1))
    relabeled = np.stack((src, rel, dst)).transpose()
    samples, labels = negative_sampling(relabeled, len(uniq_v), negative_rate, rng)
    keep = rng.choice(np.arange(sample_size), size=int(sample_size * split_size),
                      replace=False)
    graph = build_graph_from_triplets(len(uniq_v), num_rels, src[keep], rel[keep], dst[keep])
    return graph, uniq_v, samples, labels


# ---------------------------------------------------------------------------
# a3 / a4  RelGraphConv             DGL 0.4.x relgraphconv.py (SURVEY 3.3);
#                                   constructed at reference kgvae/model.py:54-59
# ---------------------------------------------------------------------------
def rgcn_bdd_layer(x, graph, weight, h_bias, loop_weight, num_bases, activation=None,
                   drop_mask=None):
    src = torch.as_tensor(graph["src"])
    dst = torch.as_tensor(graph["dst"])
    etype = torch.as_tensor(graph["etype"])
    norm = torch.as_tensor(graph["edge_norm"])
    in_feat, out_feat = loop_weight.shape
    si, so = in_feat // num_bases, out_feat // num_bases
    w = weight.index_select(0, etype).view(-1, si, so)          # [E*B, si, so]
    msg = torch.bmm(x[src].reshape(-1, 1, si), w).view(-1, out_feat)
    msg = msg * norm
    h = torch.zeros(graph["num_nodes"], out_feat, dtype=x.dtype).index_add(0, dst, msg)
    h = h + h_bias
    h = h + torch.matmul(x, loop_weight)
    if activation is not None:
        h = activation(h)
    if drop_mask is not None:
        h = h * drop_mask
    return h


def rgcn_basis_layer(x, graph, weight, w_comp, h_bias, loop_weight, activation=None,
                     drop_mask=None):
    """basis regulariser (reference kgvae/entity_classify.py:30-43); ``x`` may
    be 1-D int64 node ids (embedding-style lookup) or dense features."""
    src = torch.as_tensor(graph["src"])
    dst = torch.as_tensor(graph["dst"])
    etype = torch.as_tensor(graph["etype"])
    nb, in_feat, out_feat = weight.shape
    if w_comp is not None:
        w = torch.matmul(w_comp, weight.view(nb, -1)).view(-1, in_feat, out_feat)
    else:
        w = weight
    h_src = x[src]
    if h_src.dtype == torch.int64 and h_src.dim() == 1:
        msg = w.view(-1, out_feat).index_select(0, etype * in_feat + h_src)
    else:
        msg = torch.bmm(h_src.unsqueeze(1), w.index_select(0, etype)).squeeze(1)
    if graph.get("edge_norm") is not None:
        msg = msg * torch.as_tensor(graph["edge_norm"])
    h = torch.zeros(graph["num_nodes"], out_feat, dtype=msg.dtype).index_add(0, dst, msg)
    if h_bias is not None:
        h = h + h_bias
    if loop_weight is not None:
        if x.dtype == torch.int64 and x.dim() == 1:
            h = h + loop_weight.index_select(0, x)
        else:
            h = h + torch.matmul(x, loop_weight)
    if activation is not None:
        h = activation(h)
    if drop_mask is not None:
        h = h * drop_mask
    return h


# ---------------------------------------------------------------------------
# a5 / a7  probability utilities    reference kgvae/utils.py:323-428
# ---------------------------------------------------------------------------
def gaussian_parameters(h, dim=-1):
    m, raw = torch.split(h, h.size(dim) // 2, dim=dim)       # utils.py:337
    return m, F.softplus(raw) + 1e-8                         # utils.py:338


def sample_gaussian(m, v, eps):
    return m + eps * torch.sqrt(v)                           # utils.py:359-360


def log_normal(x, m, v):
    lp = -(x - m).pow(2) / (2 * v) - v.sqrt().log() - LOG_SQRT_2PI   # utils.py:396
    return lp.sum(-1)


def log_mean_exp(x, dim):
    mx = torch.max(x, dim)[0]                                # utils.py:413-415
    lse = mx + (x - mx.unsqueeze(dim)).exp().sum(dim).log()
    return lse - math.log(x.size(dim))                       # utils.py:428


def log_normal_mixture(z, m, v):
    return log_mean_exp(log_normal(z.unsqueeze(1), m, v), dim=-1)    # utils.py:376-377


# ---------------------------------------------------------------------------
# a6  IAF flow (MADE + permute)     reference kgvae/flow_network.py:37-98
# ---------------------------------------------------------------------------
def made_degrees(input_size, hidden_size, n_hidden):
    """Degree vectors; they double as the per-pass column index lists
    (flow_network.py:70-77; ``-1`` wraps to the last column)."""
    d_in = torch.arange(input_size)
    degs = [d_in]
    for _ in range(n_hidden + 1):
        degs.append(torch.arange(hidden_size) % (input_size - 1))
    degs.append(d_in % input_size - 1)
    return degs


def made_masks(input_size, hidden_size, n_hidden):
    degs = made_degrees(input_size, hidden_size, n_hidden)
    masks = [(d1.unsqueeze(-1) >= d0.unsqueeze(0)).float()
             for d0, d1 in zip(degs[:-1], degs[1:])]          # flow_network.py:80-81
    masks[-1] = masks[-1].repeat(2, 1)                        # flow_network.py:61-62
    return masks


def made_net(x, weights, biases, masks, relu_patterns=None):
    """``relu_patterns`` (optional): one bool mask per hidden layer ([N, hidden] or a [1, hidden] row that
    broadcasts) naming the units that count as active, in place of ``pre-activation > 0`` - see kgvae_encode."""
    n = len(weights)
    for i in range(n):
        x = F.linear(x, masks[i] * weights[i], biases[i])     # flow_network.py:15
        if i + 1 < n:
            x = torch.relu(x) if relu_patterns is None else torch.where(relu_patterns[i], x, torch.zeros_like(x))
    return x


def made_forward(z, weights, biases, masks, degrees, relu_patterns=None):
    """``len(degrees)`` full passes; pass p overwrites columns ``degrees[p]`` with
    ``z * exp(alpha + mu)``; log-det is the row-sum of the last pass's alpha
    (flow_network.py:91-96).  ``relu_patterns`` (optional): per pass, the list made_net takes."""
    x = torch.zeros_like(z)
    alpha = None
    for p, idx in enumerate(degrees):
        pattern = None if relu_patterns is None else relu_patterns[p]
        mu, alpha = torch.chunk(made_net(x, weights, biases, masks, pattern), 2, dim=1)
        x = x.clone()
        x[:, idx] = z[:, idx] * torch.exp(alpha[:, idx] + mu[:, idx])
    return x, alpha.sum(-1)


def made_inverse(x, weights, biases, masks):
    mu, alpha = made_net(x, weights, biases, masks).chunk(2, dim=-1)  # flow_network.py:108-111
    return (x - mu) * torch.exp(-alpha), (-alpha).sum(-1)


def flow_params(params, n_flows):
    """Per-MADE (weights, biases) lists from reference state-dict names."""
    out = []
    for f in range(n_flows):
        ws = [params[f"encoder.nf.{2 * f}.net.{2 * l}.weight"] for l in range(n_flows + 2)]
        bs = [params[f"encoder.nf.{2 * f}.net.{2 * l}.bias"] for l in range(n_flows + 2)]
        out.append((ws, bs))
    return out


def iaf_forward(z, params, n_flows, made_relu_patterns=None):
    """MADE, reverse columns, MADE, ...; scalar ``flow_log_prob`` is the mean over
    nodes of the summed log-dets (reference kgvae/model.py:115-123).
    ``made_relu_patterns`` (optional): per MADE, the per-pass lists made_forward takes."""
    h = z.shape[1]
    masks = made_masks(h, h, n_flows)
    degs = made_degrees(h, h, n_flows)
    log_det_sum = torch.zeros(z.shape[0], dtype=z.dtype)
    for f, (ws, bs) in enumerate(flow_params(params, n_flows)):
        pattern = None if made_relu_patterns is None else made_relu_patterns[f]
        z, log_det = made_forward(z, ws, bs, masks, degs, pattern)
        log_det_sum = log_det_sum + log_det
        z = z.flip(1)                                          # flow_network.py:28-30
    return z, log_det_sum, log_det_sum.view(-1, 1).mean()


# ---------------------------------------------------------------------------
# a2 + a3 + a5 + a6  encoder        reference kgvae/model.py:107-124
# ---------------------------------------------------------------------------
def kgvae_encode(params, graph, node_id, eps, num_bases, n_flows=0, drop_masks=(None, None), relu_pattern=None,
                 made_relu_patterns=None):
    """``relu_pattern`` (bool [N, h], optional): which units of layer 1 count as active.  ReLU has no derivative
    at 0, and a pre-activation within rounding error of 0 can land on either side depending on the summation
    order; a gradient comparison at millions of units (the benchmark-size parity test) hands the other
    implementation's pattern in here so that both sides differentiate the same piecewise-linear function.
    The forward value changes by at most the magnitude of those pre-activations (~1e-6).
    ``made_relu_patterns`` (optional): the same for the hidden layers of the IAF flow - per MADE, per pass, per
    hidden layer a bool mask ([N, h], or [1, h] for a pass whose rows are all equal, such as the first)."""
    p = params
    h0 = p["encoder.input_layer.embedding.weight"][torch.as_tensor(node_id).view(-1)]
    act1 = torch.relu if relu_pattern is None else (lambda t: t * relu_pattern.to(t.dtype))
    h1 = rgcn_bdd_layer(h0, graph, p["encoder.rconv_layer_1.weight"],
                        p["encoder.rconv_layer_1.h_bias"],
                        p["encoder.rconv_layer_1.loop_weight"], num_bases,
                        act1, drop_masks[0])
    h2 = rgcn_bdd_layer(h1, graph, p["encoder.rconv_layer_2.weight"],
                        p["encoder.rconv_layer_2.h_bias"],
                        p["encoder.rconv_layer_2.loop_weight"], num_bases,
                        None, drop_masks[1])
    z_mean, z_sigma = gaussian_parameters(h2)
    z0 = sample_gaussian(z_mean, z_sigma, eps)
    out = {"h0": h0, "h1": h1, "h2": h2, "z_mean": z_mean, "z_sigma": z_sigma, "z0": z0}
    if n_flows > 0:
        z, lds, flp = iaf_forward(z0, params, n_flows, made_relu_patterns)
        out.update(z=z, log_det_sum=lds, flow_log_prob=flp)
    else:
        out.update(z=z0, log_det_sum=None, flow_log_prob=None)
    return out


# ---------------------------------------------------------------------------
# a9  DistMult + loss               reference kgvae/link_predict.py:57-92,
#                                   kgvae/model.py:82-87
# ---------------------------------------------------------------------------
def distmult_score(z, w_relation, triplets):
    t = torch.as_tensor(triplets)
    return torch.sum(z[t[:, 0]] * w_relation[t[:, 1]] * z[t[:, 2]], dim=1)


def kl_term(z, z_mean, z_sigma, z_pre, flow_log_prob):
    m_mix, v_mix = gaussian_parameters(z_pre, dim=1)
    flp = 0.0 if flow_log_prob is None else flow_log_prob      # documented deviation
    return torch.mean(log_normal(z, z_mean, z_sigma) + flp
                      - log_normal_mixture(z, m_mix, v_mix))


def kgvae_loss(params, enc, triplets, labels, reg_param, kl_param, n_flows):
    z, w = enc["z"], params["w_relation"]
    score = distmult_score(z, w, triplets)
    if n_flows > 0:
        score = score + enc["flow_log_prob"]
    pred = F.binary_cross_entropy_with_logits(score, torch.as_tensor(labels))
    reg = torch.mean(z.pow(2)) + torch.mean(w.pow(2))
    if kl_param > 0:
        kl = kl_term(z, enc["z_mean"], enc["z_sigma"], params["encoder.z_pre"],
                     enc["flow_log_prob"])
    else:
        kl = torch.zeros(1)
    loss = pred + reg_param * reg + kl_param * kl
    return {"loss": loss, "predict_loss": pred, "reg": reg, "kl": kl, "score": score}


# ---------------------------------------------------------------------------
# a10 raw-rank evaluation           reference kgvae/utils.py:180-221,293-314
# ---------------------------------------------------------------------------
def eval_scores(emb, w, a, r, flow_log_prob=None):
    """``D x E x 1`` by ``D x 1 x V`` bmm then sum over D (utils.py:200-205)."""
    emb_ar = (emb[a] * w[r]).transpose(0, 1).unsqueeze(2)
    emb_c = emb.transpose(0, 1).unsqueeze(1)
    score = torch.sum(torch.bmm(emb_ar, emb_c), dim=0)
    return score + (0.0 if flow_log_prob is None else flow_log_prob)


def rank_of_target(score, target, policy="stable"):
    """0-indexed rank of ``target`` in a descending ordering of each score row.

    ``policy="reference"``: the reference's ``torch.sort`` + ``nonzero``
    (utils.py:180-184; tie order implementation-defined).
    ``policy="stable"``: ties broken by ascending entity id, computed as
    ``#(s > s_t) + #(s == s_t and j < t)`` - the rule the CUDA path follows.
    """
    target = torch.as_tensor(target).view(-1, 1)
    if policy == "reference":
        _, idx = torch.sort(score, dim=1, descending=True)
        return torch.nonzero(idx == target)[:, 1].view(-1)
    st = score.gather(1, target)
    col = torch.arange(score.shape[1]).view(1, -1)
    return ((score > st).sum(1) + ((score == st) & (col < target)).sum(1)).view(-1)


def rank_interval(score, target):
    """[lo, hi]: every tie order puts the target's 0-indexed rank in this range."""
    target = torch.as_tensor(target).view(-1, 1)
    st = score.gather(1, target)
    return (score > st).sum(1), (score >= st).sum(1) - 1


def perturb_and_get_rank(emb, w, a, r, b, batch_size=100, all_batches=True,
                         flow_log_prob=None, policy="stable", apply_sigmoid=True):
    n = len(a)
    n_batch = (n + batch_size - 1) // batch_size if all_batches else 1
    ranks = []
    for i in range(n_batch):
        lo, hi = i * batch_size, min(n, (i + 1) * batch_size)
        score = eval_scores(emb, w, a[lo:hi], r[lo:hi], flow_log_prob)
        if apply_sigmoid:
            score = torch.sigmoid(score)                       # utils.py:208
        ranks.append(rank_of_target(score, b[lo:hi], policy))
    return torch.cat(ranks)


def calc_mrr(emb, w, test_triplets, hits=(), eval_bz=100, all_batches=True,
             flow_log_prob=None, policy="stable", apply_sigmoid=True):
    """Returns (mrr, {hit: frac}, ranks[2T] 1-indexed); subject pass first with
    (a, r, b) = (o, r, s) (utils.py:301-306)."""
    with torch.no_grad():
        t = torch.as_tensor(test_triplets)
        s, r, o = t[:, 0], t[:, 1], t[:, 2]
        rs = perturb_and_get_rank(emb, w, o, r, s, eval_bz, all_batches, flow_log_prob,
                                  policy, apply_sigmoid)
        ro = perturb_and_get_rank(emb, w, s, r, o, eval_bz, all_batches, flow_log_prob,
                                  policy, apply_sigmoid)
        ranks = torch.cat([rs, ro]) + 1
        mrr = torch.mean(1.0 / ranks.float()).item()
        return mrr, {h: torch.mean((ranks <= h).float()).item() for h in hits}, ranks


def topk_tails(emb, w, a, r, k=1, flow_log_prob=None):
    """utils.generate (reference kgvae/utils.py:245-288) generalised from argmax to top-k: the k highest-scored
    entities per query, best first, ties by ascending entity id (the reference's ``argmax`` leaves ties to the
    backend).  Returns (idx int64 [E, k], score [E, k])."""
    score = eval_scores(emb, w, a, r, flow_log_prob)
    order = torch.sort(-score, dim=1, stable=True)[1][:, :k]         # stable: lower id first among equals
    return order, score.gather(1, order)


def filtered_ranks(score, target, known_lists):
    """Oracle *extension* (the reference reports raw ranks only, link_predict.py:7):
    known-true candidates other than the target are removed before ranking."""
    out = []
    for i in range(score.shape[0]):
        row = score[i].clone()
        t = int(target[i])
        st = row[t].item()
        keep = torch.ones_like(row, dtype=torch.bool)
        known = [k for k in known_lists[i] if k != t]
        if known:
            keep[torch.as_tensor(known)] = False
        col = torch.arange(row.numel())
        ahead = ((row > st) | ((row == st) & (col < t))) & keep
        out.append(int(ahead.sum()))
    return torch.as_tensor(out)


# ---------------------------------------------------------------------------
# parameter construction (same shapes / initialisers as the reference modules)
# ---------------------------------------------------------------------------
def init_params(num_nodes, h_dim, num_rels, num_bases, k=10, n_flows=0, seed=0):
    """Random-init parameter dict with the reference's state-dict names, shapes and
    initialiser families (kgvae/model.py:35,185-191; link_predict.py:50-55;
    DGL RelGraphConv xavier-uniform/relu gain; nn.Linear defaults for MADE)."""
    g = torch.Generator().manual_seed(seed)
    gain = math.sqrt(2.0)

    def xavier(*shape):
        t = torch.empty(*shape)
        fan_in, fan_out = torch.nn.init._calculate_fan_in_and_fan_out(t)
        bound = gain * math.sqrt(6.0 / (fan_in + fan_out))
        return (torch.rand(*shape, generator=g) * 2 - 1) * bound

    R2 = 2 * num_rels
    si = h_dim // num_bases
    p = {
        "encoder.input_layer.embedding.weight": torch.randn(num_nodes, h_dim, generator=g),
        "encoder.rconv_layer_1.weight": xavier(R2, num_bases * si * si),
        "encoder.rconv_layer_1.h_bias": torch.zeros(h_dim),
        "encoder.rconv_layer_1.loop_weight": xavier(h_dim, h_dim),
        "encoder.rconv_layer_2.weight": xavier(R2, num_bases * si * 2 * si),
        "encoder.rconv_layer_2.h_bias": torch.zeros(2 * h_dim),
        "encoder.rconv_layer_2.loop_weight": xavier(h_dim, 2 * h_dim),
        "encoder.z_pre": torch.randn(1, 2 * k, h_dim, generator=g) / math.sqrt(k * h_dim),
        "w_relation": xavier(num_rels, h_dim),
    }
    for f in range(n_flows):
        sizes = [(h_dim, h_dim)] * (n_flows + 1) + [(2 * h_dim, h_dim)]
        for l, (o, i) in enumerate(sizes):
            bound = 1.0 / math.sqrt(i)
            p[f"encoder.nf.{2 * f}.net.{2 * l}.weight"] = (torch.rand(o, i, generator=g) * 2 - 1) * bound
            p[f"encoder.nf.{2 * f}.net.{2 * l}.bias"] = (torch.rand(o, generator=g) * 2 - 1) * bound
    return p
