#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference.

Runs only in the build container: it imports ``/root/reference/kgvae/*.py``
verbatim (sys.path) over ``oracle/dgl_shim`` (DGL is not installable here) and
records inputs + every intermediate + gradients + ranks on seeded inputs.  The
resulting ``.npz`` files are committed; the GPU box never sees /root/reference.

    python tests/golden/make_golden.py

Injection points (no reference source is patched):
  * eps of ``sample_gaussian``  -> ``torch.randn_like`` is swapped for the call
  * dropout masks               -> ``RelGraphConv.dropout_mask`` hook of the shim
  * ``flow_log_prob=None``      -> attribute set to 0.0 before ``get_loss`` /
                                   passed as 0.0 to ``calc_mrr`` (SURVEY F5)

kgvae_small_noflow.npz does not store its random inputs (see ``shrink``): the tests draw
them again from torch's CPU random stream (tests/helpers.py:redraw_inputs) and check
them against the SHA-256 recorded here.  A torch release that changes how ``normal_``,
``rand``, ``randn`` or ``xavier_uniform_`` draw makes that case fail with a message
saying so; it is then restored only by running this script against the reference again.
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference/kgvae"
sys.path.insert(0, os.path.join(ROOT, "oracle", "dgl_shim"))
sys.path.insert(0, REF)
sys.path.append(os.path.dirname(HERE))

with contextlib.redirect_stdout(io.StringIO()):
    import link_predict as ref_lp          # noqa: E402  (reference, verbatim)
    import model as ref_model              # noqa: E402
    import utils as ref_utils              # noqa: E402
    import flow_network as ref_flow        # noqa: E402
torch.autograd.set_detect_anomaly(False)


def synthetic_triples(rng, n_ent, n_rel, n):
    s = rng.integers(0, n_ent, size=n)
    o = rng.integers(0, n_ent, size=n)
    r = rng.integers(0, n_rel, size=n)
    return np.stack([s, r, o], axis=1).astype(np.int64)


@contextlib.contextmanager
def preset_randn(eps):
    orig = torch.randn_like
    torch.randn_like = lambda t, *a, **k: eps.clone()
    try:
        yield
    finally:
        torch.randn_like = orig


SAMPLED = ["h1", "h2", "z_mean", "z_sigma", "z", "grad/encoder.input_layer.embedding.weight",
           "grad/encoder.rconv_layer_1.weight", "grad/encoder.rconv_layer_1.loop_weight",
           "grad/encoder.rconv_layer_2.weight", "grad/encoder.rconv_layer_2.loop_weight"]


def shrink(out, seed):
    """Keep a case under 1 MB: leave out the random inputs tests/helpers.py draws again from the seed (their
    digest stays), the unused training triples, and all but a seeded half of the rows of the large outputs."""
    from helpers import REDRAWN, inputs_sha256
    small = {key: val for key, val in out.items() if key not in REDRAWN and key not in ("train_triples", "edge_norm")}
    small["seed"] = np.asarray(seed, dtype=np.int64)
    small["inputs_sha256"] = np.asarray(inputs_sha256(out))
    rng = np.random.default_rng(seed)
    for key in SAMPLED:
        rows = np.sort(rng.choice(len(out[key]), len(out[key]) // 2, replace=False))
        small[key], small["rows/" + key] = out[key][rows], rows
    return small


def kgvae_case(name, n_ent, n_rel, h, bases, k, n_flows, n_train, batch, neg, kl_param,
               dropout, seed, shrink_to_1mb=False):
    rng = np.random.default_rng(seed)
    torch.manual_seed(seed)
    train = synthetic_triples(rng, n_ent, n_rel, n_train)
    test = synthetic_triples(rng, n_ent, n_rel, 64)
    with contextlib.redirect_stdout(io.StringIO()):
        model = ref_lp.LinkPredict(ref_model.KGVAE, n_ent, h, n_rel, num_bases=bases,
                                   num_hidden_layers=2, dropout=dropout, use_cuda=False,
                                   reg_param=0.01, kl_param=kl_param, mmd_param=0,
                                   k=k, n_flows=n_flows)
    # biases are zero-initialised by DGL; randomise so the fixture exercises them
    with torch.no_grad():
        model.encoder.rconv_layer_1.h_bias.normal_(0, 0.1)
        model.encoder.rconv_layer_2.h_bias.normal_(0, 0.1)

    # ---- sampling through the reference's legacy global numpy RNG -------
    np.random.seed(seed)
    adj_list, degrees = ref_utils.get_adj_and_degrees(n_ent, train)
    g, node_id, edge_type, node_norm, data, labels = \
        ref_utils.generate_sampled_graph_and_labels(train, batch, 0.5, n_rel, adj_list,
                                                    degrees, neg, "uniform")
    edge_norm = ref_lp.node_norm_to_edge_norm(g, torch.from_numpy(node_norm).view(-1, 1))
    n_nodes = len(node_id)
    eps = torch.randn(n_nodes, h)
    keep = 1.0 - dropout
    mask1 = (torch.rand(n_nodes, h) < keep).float() / keep
    mask2 = (torch.rand(n_nodes, 2 * h) < keep).float() / keep
    model.encoder.rconv_layer_1.dropout_mask = mask1
    model.encoder.rconv_layer_2.dropout_mask = mask2

    taps = {}
    model.encoder.rconv_layer_1.register_forward_hook(lambda m, i, o: taps.__setitem__("h1", o.detach().clone()))
    model.encoder.rconv_layer_2.register_forward_hook(lambda m, i, o: taps.__setitem__("h2", o.detach().clone()))

    model.train()
    node_id_t = torch.from_numpy(node_id).view(-1, 1).long()
    with preset_randn(eps):
        embed = model(g, node_id_t, torch.from_numpy(edge_type), edge_norm)
    if n_flows == 0:
        model.encoder.flow_log_prob = 0.0          # documented deviation (SURVEY F5)
    loss, pred, kl, mmd = model.get_loss(g, embed, torch.from_numpy(data), torch.from_numpy(labels))
    score = model.calc_score(embed, torch.from_numpy(data))
    if n_flows > 0:
        score = score + model.encoder.get_flow_log_prob()
    loss.backward()

    out = {
        "cfg": np.array([n_ent, n_rel, h, bases, k, n_flows, neg], dtype=np.int64),
        "cfg_f": np.array([0.01, kl_param, dropout], dtype=np.float64),
        "train_triples": train, "test_triples": test,
        "g_src": g._src.numpy(), "g_dst": g._dst.numpy(), "edge_type": edge_type,
        "node_norm": node_norm, "edge_norm": edge_norm.numpy(), "node_id": node_id,
        "samples": data, "labels": labels,
        "eps": eps.numpy(), "mask1": mask1.numpy(), "mask2": mask2.numpy(),
        "h1": taps["h1"].numpy(), "h2": taps["h2"].numpy(),
        "z_mean": model.encoder.z_mean.detach().numpy(),
        "z_sigma": model.encoder.z_sigma.detach().numpy(),
        "z": embed.detach().numpy(), "score": score.detach().numpy(),
        "loss": loss.detach().numpy(), "predict_loss": pred.detach().numpy(),
        "kl": np.asarray(kl.detach().numpy()).reshape(-1),
        "reg": model.regularization_loss(embed).detach().numpy(),
    }
    if n_flows > 0:
        out["flow_log_prob"] = model.encoder.flow_log_prob.detach().numpy()
    for key, val in model.state_dict().items():
        out["param/" + key] = val.detach().numpy()
    for key, val in model.named_parameters():
        if val.grad is not None:
            out["grad/" + key] = val.grad.detach().numpy()

    # ---- evaluation on the graph built from the test triples (SURVEY F6) ----
    model.eval()
    model.encoder.rconv_layer_1.dropout_mask = None
    model.encoder.rconv_layer_2.dropout_mask = None
    test_t = torch.from_numpy(test)
    tg, trel, tnorm = ref_utils.build_test_graph(n_ent, n_rel, test_t)
    tnorm_e = ref_lp.node_norm_to_edge_norm(tg, torch.from_numpy(tnorm).view(-1, 1))
    all_ids = torch.arange(n_ent).view(-1, 1)
    eps_eval = torch.randn(n_ent, h)
    with torch.no_grad(), preset_randn(eps_eval):
        emb_eval = model(tg, all_ids, torch.from_numpy(trel), tnorm_e)
    flp = model.encoder.get_flow_log_prob() if n_flows > 0 else 0.0
    with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
        s, r, o = test_t[:, 0], test_t[:, 1], test_t[:, 2]
        rs = ref_utils.perturb_and_get_rank(emb_eval, model.w_relation, o, r, s, len(test), 16, True, flp)
        ro = ref_utils.perturb_and_get_rank(emb_eval, model.w_relation, s, r, o, len(test), 16, True, flp)
        mrr = ref_utils.calc_mrr(emb_eval, model.w_relation, test_t, hits=[1, 3, 10], eval_bz=16,
                                 all_batches=True, flow_log_prob=flp)
    out.update({
        "eval_src": tg._src.numpy(), "eval_dst": tg._dst.numpy(), "eval_etype": trel,
        "eval_node_norm": tnorm, "eval_eps": eps_eval.numpy(), "eval_emb": emb_eval.numpy(),
        "eval_flow_log_prob": np.asarray(float(flp), dtype=np.float32),
        "eval_ranks": torch.cat([rs, ro]).numpy(), "eval_mrr": np.asarray(mrr),
    })
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **(shrink(out, seed) if shrink_to_1mb else out))
    print(f"{name}: nodes={n_nodes} edges={len(edge_type)} samples={len(labels)} "
          f"loss={float(loss):.6f} mrr={mrr:.6f} -> {os.path.getsize(path) / 1024:.0f} KiB")


def sampling_case():
    """Integer-exact sampler outputs at a mid-size shape (legacy np.random path)."""
    rng = np.random.default_rng(7)
    n_ent, n_rel = 3000, 24
    train = synthetic_triples(rng, n_ent, n_rel, 20000)
    np.random.seed(0)
    g, node_id, edge_type, node_norm, data, labels = \
        ref_utils.generate_sampled_graph_and_labels(train, 4000, 0.5, n_rel, None, None, 10, "uniform")
    out = {"cfg": np.array([n_ent, n_rel, 20000, 4000, 10, 7, 0], dtype=np.int64),
           "g_src": g._src.numpy().astype(np.int32), "g_dst": g._dst.numpy().astype(np.int32),
           "edge_type": edge_type.astype(np.int32), "node_norm": node_norm,
           "node_id": node_id.astype(np.int32), "samples": data.astype(np.int32),
           "labels_sum": np.asarray(labels.sum())}
    path = os.path.join(HERE, "sampling_seed0.npz")
    np.savez_compressed(path, **out)
    print(f"sampling_seed0: nodes={len(node_id)} edges={len(edge_type)} -> {os.path.getsize(path) / 1024:.0f} KiB")


def rank_case():
    """Exactly representable inputs (multiples of 1/8 in [-1,1], h=16): every product
    and partial sum is exact in fp32 for ANY accumulation order, so scores are
    order-independent and include genuine ties.  Records the reference's ranks
    (its non-stable sort) next to the scores."""
    rng = np.random.default_rng(11)
    V, R, h, T = 96, 5, 16, 80
    emb = torch.from_numpy(rng.integers(-8, 9, size=(V, h)).astype(np.float32) / 8)
    w = torch.from_numpy(rng.integers(-8, 9, size=(R, h)).astype(np.float32) / 8)
    test = torch.from_numpy(synthetic_triples(rng, V, R, T))
    s, r, o = test[:, 0], test[:, 1], test[:, 2]
    with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
        rs = ref_utils.perturb_and_get_rank(emb, w, o, r, s, T, 32, True, 0.0)
        ro = ref_utils.perturb_and_get_rank(emb, w, s, r, o, T, 32, True, 0.0)
        mrr = ref_utils.calc_mrr(emb, w, test, hits=[1, 3, 10], eval_bz=32, flow_log_prob=0.0)
    out = {"emb": emb.numpy(), "w": w.numpy(), "test_triples": test.numpy(),
           "ref_ranks": torch.cat([rs, ro]).numpy(), "ref_mrr": np.asarray(mrr)}
    path = os.path.join(HERE, "rank_exact.npz")
    np.savez_compressed(path, **out)
    print(f"rank_exact: mrr={mrr:.6f} -> {os.path.getsize(path) / 1024:.0f} KiB")


def made_case():
    """One MADE block + permute: forward, log-det, inverse, input/weight grads."""
    torch.manual_seed(3)
    D, nh, N = 12, 3, 40
    made = ref_flow.MADE(D, D, nh)
    perm = ref_flow.PermuteLayer(D)
    z = torch.randn(N, D, requires_grad=True)
    x, log_det = made.forward(z)
    xp, zero = perm.forward(x)
    (xp.pow(2).sum() + log_det.sum()).backward()
    with torch.no_grad():
        zi, ldi = made.inverse(x.detach())
    out = {"cfg": np.array([D, nh, N]), "z": z.detach().numpy(), "x": x.detach().numpy(),
           "x_perm": xp.detach().numpy(), "log_det": log_det.detach().numpy(),
           "perm_log_det": zero.numpy(), "z_grad": z.grad.numpy(),
           "inv_z": zi.numpy(), "inv_log_det": ldi.numpy()}
    for i, deg in enumerate(made.m):
        out[f"deg/{i}"] = deg.numpy()
    for key, val in made.state_dict().items():
        out["param/" + key] = val.numpy()
    for key, val in made.named_parameters():
        out["grad/" + key] = val.grad.numpy()
    path = os.path.join(HERE, "made_block.npz")
    np.savez_compressed(path, **out)
    print(f"made_block -> {os.path.getsize(path) / 1024:.0f} KiB")


def entity_case():
    """Entity classification (config 4, row a4): the reference's ``EntityClassify`` (kgvae/entity_classify.py
    :23-43, imported verbatim) - basis RelGraphConv on integer node ids, one hidden layer, softmax output -
    one full-graph training step as in its main() (:106-113): logits, cross-entropy on the training
    nodes, every gradient."""
    with contextlib.redirect_stdout(io.StringIO()):
        import entity_classify as ref_ec       # reference, verbatim
        from dgl import DGLGraph
    rng = np.random.default_rng(21)
    torch.manual_seed(21)
    n, R, E, h, C, bases = 120, 9, 900, 10, 4, 4
    src = rng.integers(0, n, E)
    dst = rng.integers(0, n - 2, E)                      # the last nodes stay without in-edges
    et = rng.integers(0, R, E)
    key = dst.astype(np.int64) * R + et                  # the loader's norm: 1 / same-type edges into dst
    _, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    norm = (1.0 / cnt[inv]).astype(np.float32)
    labels = rng.integers(0, C, n)
    train_idx = rng.permutation(n)[:40]
    g = DGLGraph()
    g.add_nodes(n)
    g.add_edges(src, dst)
    model = ref_ec.EntityClassify(len(g), h, C, R, num_bases=bases, num_hidden_layers=1, dropout=0,
                                  use_self_loop=True, use_cuda=False)
    with torch.no_grad():
        for layer in model.layers:
            layer.h_bias.normal_(0, 0.1)
    feats = torch.arange(n)
    logits = model(g, feats, torch.from_numpy(et), torch.from_numpy(norm).unsqueeze(1))
    import torch.nn.functional as F
    loss = F.cross_entropy(logits[train_idx], torch.from_numpy(labels).view(-1)[train_idx])
    loss.backward()
    out = {"cfg": np.array([n, R, E, h, C, bases], dtype=np.int64), "src": src, "dst": dst, "etype": et,
           "norm": norm, "labels": labels, "train_idx": train_idx, "logits": logits.detach().numpy(),
           "loss": loss.detach().numpy()}
    for key_, val in model.state_dict().items():
        out["param/" + key_] = val.detach().numpy()
    for key_, val in model.named_parameters():
        out["grad/" + key_] = val.grad.detach().numpy()
    path = os.path.join(HERE, "entity_classify_toy.npz")
    np.savez_compressed(path, **out)
    print(f"entity_classify_toy: loss={float(loss):.6f} layers={len(model.layers)} -> {os.path.getsize(path) / 1024:.0f} KiB")


def neighbor_sampler_case():
    """The reference's neighbourhood edge sampler (kgvae/utils.py:33-76) on a seeded graph: its picks are a
    function of the legacy global numpy stream only, so they must be reproduced integer for integer."""
    rng = np.random.default_rng(31)
    n_ent, n_rel, n_train, sample = 300, 7, 2000, 250
    train = synthetic_triples(rng, n_ent, n_rel, n_train)
    adj_list, degrees = ref_utils.get_adj_and_degrees(n_ent, train)
    np.random.seed(5)
    edges = ref_utils.sample_edge_neighborhood(adj_list, degrees, n_train, sample)
    np.random.seed(6)
    g, node_id, edge_type, node_norm, data, labels = ref_utils.generate_sampled_graph_and_labels(
        train, sample, 0.5, n_rel, adj_list, degrees, 3, "neighbor")
    out = {"cfg": np.array([n_ent, n_rel, n_train, sample], dtype=np.int64), "train_triples": train,
           "edges": np.asarray(edges, dtype=np.int64), "node_id": node_id.astype(np.int64),
           "edge_type": edge_type.astype(np.int64), "samples": data.astype(np.int64),
           "g_src": g._src.numpy().astype(np.int64), "g_dst": g._dst.numpy().astype(np.int64)}
    path = os.path.join(HERE, "neighbor_sampler_seed5.npz")
    np.savez_compressed(path, **out)
    print(f"neighbor_sampler_seed5: picked={len(edges)} nodes={len(node_id)} -> {os.path.getsize(path) / 1024:.0f} KiB")


def mmd_case():
    """The MMD term (row a8; on in the README run, --mmd-param=1): KGVAE.get_mmd (kgvae/model.py:89-102) with
    python's ``random`` seeded and the prior noise preset - 200 prior samples pushed through the flow against
    200 posterior rows; value and gradients wrt z, the prior parameters and the flow."""
    import random
    torch.manual_seed(17)
    n_ent, n_rel, h, bases, k, n_flows, N = 260, 6, 20, 4, 10, 1, 260
    with contextlib.redirect_stdout(io.StringIO()):
        model = ref_lp.LinkPredict(ref_model.KGVAE, n_ent, h, n_rel, num_bases=bases, num_hidden_layers=2,
                                   dropout=0.0, use_cuda=False, reg_param=0.01, kl_param=1e-3, mmd_param=1.0,
                                   k=k, n_flows=n_flows)
    z = torch.randn(N, h, requires_grad=True)
    eps = torch.randn(200, h)
    random.seed(9)
    with preset_randn(eps):
        mmd = model.encoder.get_mmd(z)
    mmd.backward()
    out = {"cfg": np.array([n_ent, n_rel, h, bases, k, n_flows, N], dtype=np.int64), "z": z.detach().numpy(),
           "eps": eps.numpy(), "mmd": mmd.detach().numpy(), "grad_z": z.grad.numpy()}
    for key, val in model.state_dict().items():
        out["param/" + key] = val.detach().numpy()
    for key, val in model.named_parameters():
        if val.grad is not None:
            out["grad/" + key] = val.grad.detach().numpy()
    path = os.path.join(HERE, "mmd_term.npz")
    np.savez_compressed(path, **out)
    print(f"mmd_term: mmd={float(mmd):.6f} grads={sorted(k_ for k_ in out if k_.startswith('grad/'))[:3]}... -> {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    kgvae_case("kgvae_tiny_noflow", n_ent=150, n_rel=5, h=20, bases=4, k=3, n_flows=0,
               n_train=600, batch=240, neg=3, kl_param=1e-2, dropout=0.2, seed=1)
    kgvae_case("kgvae_tiny_flow3", n_ent=150, n_rel=5, h=20, bases=4, k=10, n_flows=3,
               n_train=600, batch=240, neg=3, kl_param=1e-2, dropout=0.2, seed=2)
    kgvae_case("kgvae_small_noflow", n_ent=400, n_rel=12, h=100, bases=20, k=10, n_flows=0,
               n_train=3000, batch=800, neg=10, kl_param=1e-5, dropout=0.2, seed=4, shrink_to_1mb=True)
    sampling_case()
    rank_case()
    made_case()
    entity_case()
    neighbor_sampler_case()
    mmd_case()
