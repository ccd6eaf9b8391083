"""Pin the oracle port (oracle/kgvae_oracle.py) against vectors produced by the
UNMODIFIED reference (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from helpers import O, assert_close, at_golden_rows, golden_graph, golden_params, made_relu_patterns, oracle_train_step

CASES = ["kgvae_tiny_noflow", "kgvae_tiny_flow3", "kgvae_small_noflow"]


@pytest.mark.parametrize("case", CASES)
def test_forward_intermediates(golden, case):
    gv = golden(case)
    _, enc, out = oracle_train_step(gv, requires_grad=False)
    for key in ("h1", "h2", "z_mean", "z_sigma", "z"):
        assert_close(at_golden_rows(gv, key, enc[key]), gv[key], 2e-5, f"{case}:{key}")
    assert_close(out["score"], gv["score"], 2e-5, "score")
    assert_close(out["loss"], gv["loss"], 1e-5, "loss")
    assert_close(out["predict_loss"], gv["predict_loss"], 1e-5, "predict_loss")
    assert_close(out["kl"].reshape(-1), gv["kl"], 1e-5, "kl")
    assert_close(out["reg"], gv["reg"], 1e-5, "reg")
    if "flow_log_prob" in gv:
        assert_close(enc["flow_log_prob"], gv["flow_log_prob"], 1e-5, "flow_log_prob")


@pytest.mark.parametrize("case", CASES)
def test_gradients(golden, case):
    gv = golden(case)
    params, _, out = oracle_train_step(gv, requires_grad=True)
    out["loss"].backward()
    checked = 0
    for key, val in gv.items():
        if key.startswith("grad/"):
            name = key[len("grad/"):]
            assert_close(at_golden_rows(gv, key, params[name].grad), val, 5e-5, f"{case}:grad {name}")
            checked += 1
    assert checked >= 9


@pytest.mark.parametrize("case", CASES)
def test_graph_build_is_integer_exact(golden, case):
    """a1: reverse edges + (dst,src,rel) order + 1/in_deg, from the sampled positives."""
    gv = golden(case)
    n_ent, n_rel = int(gv["cfg"][0]), int(gv["cfg"][1])
    test = gv["test_triples"]
    g = O.build_graph_from_triplets(n_ent, n_rel, test[:, 0], test[:, 1], test[:, 2])
    assert np.array_equal(g["src"], gv["eval_src"])
    assert np.array_equal(g["dst"], gv["eval_dst"])
    assert np.array_equal(g["etype"], gv["eval_etype"])
    assert np.array_equal(g["norm"], gv["eval_node_norm"])


def test_sampler_is_integer_exact(golden):
    """a11: legacy np.random call order reproduces the reference's sampled ids bit for bit."""
    gv = golden("sampling_seed0")
    n_ent, n_rel, n_train, batch, neg, seed, _ = (int(x) for x in gv["cfg"])
    rng = np.random.default_rng(seed)
    s = rng.integers(0, n_ent, size=n_train)
    o = rng.integers(0, n_ent, size=n_train)
    r = rng.integers(0, n_rel, size=n_train)
    train = np.stack([s, r, o], axis=1).astype(np.int64)
    np.random.seed(0)
    graph, uniq_v, samples, labels = O.generate_sampled_graph_and_labels(train, batch, 0.5, n_rel, neg)
    assert np.array_equal(graph["src"], gv["g_src"])
    assert np.array_equal(graph["dst"], gv["g_dst"])
    assert np.array_equal(graph["etype"], gv["edge_type"])
    assert np.array_equal(graph["norm"], gv["node_norm"])
    assert np.array_equal(uniq_v, gv["node_id"])
    assert np.array_equal(samples, gv["samples"])
    assert float(labels.sum()) == float(gv["labels_sum"])


@pytest.mark.parametrize("case", CASES)
def test_eval_embedding_and_ranks(golden, case):
    gv = golden(case)
    n_ent, n_rel, h, bases, k, n_flows, _ = (int(x) for x in gv["cfg"])
    params = golden_params(gv)
    graph = golden_graph(gv, prefix="eval_", etype_key="eval_etype", norm_key="eval_node_norm")
    enc = O.kgvae_encode(params, graph, np.arange(n_ent), torch.from_numpy(gv["eval_eps"]), bases, n_flows)
    assert_close(enc["z"], gv["eval_emb"], 2e-5, "eval embedding")
    # rank on the reference's own embedding so only the ranking rule is under test
    emb = torch.from_numpy(gv["eval_emb"])
    flp = float(gv["eval_flow_log_prob"])
    mrr, hits, ranks = O.calc_mrr(emb, params["w_relation"], gv["test_triples"], hits=[1, 3, 10],
                                  eval_bz=16, flow_log_prob=flp, policy="reference")
    assert np.array_equal(ranks.numpy() - 1, gv["eval_ranks"])
    assert abs(mrr - float(gv["eval_mrr"])) < 1e-6
    # stable policy lies inside every tie interval and matches when there are no ties
    _, _, stable = O.calc_mrr(emb, params["w_relation"], gv["test_triples"], eval_bz=16,
                              flow_log_prob=flp, policy="stable")
    t = torch.from_numpy(gv["test_triples"])
    for (a, b), sl in (((t[:, 2], t[:, 0]), slice(0, len(t))), ((t[:, 0], t[:, 2]), slice(len(t), None))):
        sc = torch.sigmoid(O.eval_scores(emb, params["w_relation"], a, t[:, 1], flp))
        lo, hi = O.rank_interval(sc, b)
        st = stable[sl] - 1
        assert bool(((st >= lo) & (st <= hi)).all())
        untied = lo == hi
        assert np.array_equal(st[untied].numpy(), gv["eval_ranks"][sl][untied.numpy()])


def test_exact_rank_fixture(golden):
    """Order-independent scores (dyadic inputs) with genuine ties."""
    gv = golden("rank_exact")
    emb, w = torch.from_numpy(gv["emb"]), torch.from_numpy(gv["w"])
    t = torch.from_numpy(gv["test_triples"])
    _, _, ref_policy = O.calc_mrr(emb, w, t, eval_bz=32, flow_log_prob=0.0, policy="reference")
    assert np.array_equal(ref_policy.numpy() - 1, gv["ref_ranks"])
    # logits-based stable ranks lie in the reference's sigmoid tie interval
    _, _, stable = O.calc_mrr(emb, w, t, eval_bz=32, policy="stable", apply_sigmoid=False)
    sc_s = torch.sigmoid(O.eval_scores(emb, w, t[:, 2], t[:, 1]))
    sc_o = torch.sigmoid(O.eval_scores(emb, w, t[:, 0], t[:, 1]))
    lo = torch.cat([O.rank_interval(sc_s, t[:, 0])[0], O.rank_interval(sc_o, t[:, 2])[0]])
    hi = torch.cat([O.rank_interval(sc_s, t[:, 0])[1], O.rank_interval(sc_o, t[:, 2])[1]])
    assert bool(((stable - 1 >= lo) & (stable - 1 <= hi)).all())
    assert bool((torch.from_numpy(gv["ref_ranks"]) >= lo).all() and (torch.from_numpy(gv["ref_ranks"]) <= hi).all())
    assert int((lo != hi).sum()) > 0     # the fixture really contains ties


def test_made_block(golden):
    gv = golden("made_block")
    D, nh, N = (int(x) for x in gv["cfg"])
    ws = [torch.from_numpy(gv[f"param/net.{2 * l}.weight"]).requires_grad_(True) for l in range(nh + 2)]
    bs = [torch.from_numpy(gv[f"param/net.{2 * l}.bias"]).requires_grad_(True) for l in range(nh + 2)]
    masks, degs = O.made_masks(D, D, nh), O.made_degrees(D, D, nh)
    for l in range(nh + 2):
        assert np.array_equal(masks[l].numpy(), gv[f"param/net.{2 * l}.mask"])
    for i, d in enumerate(degs):
        assert np.array_equal(d.numpy(), gv[f"deg/{i}"])
    z = torch.from_numpy(gv["z"]).requires_grad_(True)
    x, log_det = O.made_forward(z, ws, bs, masks, degs)
    assert_close(x, gv["x"], 1e-5, "made x")
    assert_close(log_det, gv["log_det"], 1e-5, "made log_det")
    assert_close(x.flip(1), gv["x_perm"], 1e-5, "permute")
    (x.flip(1).pow(2).sum() + log_det.sum()).backward()
    assert_close(z.grad, gv["z_grad"], 5e-5, "made dz")
    for l in range(nh + 2):
        assert_close(ws[l].grad, gv[f"grad/net.{2 * l}.weight"], 5e-5, f"dW{l}")
        assert_close(bs[l].grad, gv[f"grad/net.{2 * l}.bias"], 5e-5, f"db{l}")
    zi, ldi = O.made_inverse(x.detach(), [w.detach() for w in ws], [b.detach() for b in bs], masks)
    assert_close(zi, gv["inv_z"], 1e-5, "inverse z")
    assert_close(ldi, gv["inv_log_det"], 1e-5, "inverse log_det")


def test_made_relu_patterns_are_the_plain_function(golden):
    """``relu_patterns`` / ``made_relu_patterns``: handed the oracle's own ReLU pattern, the oracle computes the plain
    function bit for bit (forward and every gradient, one MADE and a two-MADE flow); with one unit flipped, only the
    row that unit belongs to changes."""
    gv = golden("made_block")
    D, nh, N = (int(x) for x in gv["cfg"])
    masks, degs = O.made_masks(D, D, nh), O.made_degrees(D, D, nh)
    W = [torch.from_numpy(gv[f"param/net.{2 * l}.weight"]).double() for l in range(nh + 2)]
    B = [torch.from_numpy(gv[f"param/net.{2 * l}.bias"]).double() for l in range(nh + 2)]
    Z = torch.from_numpy(gv["z"]).double()
    gen = torch.Generator().manual_seed(3)
    gx, gl = torch.randn(N, D, generator=gen, dtype=torch.float64), torch.randn(N, generator=gen, dtype=torch.float64)

    def run(patterns):
        ws, bs = [t.clone().requires_grad_(True) for t in W], [t.clone().requires_grad_(True) for t in B]
        z = Z.clone().requires_grad_(True)
        x, log_det = O.made_forward(z, ws, bs, masks, degs, patterns)
        ((x * gx).sum() + (log_det * gl).sum()).backward()
        return [x.detach(), log_det.detach(), z.grad] + [t.grad for t in ws + bs]

    plain = run(None)
    x_replay, pats, _ = made_relu_patterns(Z, W, B, masks, degs)
    assert torch.equal(x_replay, plain[0])
    assert len(pats) == len(degs) and all(len(p) == nh + 1 for p in pats)
    for a, b in zip(run(pats), plain):
        assert torch.equal(a, b)
    # first pass: x = 0, every row has the same pattern - one [1, h] row stands for all of them
    first_row = [[t[:1] for t in pats[0]]] + pats[1:]
    for a, b in zip(run(first_row), plain):
        assert torch.equal(a, b)

    # flip one active unit of degree 0 (it feeds every output but the first) in the last pass, whose outputs are final
    row = int(torch.nonzero(pats[-1][0][:, 0])[0, 0])
    flipped = [[t.clone() for t in p] for p in pats]
    flipped[-1][0][row, 0] = False
    _, _, (n_flip, _) = made_relu_patterns(Z, W, B, masks, degs, against=flipped)
    assert n_flip == 1
    got = run(flipped)
    others = torch.arange(N) != row
    for i in (0, 2):                                         # x and dz: row-local
        assert torch.equal(got[i][others], plain[i][others])
        assert not torch.equal(got[i][row], plain[i][row])
    assert torch.equal(got[1][others], plain[1][others])

    # the flow: MADE, reverse, MADE, reverse - patterns per MADE through iaf_forward and kgvae_encode's plumbing
    h, n_flows = 10, 2
    params = {k: v.double().requires_grad_(True) for k, v in O.init_params(30, h, 3, 2, 4, n_flows, seed=5).items()}
    z0 = torch.randn(30, h, generator=gen, dtype=torch.float64)
    z_p, lds_p, flp_p = O.iaf_forward(z0, params, n_flows)
    (z_p.pow(2).sum() + flp_p).backward()
    plain_grads = {k: v.grad.clone() for k, v in params.items() if v.grad is not None}
    flow_pats, zc = [], z0
    with torch.no_grad():
        for ws, bs in O.flow_params(params, n_flows):
            zc, pats_f, _ = made_relu_patterns(zc, ws, bs, O.made_masks(h, h, n_flows), O.made_degrees(h, h, n_flows))
            flow_pats.append(pats_f)
            zc = zc.flip(1)
    assert torch.equal(zc, z_p.detach())
    for v in params.values():
        v.grad = None
    z_q, lds_q, flp_q = O.iaf_forward(z0, params, n_flows, flow_pats)
    (z_q.pow(2).sum() + flp_q).backward()
    assert torch.equal(z_q, z_p) and torch.equal(lds_q, lds_p)
    assert plain_grads.keys() == {k for k, v in params.items() if v.grad is not None}
    for k, g in plain_grads.items():
        assert torch.equal(params[k].grad, g), k


def test_bdd_equals_dense_block_diagonal():
    """Property (SURVEY 8c): bdd message == dense block-diagonal matmul."""
    torch.manual_seed(0)
    N, E, R, B, si, so = 30, 90, 4, 3, 4, 5
    x = torch.randn(N, B * si)
    graph = {"num_nodes": N, "src": np.random.default_rng(0).integers(0, N, E),
             "dst": np.random.default_rng(1).integers(0, N, E),
             "etype": np.random.default_rng(2).integers(0, R, E),
             "edge_norm": np.random.default_rng(3).random((E, 1)).astype(np.float32)}
    weight = torch.randn(R, B * si * so)
    loop = torch.randn(B * si, B * so)
    bias = torch.randn(B * so)
    got = O.rgcn_bdd_layer(x, graph, weight, bias, loop, B)
    want = x @ loop + bias
    for e in range(E):
        dense = torch.block_diag(*weight[graph["etype"][e]].view(B, si, so))
        want[graph["dst"][e]] += float(graph["edge_norm"][e, 0]) * (x[graph["src"][e]] @ dense)
    assert_close(got, want, 1e-5, "bdd vs dense")


def test_made_is_autoregressive():
    D, nh = 8, 3
    masks = O.made_masks(D, D, nh)
    conn = masks[0]
    for m in masks[1:-1]:
        conn = m @ conn
    conn = masks[-1][:D] @ conn
    assert float(torch.triu(conn, diagonal=0).abs().sum()) == 0.0   # out_j sees only in_{<j}


def test_entity_classify_against_reference(golden):
    """Row a4: the oracle's basis layers reproduce the reference's EntityClassify (entity_classify.py:23-43,
    imported verbatim by make_golden.py): logits, cross-entropy on the training nodes, every gradient."""
    gv = golden("entity_classify_toy")
    n, R, E, h, C, bases = (int(v) for v in gv["cfg"])
    graph = {"num_nodes": n, "src": gv["src"], "dst": gv["dst"], "etype": gv["etype"],
             "edge_norm": gv["norm"].reshape(-1, 1)}
    p = {k[len("param/"):]: torch.from_numpy(v.copy()).requires_grad_(True) for k, v in gv.items() if k.startswith("param/")}
    acts = [torch.relu, torch.relu, lambda t: torch.softmax(t, dim=1)]
    x = torch.arange(n)
    for i, act in enumerate(acts):
        x = O.rgcn_basis_layer(x, graph, p[f"layers.{i}.weight"], p[f"layers.{i}.w_comp"], p[f"layers.{i}.h_bias"],
                               p[f"layers.{i}.loop_weight"], act)
    assert_close(x, gv["logits"], 2e-6, "logits")
    idx = torch.from_numpy(gv["train_idx"])
    loss = torch.nn.functional.cross_entropy(x[idx], torch.from_numpy(gv["labels"])[idx])
    assert_close(loss, gv["loss"], 2e-6, "loss")
    loss.backward()
    for name, t in p.items():
        assert_close(t.grad, gv["grad/" + name], 2e-5, f"grad {name}")
