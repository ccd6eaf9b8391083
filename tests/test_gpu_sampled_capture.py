"""Sampled-subgraph training steps as one CUDA-graph replay: ``utils.SampledDeviceSampler`` pads the node set of a
uniform edge sample to a fixed budget, ``kg_sample_relabel`` relabels it on the device, the rows kernels keep the
padding out of the KL and regulariser, and ``CapturedTrainStep(sampler=...)`` replays the whole iteration."""
import copy
import os

import numpy as np
import pytest
import torch

import gcn_vae_b200 as K
from helpers import RTOL, rel_err

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _relabel_reference(picked):
    uniq, inv = np.unique(np.concatenate([picked[:, 0], picked[:, 2]]), return_inverse=True)
    B = picked.shape[0]
    return uniq, inv[:B], inv[B:]


def _check_relabel(picked, num_nodes, cap, out):
    node_id, src, rel, dst, n_valid = (t.cpu().numpy() for t in out)
    uniq, s_ref, d_ref = _relabel_reference(picked)
    n = len(uniq)
    assert int(n_valid[0]) == n and node_id.shape == (cap,)
    assert np.array_equal(node_id[:n], uniq)
    assert np.array_equal(src, s_ref) and np.array_equal(dst, d_ref) and np.array_equal(rel, picked[:, 1])
    assert np.array_equal(node_id[n:], np.arange(n, cap)) and node_id.max() < num_nodes
    assert np.bincount(node_id, minlength=num_nodes).max() <= 2


def _relabel_cases():
    rng = np.random.default_rng(0)
    one = np.array([[3, 1, 7]])
    same = np.stack([np.full(100, 7), rng.integers(0, 5, 100), np.full(100, 7)], 1)
    dense = np.stack([rng.integers(0, 60, 200), rng.integers(0, 5, 200), rng.integers(0, 60, 200)], 1)
    fb = K.datasets.synthetic_kg("FB15k-237", seed=0)
    fb_pick = fb.train[rng.choice(len(fb.train), 20000, replace=False)]
    fb_cap = min(40000, len(np.unique(fb.train[:, [0, 2]])))
    return [("B=1", one, 50, 2), ("one entity", same, 500, 200), ("2B > entities", dense, 60, 60),
            ("FB15k-237 B=20000", fb_pick, fb.num_nodes, fb_cap)]


@pytest.mark.parametrize("case", _relabel_cases(), ids=lambda c: c[0])
def test_sample_relabel_matches_np_unique(case):
    _, picked, num_nodes, cap = case
    out = K.ops.sample_relabel(torch.from_numpy(picked).to(DEV, torch.int32), num_nodes, cap)
    _check_relabel(picked, num_nodes, cap, out)


def test_sample_relabel_clamps_n_valid_to_the_budget():
    """A caller whose budget is below the number of distinct ids still gets n_valid <= cap, so nothing drawn from
    [0, n_valid) indexes past the node set; the rows that are kept are the smallest ids."""
    rng = np.random.default_rng(2)
    picked = np.stack([rng.integers(0, 60, 200), rng.integers(0, 5, 200), rng.integers(0, 60, 200)], 1)
    uniq = np.unique(picked[:, [0, 2]])
    cap = len(uniq) - 10
    node_id, _, _, _, n_valid = K.ops.sample_relabel(torch.from_numpy(picked).to(DEV, torch.int32), 60, cap)
    assert int(n_valid) == cap and np.array_equal(node_id.cpu().numpy(), uniq[:cap])


def test_sample_relabel_replays_in_a_cuda_graph():
    """Captured once, replayed on two different draws: the same outputs as eager calls on those draws."""
    rng = np.random.default_rng(1)
    num_nodes, B = 3000, 1500
    draws = [np.stack([rng.integers(0, num_nodes, B), rng.integers(0, 9, B), rng.integers(0, num_nodes, B)], 1)
             for _ in range(3)]
    cap = 2 * B
    static = torch.from_numpy(draws[0]).to(DEV, torch.int32)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        K.ops.sample_relabel(static, num_nodes, cap)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = K.ops.sample_relabel(static, num_nodes, cap)
    seen = []
    for d in draws[1:]:
        static.copy_(torch.from_numpy(d).to(DEV, torch.int32))
        graph.replay()
        torch.cuda.synchronize()
        ref = K.ops.sample_relabel(torch.from_numpy(d).to(DEV, torch.int32), num_nodes, cap)
        for a, b in zip(out, ref):
            assert torch.equal(a, b)
        _check_relabel(d, num_nodes, cap, out)
        seen.append(int(out[4]))
    assert seen[0] != seen[1]


# ---------------------------------------------------------------------------------------------------------------
# rows kernels against the existing kernels run on the first n_valid rows
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h", [37, 40, 500])      # 37: the scalar (non-float4) forward
@pytest.mark.parametrize("k", [1, 4, 10, 16])
@pytest.mark.parametrize("which", ["1", "cap-1", "cap"])
def test_rows_kernels_match_the_existing_kernels_on_the_valid_rows(which, k, h):
    L = K._lib
    cap = 301
    nv = {"1": 1, "cap-1": cap - 1, "cap": cap}[which]
    g = torch.Generator(device=DEV).manual_seed(k * 1000 + h + nv)
    z = torch.randn(cap, h, device=DEV, generator=g)
    zm = torch.randn(cap, h, device=DEV, generator=g) * 0.5
    zv = torch.rand(cap, h, device=DEV, generator=g) + 0.1
    zp = torch.randn(2 * k, h, device=DEV, generator=g) * 0.3
    add = torch.randn(cap, h, device=DEV, generator=g)
    coefs = torch.tensor([0.7, 1.3, -0.2], device=DEV)
    n_valid = torch.tensor([nv], dtype=torch.int32, device=DEV)
    nan = lambda *shape: torch.full(shape, float("nan"), device=DEV)

    # reference: the existing kernels on an [nv, h] input
    pws_r, rows_r, resp_r = nan(3, k, h), nan(nv), nan(nv, k)
    L.call("kg_kl_mog_fwd", L.f32(z[:nv]), L.f32(zm[:nv]), L.f32(zv[:nv]), L.f32(zp), nv, h, k, L.f32(pws_r),
           L.f32(rows_r), L.f32(resp_r), L.stream())
    dz_r, dm_r, dv_r, dzp_r = nan(nv, h), nan(nv, h), nan(nv, h), torch.zeros(2 * k, h, device=DEV)
    L.call("kg_kl_mog_bwd_fused", L.f32(z[:nv]), L.f32(zm[:nv]), L.f32(zv[:nv]), L.f32(zp), L.f32(pws_r), L.f32(resp_r),
           1.0 / nv, nv, h, k, L.f32(coefs), L.f32(add[:nv]), L.f32(dz_r), L.f32(dm_r), L.f32(dv_r), L.f32(dzp_r),
           L.stream())
    # rows variants on the whole [cap, h] input
    pws, rows, resp = nan(3, k, h), nan(cap), nan(cap, k)
    L.call("kg_kl_mog_fwd_rows", L.f32(z), L.f32(zm), L.f32(zv), L.f32(zp), cap, h, k, L.i32(n_valid), L.f32(pws),
           L.f32(rows), L.f32(resp), L.stream())
    dz, dm, dv, dzp = nan(cap, h), nan(cap, h), nan(cap, h), torch.zeros(2 * k, h, device=DEV)
    L.call("kg_kl_mog_bwd_fused_rows", L.f32(z), L.f32(zm), L.f32(zv), L.f32(zp), L.f32(pws), L.f32(resp), cap, h, k,
           L.i32(n_valid), L.f32(coefs), L.f32(add), L.f32(dz), L.f32(dm), L.f32(dv), L.f32(dzp), L.stream())
    torch.cuda.synchronize()

    assert torch.equal(rows[:nv], rows_r) and torch.equal(resp[:nv], resp_r) and torch.equal(pws, pws_r)
    assert bool((rows[nv:] == 0).all())
    for got, ref in ((dz, dz_r), (dm, dm_r), (dv, dv_r)):
        assert torch.equal(got[:nv], ref)
        assert bool((got[nv:] == 0).all())
    assert rel_err(dzp, dzp_r) <= 1e-6

    ss = K.ops._sum_squares_rows(z, n_valid)
    assert rel_err(ss, (z[:nv].double() ** 2).sum()) <= 1e-6


# ---------------------------------------------------------------------------------------------------------------
# the sampler's procedure
# ---------------------------------------------------------------------------------------------------------------
def _toy_train(seed=3, n_ent=500, n_rel=7, T=4000):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(0, n_ent, T), rng.integers(0, n_rel, T), rng.integers(0, n_ent, T)], 1)


def test_sampled_device_sampler_follows_the_reference_procedure():
    """kgvae/utils.py:79-124,158-171 with a fixed node budget: B distinct training triples, relabelled in ascending
    id order; negatives replace exactly one end by a sampled node (heads about half); the graph is a split_size share
    of the positives in both directions with reverse relation ids and 1 / in-degree norms; padding nodes have no
    edges; draws differ and so does n_valid."""
    n_ent, n_rel, T, B, rate = 500, 7, 4000, 600, 5
    train = _toy_train(n_ent=n_ent, n_rel=n_rel, T=T)
    sm = K.utils.SampledDeviceSampler(torch.from_numpy(train).to(DEV), B, 0.5, n_rel, rate)
    assert sm.n == min(2 * B, len(np.unique(train[:, [0, 2]])))
    torch.manual_seed(0)
    draws = [sm.sample() for _ in range(8)]
    a = draws[0]
    n = int(a["n_valid"])
    node_id = a["node_id"].cpu().numpy().reshape(-1)
    smp = a["samples"].cpu().numpy()
    assert node_id.shape == (sm.n,) and smp.shape == (B * (rate + 1), 3)
    pos = smp[:B]
    # the positives are B distinct picks among the training triples (as a multiset), relabelled in ascending id order
    orig = np.stack([node_id[pos[:, 0]], pos[:, 1], node_id[pos[:, 2]]], 1)
    count = {}
    for t in map(tuple, train):
        count[t] = count.get(t, 0) + 1
    for t in map(tuple, orig):
        count[t] = count.get(t, 0) - 1
        assert count[t] >= 0, t
    uniq = np.unique(orig[:, [0, 2]])
    assert n == len(uniq) and np.array_equal(node_id[:n], uniq) and np.array_equal(node_id[n:], np.arange(n, sm.n))
    neg = smp[B:].reshape(rate, B, 3)
    same_s, same_o = neg[:, :, 0] == pos[None, :, 0], neg[:, :, 2] == pos[None, :, 2]
    assert np.array_equal(neg[:, :, 1], np.broadcast_to(pos[None, :, 1], (rate, B)))
    assert (same_s | same_o).all()
    assert 0.45 < float((~same_s).mean()) < 0.55
    assert smp[:, [0, 2]].min() >= 0 and smp[:, [0, 2]].max() < n
    lab = a["labels"].cpu().numpy()
    assert lab[:B].min() == 1 and lab[B:].max() == 0
    src, dst, et = (a[k].cpu().numpy() for k in ("src", "dst", "etype"))
    E = len(src) // 2
    assert E == B // 2 and np.array_equal(src[:E], dst[E:]) and np.array_equal(dst[:E], src[E:])
    assert np.array_equal(et[E:], et[:E] + n_rel) and et[:E].max() < n_rel
    pos_set = {tuple(p) for p in pos}
    assert all((s, r, o) in pos_set for s, r, o in zip(src[:E], et[:E], dst[:E]))
    deg = np.bincount(dst, minlength=sm.n)
    assert deg[n:].sum() == 0 and max(src.max(), dst.max()) < n
    assert np.allclose(a["norm"].cpu().numpy().reshape(-1), 1.0 / deg[dst])
    b = draws[1]
    assert not np.array_equal(smp, b["samples"].cpu().numpy()) and not np.array_equal(src, b["src"].cpu().numpy())
    assert len({int(d["n_valid"]) for d in draws}) > 1


# ---------------------------------------------------------------------------------------------------------------
# a padded step computes what the unpadded step computes
# ---------------------------------------------------------------------------------------------------------------
def _layers(model):
    enc = model.encoder
    return [enc.rconv_layer_1, enc.rconv_layer_2] if isinstance(enc, K.KGVAE) else list(enc.layers[1:])


def _run_step(model, t, n_rows, n_valid, eps, masks):
    """forward + loss + backward on the first ``n_rows`` rows of the sample ``t``; returns outputs and gradients."""
    g = K.Graph.from_device_edges(n_rows, t["src"], t["dst"])
    g.n_valid = n_valid
    outs = []
    hooks = [layer.register_forward_hook(lambda m, i, o: outs.append(o.detach().clone())) for layer in _layers(model)]
    for layer, m in zip(_layers(model), masks):
        layer.dropout_mask = m[:n_rows]
    enc = model.encoder
    if isinstance(enc, K.KGVAE):
        enc.preset_eps = eps[:n_rows]
    model.zero_grad(set_to_none=True)
    try:
        embed = model(g, t["node_id"][:n_rows], t["etype"], t["norm"])
        embed.retain_grad()
        loss, pred, kl, _ = model.get_loss(g, embed, t["samples"], t["labels"])
        loss.backward()
    finally:
        for hk in hooks:
            hk.remove()
    res = {"loss": loss, "pred": pred, "kl": kl, "z": embed.detach(), "dz": embed.grad, "h": outs}
    if isinstance(enc, K.KGVAE):
        res["flow_log_prob"] = enc.flow_log_prob
        with torch.no_grad():
            trip = K.ops.as_i32(t["samples"])
            res["reg"] = K.ops.LossHeadFn.apply(embed, enc.z_mean, enc.z_sigma, enc.z_pre, model.w_relation, trip,
                                                t["labels"], model._flow_shift(), model.reg_param, model.kl_param,
                                                n_valid)[2]
    else:
        with torch.no_grad():
            res["reg"] = model.regularization_loss(embed, n_valid)
    res["grads"] = {name: p.grad.detach().clone() for name, p in model.named_parameters() if p.grad is not None}
    model.release_graph()
    return res


SHAPES = {"toy": dict(data="toy", h=40, bases=8, k=4, B=600),
          "FB15k-237": dict(data="FB15k-237", h=500, bases=100, k=10, B=20000)}


@pytest.mark.parametrize("shape", ["toy", "FB15k-237"])
@pytest.mark.parametrize("cfg", [(K.KGVAE, 0, 0.0), (K.KGVAE, 0, 1e-3), (K.KGVAE, 3, 0.0), (K.KGVAE, 3, 1e-3),
                                 (K.RGCN, 0, 0.0)], ids=["vae", "vae-kl", "flows", "flows-kl", "rgcn"])
def test_padded_step_equals_the_unpadded_step(shape, cfg):
    """One sample, two eager steps with the same eps and dropout masks on rows [0, n): on the padded node set
    (Graph.n_valid set) and on its first n rows.  Losses, layer outputs and every parameter gradient agree; the
    gradient reaching the padding rows of z is exactly zero."""
    model_class, n_flows, kl = cfg
    s = SHAPES[shape]
    data = K.datasets.synthetic_kg(s["data"], seed=0)
    h = s["h"]
    torch.manual_seed(0)
    model = K.LinkPredict(model_class, data.num_nodes, h, data.num_rels, num_bases=s["bases"],
                          num_hidden_layers=2, dropout=0.2, use_cuda=True, reg_param=0.01, kl_param=kl,
                          k=s["k"], n_flows=n_flows).to(DEV).train()
    sm = K.utils.SampledDeviceSampler(torch.from_numpy(data.train).to(DEV), s["B"], 0.5, data.num_rels, 10)
    t = sm.sample()
    cap, n = sm.n, int(t["n_valid"])
    assert n < cap
    widths = [h, 2 * h] if model_class is K.KGVAE else [h, h]
    masks = [(torch.rand(cap, w, device=DEV) < 0.8).float() / 0.8 for w in widths]
    eps = torch.randn(cap, h, device=DEV)
    pad = _run_step(model, t, cap, t["n_valid"], eps, masks)
    ref = _run_step(model, t, n, None, eps, masks)

    terms = ["loss", "pred", "kl", "reg"] + (["flow_log_prob"] if n_flows else [])
    for key in terms:
        assert rel_err(pad[key].reshape(()), ref[key].reshape(())) <= 1e-5, key
    for i, (a, b) in enumerate(zip(pad["h"], ref["h"])):
        assert rel_err(a[:n], b) <= 1e-5, f"h{i + 1}"
    assert rel_err(pad["z"][:n], ref["z"]) <= 1e-5
    assert bool((pad["dz"][n:] == 0).all())
    assert set(pad["grads"]) == set(ref["grads"])
    for name, gr in ref["grads"].items():
        assert rel_err(pad["grads"][name], gr) <= RTOL, name


# ---------------------------------------------------------------------------------------------------------------
# MMD on a padded node set
# ---------------------------------------------------------------------------------------------------------------
def test_mmd_draws_distinct_valid_rows():
    torch.manual_seed(0)
    n_rel, h, k = 7, 40, 10
    train = _toy_train(n_rel=n_rel)
    model = K.LinkPredict(K.KGVAE, 500, h, n_rel, num_bases=8, dropout=0.2, use_cuda=True, reg_param=0.01,
                          kl_param=1e-3, mmd_param=1.0, k=k, n_flows=1).to(DEV)
    sm = K.utils.SampledDeviceSampler(torch.from_numpy(train).to(DEV), 600, 0.5, n_rel, 4)
    t = sm.sample()
    nv = t["n_valid"]
    g = K.Graph.from_device_edges(sm.n, t["src"], t["dst"])
    g.n_valid = nv
    enc = model.encoder
    with torch.no_grad():
        z = model(g, t["node_id"], t["etype"], t["norm"])
        torch.manual_seed(5)
        mmd = enc.get_mmd(z, nv)
        rows = enc.mmd_rows.cpu().numpy()
        assert len(rows) == 200 and len(np.unique(rows)) == 200 and rows.max() < int(nv)
        torch.manual_seed(5)
        m_mix, s_mix = K.utils.gaussian_parameters(enc.z_pre, dim=1)
        z_pri = K.utils.sample_gaussian(m_mix, s_mix, repeat=200 // k)
        for flow in enc.nf:
            z_pri, _ = flow.forward(z_pri)
        z_post = z[torch.from_numpy(rows).to(DEV)]
        ck = enc.compute_kernel
        ref = ck(z_pri, z_pri).mean() + ck(z_post, z_post).mean() - 2 * ck(z_pri, z_post).mean()
    assert rel_err(mmd, ref) <= 1e-5
    # fewer than 200 valid rows: no value (the unpadded path raises through random.sample)
    with torch.no_grad():
        assert bool(torch.isnan(enc.get_mmd(z, torch.tensor([150], dtype=torch.int32, device=DEV))))
    with pytest.raises(ValueError, match="200"):
        enc.get_mmd(z[:150], torch.tensor([150], dtype=torch.int32, device=DEV))
    model.release_graph()

    opt = torch.optim.Adam(model.parameters(), lr=1e-3, fused=True, capturable=True)
    cap = K.link_predict.CapturedTrainStep(model, opt, None, sm.n, warmup=1, sampler=sm)
    mmds = []
    for _ in range(3):
        cap.step()
        mmds.append(float(cap.mmd.detach()))
    assert all(np.isfinite(mmds)) and len(set(mmds)) > 1
    cap.close()


# ---------------------------------------------------------------------------------------------------------------
# replay == eager
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_flows", [0, 1])
def test_captured_sampled_step_replays_the_eager_step(n_flows):
    """CapturedTrainStep(sampler=SampledDeviceSampler(...)) leaves the model where the same eager iterations - same
    seeds, so the same edge samples, negatives, splits, noise and dropout - leave it."""
    n_rel = 7
    train = torch.from_numpy(_toy_train(n_rel=n_rel)).to(DEV)
    torch.manual_seed(0)
    base = K.LinkPredict(K.KGVAE, 500, 40, n_rel, num_bases=8, dropout=0.2, use_cuda=True, reg_param=0.01,
                         kl_param=1e-3, k=4, n_flows=n_flows).to(DEV)
    sm = K.utils.SampledDeviceSampler(train, 600, 0.5, n_rel, 4)

    def eager_run():
        m = copy.deepcopy(base).train()
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, fused=True, capturable=True)
        bk = m.grad_buckets()
        losses, batches = [], []
        for i in range(3):
            torch.manual_seed(100 + i)
            t = sm.sample()
            batches.append(t["samples"].clone())
            g = K.Graph.from_device_edges(sm.n, t["src"], t["dst"])
            g.n_valid = t["n_valid"]
            bk.zero()
            emb = m(g, t["node_id"], t["etype"], t["norm"])
            loss = m.get_loss(g, emb, t["samples"], t["labels"])[0]
            loss.backward()
            bk.finish()
            bk.clip_(1.0)
            opt.step()
            losses.append(float(loss))
        m.release_graph()
        return m, losses, batches

    def captured_run():
        m = copy.deepcopy(base).train()
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, fused=True, capturable=True)
        torch.manual_seed(100)
        cap = K.link_predict.CapturedTrainStep(m, opt, None, sm.n, warmup=1, sampler=sm)   # warm-up = step 0
        assert cap.launches_per_step > 10
        losses = []
        for i in (1, 2):
            torch.manual_seed(100 + i)
            losses.append(float(cap.step()))
        cap.close()
        return m, losses

    m_e, l_e, batches = eager_run()
    m_c, l_c = captured_run()
    assert not torch.equal(batches[1], batches[2])
    assert np.allclose(l_e[1:], l_c, rtol=1e-5), (l_e, l_c)
    for (name, p), q in zip(m_e.named_parameters(), m_c.parameters()):
        err = float((p - q).abs().max() / p.abs().max().clamp(min=1e-12))
        assert err < 1e-3, (name, err)


# ---------------------------------------------------------------------------------------------------------------
# the driver
# ---------------------------------------------------------------------------------------------------------------
def _args(tmp_path, *extra):
    argv = ["-d", "toy", "--gpu", "0", "--n-hidden", "40", "--n-bases", "8", "--graph-batch-size", "600",
            "--negative-sample", "4", "--n-epochs", "4", "--evaluate-every", "2", "--eval-batch-size", "64",
            "--mog-k", "4", "--n-flows", "1", "--kl-param", "1e-3",
            "--model-state-file", os.path.join(str(tmp_path), "model_state.pth"), *extra]
    return K.link_predict.build_parser().parse_args(argv)


def test_driver_capture_step_with_the_device_sampler(tmp_path, capsys):
    """--capture-step --device-sampler with --graph-batch-size below the training set: every iteration - edge sample
    included - is one replay; validation, checkpoints and the printed line are the eager loop's."""
    np.random.seed(0)
    torch.manual_seed(0)
    args = _args(tmp_path, "--capture-step", "--device-sampler", "--n-flows", "0", "--n-epochs", "16",
                 "--evaluate-every", "8", "--lr", "1e-2")
    best = K.link_predict.main(args)
    out = capsys.readouterr().out
    assert "Epoch 0002" in out and "Epoch 0016" in out and "start eval" in out and "training done" in out
    losses = [float(line.split("Loss")[1].split("|")[0]) for line in out.splitlines() if line.startswith("Epoch")]
    assert len(losses) == 15 and all(np.isfinite(losses))
    assert np.mean(losses[-3:]) < np.mean(losses[:3])
    assert 0.0 < best <= 1.0
    assert torch.load(args.model_state_file, map_location="cpu")["epoch"] in (8, 16)


def test_driver_capture_step_with_the_device_sampler_readme_terms(tmp_path, capsys):
    """The README run's loss terms (--n-flows 3 --mmd-param 1 --mog-k 10) in the captured sampled iteration."""
    np.random.seed(2)
    torch.manual_seed(2)
    best = K.link_predict.main(_args(tmp_path, "--capture-step", "--device-sampler", "--n-flows", "3",
                                     "--mmd-param", "1", "--mog-k", "10", "--n-epochs", "4"))
    out = capsys.readouterr().out
    lines = [line for line in out.splitlines() if line.startswith("Epoch")]
    assert "Epoch 0004" in out and len(lines) == 3 and 0.0 < best <= 1.0
    mmd = [float(line.split("mmd")[1]) for line in lines]
    assert all(np.isfinite(mmd)) and max(mmd) > 0
