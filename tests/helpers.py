"""Shared helpers for the parity tests (oracle side only - never imported by the package)."""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import kgvae_oracle as O  # noqa: E402

RTOL = 1e-4   # north_star: embeddings, loss and scores within 1e-4 relative in fp32


def rel_err(a, b):
    """max |a-b| / max(|b|_max, tiny): error relative to the tensor's scale."""
    a, b = (t.detach().cpu() if isinstance(t, torch.Tensor) else torch.as_tensor(np.asarray(t)) for t in (a, b))
    a, b = a.to(torch.float64), b.to(torch.float64)
    if a.numel() == 1 and b.numel() == 1:      # the reference mixes [] and [1] scalars
        a, b = a.reshape(()), b.reshape(())
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.numel() == 0:
        return 0.0
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def assert_close(a, b, rtol=RTOL, what=""):
    e = rel_err(a, b)
    assert e <= rtol, f"{what}: relative error {e:.3e} > {rtol:.1e}"


def kernels_run(fn):
    """Names of the CUDA kernels ``fn`` launches (torch.profiler), joined by " | "."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " | ".join(e.name for e in prof.events())


def at_golden_rows(gv, key, t):
    """The rows of ``t`` that golden case ``gv`` keeps of output ``key``: all of them, unless the case stores a
    seeded sample of the rows (``rows/<key>``) to stay small."""
    rows = gv.get("rows/" + key)
    return t if rows is None else t[torch.as_tensor(rows)]


# A golden case too large to store whole (kgvae_small_noflow) leaves out the random inputs of its reference run and
# keeps the SHA-256 of them instead; they are drawn again here from the case's seed, in the order the run drew them:
# parameter initialisation (embedding, the two bdd layers, MoG prior, relation matrix), bias noise, eps, dropout
# masks, then the evaluation pass's eps.
REDRAWN = ["param/encoder.input_layer.embedding.weight", "param/encoder.rconv_layer_1.weight",
           "param/encoder.rconv_layer_1.loop_weight", "param/encoder.rconv_layer_2.weight",
           "param/encoder.rconv_layer_2.loop_weight", "param/encoder.z_pre", "param/w_relation",
           "param/encoder.rconv_layer_1.h_bias", "param/encoder.rconv_layer_2.h_bias",
           "eps", "mask1", "mask2", "eval_eps"]


def inputs_sha256(arrays):
    h = hashlib.sha256()
    for key in REDRAWN:
        h.update(np.ascontiguousarray(arrays[key]).tobytes())
    return h.hexdigest()


def redraw_inputs(gv):
    """REDRAWN of a case without IAF flows, checked against the digest the case recorded."""
    n_ent, n_rel, h, bases, k, n_flows, _ = (int(x) for x in gv["cfg"])
    assert n_flows == 0
    keep = 1.0 - float(gv["cfg_f"][2])
    n, si = len(gv["node_id"]), h // bases
    g = torch.Generator().manual_seed(int(gv["seed"]))
    xavier = lambda *shape: torch.nn.init.xavier_uniform_(torch.empty(*shape), torch.nn.init.calculate_gain("relu"),
                                                          generator=g)
    drawn = [torch.empty(n_ent, h).normal_(generator=g),
             xavier(2 * n_rel, bases * si * si), xavier(h, h), xavier(2 * n_rel, bases * si * 2 * si), xavier(h, 2 * h),
             torch.randn(1, 2 * k, h, generator=g) / np.sqrt(k * h)]
    drawn += [xavier(n_rel, h), torch.zeros(h).normal_(0, 0.1, generator=g), torch.zeros(2 * h).normal_(0, 0.1, generator=g),
              torch.randn(n, h, generator=g)]
    drawn += [(torch.rand(n, w, generator=g) < keep).float() / keep for w in (h, 2 * h)]
    drawn.append(torch.randn(n_ent, h, generator=g))
    out = {key: t.numpy() for key, t in zip(REDRAWN, drawn)}
    assert inputs_sha256(out) == str(gv["inputs_sha256"]), \
        "torch's random stream no longer reproduces the inputs this golden case was recorded with"
    return out


def golden_params(gv, requires_grad=False):
    p = {}
    for key, val in gv.items():
        if key.startswith("param/") and not key.endswith(".mask") and not key.endswith("pi"):
            t = torch.from_numpy(val.copy())
            if requires_grad:
                t.requires_grad_(True)
            p[key[len("param/"):]] = t
    return p


def golden_graph(gv, prefix="g_", etype_key="edge_type", norm_key="node_norm", n=None):
    dst = gv[prefix + "dst"].astype(np.int64)
    norm = gv[norm_key].astype(np.float32)
    return {"num_nodes": int(len(norm) if n is None else n),
            "src": gv[prefix + "src"].astype(np.int64), "dst": dst,
            "etype": gv[etype_key].astype(np.int64), "norm": norm,
            "edge_norm": norm[dst].reshape(-1, 1)}


def made_relu_patterns(z, weights, biases, masks, degrees, against=None):
    """The plain oracle MADE forward (O.made_forward without a pattern), replayed pass by pass to expose the hidden
    layers.  Returns (x, patterns, flips): ``patterns[p][l]`` is ``pre-activation > 0`` of hidden layer l in pass p,
    the nesting ``O.made_forward(relu_patterns=...)`` takes.  ``against``: another implementation's patterns, same
    nesting (a pass may give one [1, h] row for all rows, as the first pass does on the GPU); then ``flips`` is
    (number of units whose sign differs, largest |pre-activation| among them relative to its layer's largest)."""
    import torch.nn.functional as F
    x = torch.zeros_like(z)
    patterns, n_flip, worst = [], 0, 0.0
    for p, idx in enumerate(degrees):
        h, layer = x, []
        for i in range(len(weights)):
            h = F.linear(h, masks[i] * weights[i], biases[i])
            if i + 1 < len(weights):
                layer.append(h > 0)
                if against is not None:
                    other = against[p][i].to(h.device)
                    pre = h[:other.shape[0]]
                    diff = other != (pre > 0)
                    if bool(diff.any()):
                        n_flip += int(diff.sum())
                        worst = max(worst, float(pre.abs()[diff].max() / pre.abs().max()))
                h = torch.relu(h)
        mu, alpha = torch.chunk(h, 2, dim=1)
        x = x.clone()
        x[:, idx] = z[:, idx] * torch.exp(alpha[:, idx] + mu[:, idx])
        patterns.append(layer)
    return x, patterns, (n_flip, worst)


def oracle_train_step(gv, requires_grad=True):
    """Run the oracle port on a golden case's inputs; returns (params, enc, loss dict)."""
    n_ent, n_rel, h, bases, k, n_flows, neg = (int(x) for x in gv["cfg"])
    reg_param, kl_param, dropout = (float(x) for x in gv["cfg_f"])
    params = golden_params(gv, requires_grad)
    graph = golden_graph(gv)
    enc = O.kgvae_encode(params, graph, gv["node_id"], torch.from_numpy(gv["eps"]), bases, n_flows,
                         (torch.from_numpy(gv["mask1"]), torch.from_numpy(gv["mask2"])))
    out = O.kgvae_loss(params, enc, gv["samples"], gv["labels"], reg_param, kl_param, n_flows)
    return params, enc, out
