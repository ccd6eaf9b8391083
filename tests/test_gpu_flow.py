"""The IAF flow (flow_network.MADE + PermuteLayer; reference kgvae/flow_network.py:37-112, kgvae/model.py:115-123)
against plain float64 references on the CPU, at the widths the benchmark runs.

* Kernel level: the flow's element update (kg_iaf_update_fwd / _bwd) against ``x[:, idx] = z[:, idx] * exp(alpha +
  mu)`` through autograd's index_put, the column reversal against ``flip``, the M <= 8 GEMM kernel and the SIMT tile
  kernel at the shapes the flow hands them (one-row passes, K = 1 weight gradients, row slices of wider buffers),
  and the dispatch boundaries between the three GEMM kernels.
* Module level: ``MADE(D, D, n_hidden)`` at D = 500 and at smoke()'s D = 40, at row counts that select each GEMM
  path, forward, inverse and every gradient.
* Model level: one train step of the benchmarked flow configuration (WN18 shape, h = 500, 3 flows) and one of
  smoke()'s configuration, compared stage by stage so that a failure names the stage.
* Bitwise repeatability of every kernel on the path from z_mean to the flowed z (none of them uses atomics).

At tens of millions of hidden units a few MADE pre-activations lie within rounding error of 0 and land on different
sides of the ReLU in fp32 and fp64.  ReLU has no derivative there, so gradient comparisons hand the GPU's ReLU
pattern to the oracle (``made_relu_patterns``) and bound how many units that concerns and how close to 0 they are.
"""
import types

import numpy as np
import pytest
import torch

from helpers import O, RTOL, assert_close, kernels_run, made_relu_patterns, rel_err

import gcn_vae_b200 as K
from gcn_vae_b200 import _lib as L
from gcn_vae_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

FLIP_FRACTION = 1e-5     # at most this share of the hidden units may sit on the other side of the ReLU ...
FLIP_MAGNITUDE = 1e-4    # ... and only within this distance of 0, relative to the layer's largest pre-activation


def _assert_elementwise(got, want, tol, what, scale=None):
    """|got - want| <= tol * scale element by element (scale: |want| unless given)."""
    got = got.detach().cpu().double()
    scale = want.abs() if scale is None else scale
    err = (got - want).abs()
    bad = err > tol * scale
    if bool(bad.any()):
        worst = float((err / scale.clamp_min(1e-300)).max())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements off by more than {tol:.0e}, "
                             f"worst {worst:.2e}")


def _poison_workspaces(monkeypatch):
    """ops takes its scratch (GEMM workspaces, prepared operands) from L.workspace: hand out 0xFF bytes (NaN)."""
    def poisoned(nbytes, device):
        return torch.full((max(int(nbytes), 16),), 0xFF, dtype=torch.uint8, device=device)
    monkeypatch.setattr(L, "workspace", poisoned)


def _nan_buffer(*shape):
    n = int(np.prod(shape))
    return torch.full((4 * n,), 0xFF, dtype=torch.uint8, device=DEV).view(torch.float32).view(*shape)


# ------------------------------------------------------------------------------------------ IAF element update
def _index_lists(d):
    """Index lists of one pass: every column once (first and last pass); the reference's middle passes,
    arange(D) % (D - 1) (column 0 twice, the last column not at all); an arbitrary list with multiplicities 0-3."""
    g = torch.Generator().manual_seed(d)
    lists = {"all": torch.arange(d)}
    if d > 1:
        lists["middle"] = torch.arange(d) % (d - 1)
    mult = torch.randint(0, 4, (d,), generator=g)
    if d > 1:
        mult[0], mult[-1] = 3, 0
    idx = torch.repeat_interleave(torch.arange(d), mult)
    lists["arbitrary"] = idx[torch.randperm(len(idx), generator=g)]
    return lists


def _iaf_reference(z, net, x_old, idx, gx, gl):
    """fp64 restatement of flow_network.py:93-96; autograd's index_put hands a column listed twice its gradient
    twice, as in the reference."""
    z, net, x_old = (t.double().requires_grad_(True) for t in (z, net, x_old))
    mu, alpha = net.chunk(2, dim=1)
    x = x_old.clone()
    x[:, idx] = z[:, idx] * torch.exp(alpha[:, idx] + mu[:, idx])
    log_det = alpha.sum(-1)
    loss = (x * gx.double()).sum()
    if gl is not None:
        loss = loss + (log_det * gl.double()).sum()
    loss.backward()
    return x.detach(), log_det.detach(), z.grad, net.grad, x_old.grad


@pytest.mark.parametrize("n", [1, 7, 4097])
@pytest.mark.parametrize("d", [1, 2, 31, 33, 40, 500, 1000])
def test_iaf_update_against_index_put(n, d):
    g = torch.Generator().manual_seed(1000 * n + d)
    z, x_old = torch.randn(n, d, generator=g), torch.randn(n, d, generator=g)
    # alpha and mu on a 2^-12 grid in [-10, 10]: alpha + mu (up to +-20) is exact in fp32, so the comparison sees
    # the kernel's exp and products only, not the rounding of the sum the reference's fp32 code shares
    grid = lambda: torch.round((torch.rand(n, d, generator=g) * 20 - 10) * 4096) / 4096
    net = torch.cat([grid(), grid()], dim=1)
    gx, gl = torch.randn(n, d, generator=g), torch.randn(n, generator=g)
    zd, netd, xd, gxd, gld = (t.to(DEV) for t in (z, net, x_old, gx, gl))
    alpha_abs = net[:, d:].double().abs().sum(-1)
    for name, idx in _index_lists(d).items():
        what = f"n={n} d={d} {name}"
        mult = torch.bincount(idx, minlength=d).to(torch.int32)
        keep = mult == 0
        multd = mult.to(DEV)
        x_want, ld_want, dz_want, dnet_want, dxo_want = _iaf_reference(z, net, x_old, idx, gx, gl)

        # forward, with and without the log-det
        for want_ld in (True, False):
            x_new, log_det = ops.IafUpdateFn.apply(zd, netd, xd, multd, want_ld)
            _assert_elementwise(x_new, x_want, 1e-6, f"{what}: x")
            assert torch.equal(x_new[:, keep.to(DEV)], xd[:, keep.to(DEV)]), f"{what}: multiplicity-0 columns"
            if want_ld:
                _assert_elementwise(log_det, ld_want, 1e-6, f"{what}: log_det", scale=alpha_abs)
            else:
                assert log_det is None

        # backward through autograd: both upstream gradients
        leaves = [t.clone().requires_grad_(True) for t in (zd, netd, xd)]
        x_new, log_det = ops.IafUpdateFn.apply(*leaves, multd, True)
        ((x_new * gxd).sum() + (log_det * gld).sum()).backward()
        _check_iaf_grads([t.grad for t in leaves], (dz_want, dnet_want, dxo_want), gx, gl, keep, d, what)

        # the kernel with dlog_det = NULL, and with no gradient for x
        ctx = types.SimpleNamespace(saved_tensors=(zd, netd, multd))
        got = ops.IafUpdateFn.backward(ctx, gxd, None)[:3]
        _check_iaf_grads(got, _iaf_reference(z, net, x_old, idx, gx, None)[2:], gx, None, keep, d, what + " no dlog_det")
        got = ops.IafUpdateFn.backward(ctx, None, gld)[:3]
        _check_iaf_grads(got, _iaf_reference(z, net, x_old, idx, torch.zeros_like(gx), gl)[2:],
                         torch.zeros_like(gx), gl, keep, d, what + " no dx")


def _check_iaf_grads(got, want, gx, gl, keep, d, what):
    dz, dnet, dxo = got
    dz_want, dnet_want, dxo_want = want
    _assert_elementwise(dz, dz_want, 1e-6, f"{what}: dz")
    _assert_elementwise(dnet[:, :d], dnet_want[:, :d], 1e-6, f"{what}: dmu")
    # d alpha = d mu + dlog_det: a sum, so its scale is the sum of the terms' magnitudes
    scale = dnet_want[:, :d].abs() + (0 if gl is None else gl.double().abs().view(-1, 1))
    _assert_elementwise(dnet[:, d:], dnet_want[:, d:], 1e-6, f"{what}: dalpha", scale=scale)
    assert torch.equal(dxo.cpu(), torch.where(keep, gx, torch.zeros_like(gx))), f"{what}: dx_old"
    assert torch.equal(dxo_want.float(), torch.where(keep, gx, torch.zeros_like(gx)))


@pytest.mark.parametrize("d", [1, 2, 33, 500])
def test_reverse_columns_is_flip(d):
    g = torch.Generator().manual_seed(d)
    for n in (1, 7, 4097):
        x = torch.randn(n, d, generator=g)
        gy = torch.randn(n, d, generator=g)
        xd = x.to(DEV).requires_grad_(True)
        y = ops.ReverseColumnsFn.apply(xd)
        y.backward(gy.to(DEV))
        assert torch.equal(y.detach().cpu(), torch.flip(x, [1])), (n, d)
        assert torch.equal(xd.grad.cpu(), torch.flip(gy, [1])), (n, d)


# ------------------------------------------------------------------------------------------ GEMM kernels
def _gemm_case(M, N, K, ta, tb, pad, flags, gen):
    """kg_gemm_f32 called directly on row slices: A, B and C live in buffers ``pad`` columns wider than the operand
    (lda, ldb, ldc > width when pad > 0), C has one guard row below it.  flags: bias, addend, relu, mask,
    accumulate.  Checks the product against fp64 (2e-5 of the tensor's scale) and that every byte of C's buffer
    outside the M x N window is unchanged."""
    bias_on, add_on, relu, mask_on, acc = flags
    a_rows, a_cols = (K, M) if ta else (M, K)
    b_rows, b_cols = (N, K) if tb else (K, N)
    a_buf = torch.randn(a_rows, a_cols + pad, device=DEV, generator=gen)
    b_buf = torch.randn(b_rows, b_cols + pad, device=DEV, generator=gen)
    ldc = N + pad
    c_buf = torch.randn(M + 1, ldc, device=DEV, generator=gen)
    bias = torch.randn(N, device=DEV, generator=gen) if bias_on else None
    add = torch.randn(M, ldc, device=DEV, generator=gen) if add_on else None      # addend and mask share ldc
    mask = (torch.rand(M, ldc, device=DEV, generator=gen) < 0.8).float() / 0.8 if mask_on else None
    c_before = c_buf.clone()
    L.call("kg_gemm_f32", a_buf.data_ptr(), a_cols + pad, int(ta), b_buf.data_ptr(), b_cols + pad, int(tb),
           c_buf.data_ptr(), ldc, M, N, K, None if bias is None else bias.data_ptr(),
           None if add is None else add.data_ptr(), int(relu), None if mask is None else mask.data_ptr(), int(acc),
           None, 0, L.stream())
    A = a_buf[:, :a_cols].cpu().double()
    B = b_buf[:, :b_cols].cpu().double()
    want = (A.t() if ta else A) @ (B.t() if tb else B)
    if bias_on:
        want = want + bias.cpu().double()
    if add_on:
        want = want + add[:, :N].cpu().double()
    if relu:
        want = torch.relu(want)
    if mask_on:
        want = want * mask[:, :N].cpu().double()
    if acc:
        want = want + c_before[:M, :N].cpu().double()
    what = f"gemm {M}x{N}x{K} ta={ta} tb={tb} pad={pad} flags={flags}"
    assert_close(c_buf[:M, :N], want, 2e-5, what)
    outside = torch.ones(M + 1, ldc, dtype=torch.bool, device=DEV)
    outside[:M, :N] = False
    assert torch.equal(c_buf[outside], c_before[outside]), f"{what}: wrote outside the ldc window"


ORIENTATIONS = [(0, 0), (0, 1), (1, 0), (1, 1)]


@pytest.mark.parametrize("ta,tb", ORIENTATIONS)
@pytest.mark.parametrize("M", [1, 2, 3, 4, 5, 6, 7, 8])
def test_gemm_small_m_kernel(M, ta, tb):
    """M <= 8 and K >= 32: gemm_small_m_kernel (B k-contiguous: a warp per column; otherwise a lane per column and
    the CTA's eight warps splitting K).  Every K x N below, leading dimensions equal to and larger than the width,
    the five epilogue switches cycling through all 32 combinations over the cases."""
    gen = torch.Generator(device=DEV).manual_seed(100 * M + 10 * ta + tb)
    i = 0
    for K_ in (32, 33, 40, 500, 1000, 4097):
        for N in (1, 31, 33, 500, 1000):
            assert not ops.uses_tensor_cores(M, N, K_)
            bits = (7 * i + 3 * M + 5 * ta + 11 * tb) % 32
            flags = tuple(bool(bits >> b & 1) for b in range(5))
            _gemm_case(M, N, K_, ta, tb, 0 if (i + M) % 2 else 5, flags, gen)
            i += 1


@pytest.mark.parametrize("ta,tb", ORIENTATIONS)
@pytest.mark.parametrize("M,N,K", [(9, 500, 500), (9, 33, 4097), (8, 500, 31), (1, 1000, 31),   # next to M <= 8, K >= 32
                                   (500, 500, 1), (1000, 500, 1), (500, 1000, 7),               # K = 1: one-row pass dW
                                   (40, 40, 300)])                                              # split-K
def test_gemm_tile_kernel_flow_shapes(M, N, K, ta, tb):
    """The SIMT tile kernel at the flow's small-K shapes: the weight gradients of the one-row first pass (K = 1) and
    of smoke()'s MADE (40 x 40 over 300 rows, which takes split-K when there is no bias), and the shapes just past
    the M <= 8 kernel's rule.  Plain (split-K allowed) and with the whole epilogue, contiguous and as row slices."""
    assert not ops.uses_tensor_cores(M, N, K)
    gen = torch.Generator(device=DEV).manual_seed(M + N + K + 10 * ta + tb)
    for pad in (0, 3):
        _gemm_case(M, N, K, ta, tb, pad, (False,) * 5, gen)
        _gemm_case(M, N, K, ta, tb, pad, (True,) * 5, gen)
        _gemm_case(M, N, K, ta, tb, pad, (False, False, False, True, True), gen)     # masked accumulate


@pytest.mark.parametrize("M,N,K,path", [(64, 64, 1000, "tile"), (64, 64, 1024, "tc"), (63, 500, 500, "tile"),
                                        (64, 500, 500, "tc"), (8, 500, 32, "small_m"), (9, 500, 32, "tile"),
                                        (8, 500, 31, "tile"), (1, 1000, 500, "small_m")])
def test_gemm_dispatch_boundaries(M, N, K, path):
    """Shapes on either side of kg_gemm_f32_uses_tensor_cores (K >= 32, M, N >= 64, M N K >= 2^22) and of the
    M <= 8 rule: the kernel that runs is the one the rule names, and the result is right on both sides."""
    assert ops.uses_tensor_cores(M, N, K) == (path == "tc")
    kernel = {"tc": "gemm_tc_kernel", "tile": "gemm_kernel<", "small_m": "gemm_small_m_kernel"}
    g = torch.Generator().manual_seed(M * N + K)
    for ta, tb in ORIENTATIONS:
        a = torch.randn((K, M) if ta else (M, K), generator=g)
        b = torch.randn((N, K) if tb else (K, N), generator=g)
        bias = torch.randn(N, generator=g)
        out = torch.empty(M, N, device=DEV)
        ad, bd, biasd = a.to(DEV), b.to(DEV), bias.to(DEV)
        names = kernels_run(lambda: ops.gemm(ad, bd, out, trans_a=bool(ta), trans_b=bool(tb), bias=biasd, relu=True))
        for p, k in kernel.items():       # demangled or mangled (gemm_kernelILb1E...) names
            ran = k in names or k.replace("<", "I") in names
            assert ran == (p == path), f"{M}x{N}x{K}: expected the {path} kernel, ran: {names}"
        want = torch.relu((a.t() if ta else a).double() @ (b.t() if tb else b).double() + bias.double())
        assert_close(out, want, 2e-5, f"gemm {M}x{N}x{K} ta={ta} tb={tb}")


# ------------------------------------------------------------------------------------------ MADE module
class _ReluTap:
    """Forward hooks on a MADE's MaskedLinear layers: ``output > 0`` of every call with relu=True, in call order,
    grouped per pass as O.made_forward(relu_patterns=...) takes them."""

    def __init__(self, made):
        self.made, self.calls = made, []
        self.handles = [layer.register_forward_hook(self._hook, with_kwargs=True) for layer in made._linears()]

    def _hook(self, module, args, kwargs, out):
        if kwargs.get("relu"):
            self.calls.append(out.detach() > 0)

    def patterns(self):
        per_pass = len(self.made._linears()) - 1
        assert len(self.calls) == per_pass * len(self.made.m)
        return [[t.cpu() for t in self.calls[p:p + per_pass]] for p in range(0, len(self.calls), per_pass)]

    def remove(self):
        for h in self.handles:
            h.remove()


def _assert_flips_bounded(flips, n_units, what):
    n_flip, worst = flips
    assert n_flip <= max(8, FLIP_FRACTION * n_units), f"{what}: {n_flip} of {n_units} ReLU units differ in sign"
    assert worst < FLIP_MAGNITUDE, f"{what}: a ReLU unit {worst:.1e} of its layer's scale from 0 differs in sign"


@pytest.mark.parametrize("N", [1, 63, 64, 4097])
@pytest.mark.parametrize("D,n_hidden", [(500, 3), (500, 1), (40, 1)])
def test_made_against_oracle(D, n_hidden, N):
    """MADE(D, D, n_hidden) against O.made_forward / O.made_inverse.  At D = 500: N = 1 runs everything on the M <= 8
    kernel, N = 63 the SIMT forward with tensor-core weight gradients, N = 64 all tensor-core with one partial
    128-row tile, N = 4097 tensor-core with a ragged last tile.  (40, 1) is smoke()'s flow."""
    torch.manual_seed(10 * D + n_hidden)
    made = K.MADE(D, D, n_hidden).to(DEV)
    g = torch.Generator().manual_seed(N)
    z, gx, gl = torch.randn(N, D, generator=g), torch.randn(N, D, generator=g), torch.randn(N, generator=g)
    zd = z.to(DEV).requires_grad_(True)
    tap = _ReluTap(made)
    x, log_det = made(zd)
    ((x * gx.to(DEV)).sum() + (log_det * gl.to(DEV)).sum()).backward()
    tap.remove()
    pats = tap.patterns()
    assert tuple(pats[0][0].shape) == (1, D)             # the first pass ran one row

    linears = made._linears()
    ws = [l.weight.detach().cpu().double().requires_grad_(True) for l in linears]
    bs = [l.bias.detach().cpu().double().requires_grad_(True) for l in linears]
    masks, degs = O.made_masks(D, D, n_hidden), O.made_degrees(D, D, n_hidden)
    z64 = z.double().requires_grad_(True)
    with torch.no_grad():
        x_plain, _, flips = made_relu_patterns(z64, ws, bs, masks, degs, against=pats)
    _assert_flips_bounded(flips, len(degs) * (n_hidden + 1) * N * D, f"MADE({D}, {n_hidden}) N={N}")
    xr, ldr = O.made_forward(z64, ws, bs, masks, degs, pats)
    ((xr * gx.double()).sum() + (ldr * gl.double()).sum()).backward()
    what = f"MADE({D}, {n_hidden}) N={N}"
    assert_close(x, x_plain, RTOL, f"{what}: x")
    assert_close(x, xr, RTOL, f"{what}: x (GPU ReLU pattern)")
    assert_close(log_det, ldr, RTOL, f"{what}: log_det")
    assert_close(zd.grad, z64.grad, RTOL, f"{what}: dz")
    for i, layer in enumerate(linears):
        assert_close(layer.weight.grad, ws[i].grad, RTOL, f"{what}: net.{2 * i}.weight grad")
        assert_close(layer.bias.grad, bs[i].grad, RTOL, f"{what}: net.{2 * i}.bias grad")

    with torch.no_grad():
        zi, ldi = made.inverse(x.detach())
        zi_r, ldi_r = O.made_inverse(x.detach().cpu().double(), ws, bs, masks)
    assert_close(zi, zi_r, RTOL, f"{what}: inverse z")
    assert_close(ldi, ldi_r, RTOL, f"{what}: inverse log_det")


# ------------------------------------------------------------------------------------------ one train step
def _flow_step_errors(train, n_ent, n_rel, h, bases, k, n_flows, kl_param, sample_size, neg):
    """One train step of LinkPredict(KGVAE) with n_flows IAF blocks on a sampled batch (the order of random draws is
    smoke()'s), and the same step in the fp64 oracle.  Returns ({stage: relative error}, {stage: flip count})."""
    torch.manual_seed(0)
    model = K.LinkPredict(K.KGVAE, n_ent, h, n_rel, num_bases=bases, dropout=0.2, use_cuda=True, reg_param=0.01,
                          kl_param=kl_param, k=k, n_flows=n_flows).to(DEV)
    np.random.seed(0)
    g, node_id, edge_type, node_norm, samples, labels = K.utils.generate_sampled_graph_and_labels(
        train, sample_size, 0.5, n_rel, None, None, neg, "uniform")
    n = len(node_id)
    eps = torch.randn(n, h)
    m1 = (torch.rand(n, h) < 0.8).float() / 0.8
    m2 = (torch.rand(n, 2 * h) < 0.8).float() / 0.8
    enc = model.encoder
    enc.preset_eps, enc.rconv_layer_1.dropout_mask, enc.rconv_layer_2.dropout_mask = eps.to(DEV), m1.to(DEV), m2.to(DEV)
    edge_norm = K.node_norm_to_edge_norm(g, torch.from_numpy(node_norm).view(-1, 1)).to(DEV)

    taps = {}
    put = lambda key: (lambda m, i, o: taps.__setitem__(key, o.detach().cpu()))
    hooks = [enc.rconv_layer_1.register_forward_hook(put("h1")), enc.rconv_layer_2.register_forward_hook(put("h2"))]
    mades = [m for m in enc.nf if isinstance(m, K.MADE)]
    perms = [m for m in enc.nf if isinstance(m, K.PermuteLayer)]
    # KGVAE.forward calls flow.forward(z) directly, which bypasses module hooks: the flow blocks are tapped by
    # wrapping their forward on the instance instead
    def tap_flow(module, key, value_of):
        inner = module.forward

        def forward(x):
            out = inner(x)
            taps[key] = value_of(x, out).detach().cpu()
            return out
        module.forward = forward
    tap_flow(mades[0], "z0", lambda x, out: x)
    for f, p in enumerate(perms):
        tap_flow(p, f"z{f + 1}", lambda x, out: out[0])
    relu_taps = [_ReluTap(m) for m in mades]
    model.train()
    embed = model(g, torch.from_numpy(node_id).view(-1, 1).to(DEV), torch.from_numpy(edge_type).to(DEV), edge_norm)
    loss, pred, kl, _ = model.get_loss(g, embed, torch.from_numpy(samples).to(DEV), torch.from_numpy(labels).to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    for hk in hooks:
        hk.remove()
    for m in [mades[0]] + perms:
        del m.forward
    for t in relu_taps:
        t.remove()
    flow_pats = [t.patterns() for t in relu_taps]

    params = {key: val.detach().cpu().double().requires_grad_(True) for key, val in model.state_dict().items()
              if val.dtype.is_floating_point and not key.endswith(("mask", "pi"))}
    graph = {"num_nodes": n, "src": g._src, "dst": g._dst, "etype": edge_type, "norm": node_norm,
             "edge_norm": node_norm[g._dst].reshape(-1, 1).astype(np.float64)}
    eps64, masks64 = eps.double(), (m1.double(), m2.double())
    labels64 = np.asarray(labels, dtype=np.float64)
    flips = {}
    with torch.no_grad():
        # the plain function, stage by stage: the encoder without the flow, then MADE + reverse per block
        plain = O.kgvae_encode(params, graph, node_id, eps64, bases, 0, masks64)
        stages = {key: plain[key] for key in ("h1", "h2", "z_mean", "z_sigma")}
        stages["z0"] = plain["z"]
        zc = plain["z"]
        masks, degs = O.made_masks(h, h, n_flows), O.made_degrees(h, h, n_flows)
        for f, (ws, bs) in enumerate(O.flow_params(params, n_flows)):
            zc, _, fl = made_relu_patterns(zc, ws, bs, masks, degs, against=flow_pats[f])
            _assert_flips_bounded(fl, len(degs) * (n_flows + 1) * n * h, f"MADE {f}")
            flips[f"MADE {f}"] = fl[0]
            zc = zc.flip(1)
            stages[f"z{f + 1}"] = zc
    l1_flip = ((plain["h1"] > 0) != (taps["h1"] > 0)) & (m1 > 0)
    flips["layer 1"] = int(l1_flip.sum())
    assert flips["layer 1"] <= max(8, FLIP_FRACTION * n * h), f"{flips['layer 1']} layer-1 ReLU units differ in sign"
    if flips["layer 1"]:
        assert float((plain["h1"] - taps["h1"]).abs()[l1_flip].max() / plain["h1"].abs().max()) < FLIP_MAGNITUDE

    ref_enc = O.kgvae_encode(params, graph, node_id, eps64, bases, n_flows, masks64,
                             relu_pattern=(taps["h1"] > 0) | (m1 == 0), made_relu_patterns=flow_pats)
    ref = O.kgvae_loss(params, ref_enc, samples, labels64, 0.01, kl_param, n_flows)
    ref["loss"].backward()

    errs = {key: rel_err(taps[key], want) for key, want in stages.items() if key in taps}
    errs["z_mean"] = rel_err(enc.z_mean, stages["z_mean"])
    errs["z_sigma"] = rel_err(enc.z_sigma, stages["z_sigma"])
    errs["z (GPU ReLU pattern)"] = rel_err(embed, ref_enc["z"])
    errs["log_det_sum"] = rel_err(enc.log_det_sum.reshape(-1), ref_enc["log_det_sum"])
    errs["flow_log_prob"] = rel_err(enc.flow_log_prob, ref_enc["flow_log_prob"])
    errs["loss"] = rel_err(loss, ref["loss"])
    errs["predict_loss"] = rel_err(pred, ref["predict_loss"])
    errs["kl"] = rel_err(kl, ref["kl"])
    n_grads = 0
    for name, p in model.named_parameters():
        if p.grad is not None:
            assert params[name].grad is not None, name
            errs[f"grad {name}"] = rel_err(p.grad, params[name].grad)
            n_grads += 1
    assert n_grads == 9 + 2 * n_flows * (n_flows + 2)
    assert all(f"z{f + 1}" in errs for f in range(n_flows)) and "z0" in errs
    return errs, flips


def _report(errs, flips, limit, title):
    lines = [f"{title}: ReLU units on the other side of 0: {flips}"]
    lines += [f"  {key:<48s} {val:.2e}{'   > limit' if val > limit else ''}" for key, val in errs.items()]
    print("\n".join(lines))
    bad = [key for key, val in errs.items() if not val <= limit]
    assert not bad, f"stages over {limit:.0e}: {bad}\n" + "\n".join(lines)


def test_wn18_flow_step_against_oracle():
    """bench.py configs[2] (wn18 shape, --n-flows 3) at the block shape: h = 500, 25 bases (20x20 then 20x40
    blocks), three MADE(500, 500, 3) blocks, kl_param 1e-3, on a sampled batch of about 2 900 nodes."""
    data = K.datasets.synthetic_kg("wn18", seed=0)
    errs, flips = _flow_step_errors(data.train, data.num_nodes, data.num_rels, 500, 25, 10, 3, 1e-3, 1500, 10)
    _report(errs, flips, RTOL, "wn18 flow step")


def test_smoke_configuration_step_against_oracle():
    """smoke()'s exact configuration (300 entities, h = 40, 8 blocks, one MADE(40, 40, 1)) at 5e-6: it normally
    agrees to ~1e-7, so a recurrence of the 8.6e-5 reading on z fails here and names the stage it came from."""
    data = K.datasets.synthetic_kg("toy", seed=3)
    data.train[:, [0, 2]] %= 300
    data.train[:, 1] %= 6
    errs, flips = _flow_step_errors(data.train, 300, 6, 40, 8, 4, 1, 1e-3, 600, 4)
    _report(errs, flips, 5e-6, "smoke configuration step")


# ------------------------------------------------------------------------------------------ bitwise gate
def _poison_allocator():
    """Refill the caching allocator's free blocks with 0xFF bytes, so that torch.empty inside the ops hands out NaN."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    blocks = [torch.full((256 << 20,), 0xFF, dtype=torch.uint8, device=DEV)]
    blocks += [torch.full((1 << 20,), 0xFF, dtype=torch.uint8, device=DEV) for _ in range(32)]
    blocks += [torch.full((512,), 0xFF, dtype=torch.uint8, device=DEV) for _ in range(256)]
    torch.cuda.synchronize()
    del blocks


def test_flow_forward_bitwise_repeatable(monkeypatch):
    """The kernels from z_mean to the flowed z have a fixed summation order (no atomics, no split-K): 32 interleaved
    rounds of each must agree bit for bit with the first, with every output, workspace and - for the MADE as a whole
    - every fresh allocation filled with 0xFF bytes before the launch.  Any difference is a race or a read of memory
    the kernel did not write."""
    _poison_workspaces(monkeypatch)
    gen = torch.Generator(device=DEV).manual_seed(9)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=gen)
    n, h, k = 2900, 500, 10
    h2, eps = rnd(n, 2 * h), rnd(n, h)
    zm, zv = rnd(n, h), torch.rand(n, h, device=DEV, generator=gen) + 0.2
    zs, z_pre = rnd(n, h), rnd(2 * k, h) * 0.5
    net = rnd(n, 2 * h) * 0.5
    x_old = rnd(n, h)
    mult = torch.bincount(torch.arange(h) % (h - 1), minlength=h).to(torch.int32).to(DEV)

    def reparam():
        out = [_nan_buffer(n, h) for _ in range(3)]
        L.call("kg_reparam_fwd", L.f32(h2), L.f32(eps), n, h, *(L.f32(t) for t in out), L.stream())
        return out

    def kl_mog():
        ws, rows, resp = _nan_buffer(3, k, h), _nan_buffer(n), _nan_buffer(n, k)
        L.call("kg_kl_mog_fwd", L.f32(zs), L.f32(zm), L.f32(zv), L.f32(z_pre), n, h, k, L.f32(ws), L.f32(rows),
               L.f32(resp), L.stream())
        return [ws, rows, resp]

    def gemm(M, N, K_, tb, bias, relu):
        a, b = rnd(M, K_), rnd(N, K_) if tb else rnd(K_, N)
        bv = rnd(N) if bias else None
        assert not ops.uses_tensor_cores(M, N, K_)

        def run():
            out = _nan_buffer(M, N)
            ops.gemm(a, b, out, trans_b=tb, bias=bv, relu=relu)
            return [out]
        return run

    def iaf():
        x_new, log_det = _nan_buffer(n, h), _nan_buffer(n)
        L.call("kg_iaf_update_fwd", L.f32(zs), L.f32(net), L.f32(x_old), L.i32(mult), n, h, L.f32(x_new),
               L.f32(log_det), L.stream())
        return [x_new, log_det]

    def reverse():
        out = _nan_buffer(n, h)
        L.call("kg_reverse_columns", L.f32(zs), n, h, L.f32(out), L.stream())
        return [out]

    def made_fwd(D, n_hidden, N):
        torch.manual_seed(D)
        made = K.MADE(D, D, n_hidden).to(DEV)
        z = rnd(N, D)

        def run():
            _poison_allocator()
            with torch.no_grad():
                x, log_det = made(z)
            return [x, log_det]
        return run

    cases = {
        "reparam_fwd": reparam, "kl_mog_fwd": kl_mog,
        "tile 300x80x40 +bias": gemm(300, 80, 40, True, True, False),           # smoke's MADE output layer
        "tile 300x40x40 +bias relu": gemm(300, 40, 40, True, True, True),
        "tile 300x40x40 no epilogue (K < 128)": gemm(300, 40, 40, False, False, False),
        "small-M 1x500x500 B k-contiguous": gemm(1, 500, 500, True, True, True),   # first pass, D = 500
        "small-M 1x500x1000 B n-contiguous": gemm(1, 500, 1000, False, False, False),
        "iaf_update_fwd": iaf, "reverse_columns": reverse,
        "MADE(40, 40, 1) N=300": made_fwd(40, 1, 300), "MADE(500, 500, 3) N=2900": made_fwd(500, 3, 2900),
    }
    first = {name: [t.clone() for t in fn()] for name, fn in cases.items()}
    for name, outs in first.items():
        assert all(bool(torch.isfinite(t).all()) for t in outs), f"{name}: non-finite output"
    bad = {}
    for _ in range(32):
        for name, fn in cases.items():
            if not all(torch.equal(a, b) for a, b in zip(fn(), first[name])):
                bad[name] = bad.get(name, 0) + 1
    assert not bad, f"launches that differ bitwise from the first (of 32 each): {bad}"
