"""Per-kernel parity: each C-ABI entry point (through ops.py) against the oracle / plain fp32
torch on the same seeded inputs.  Tolerance 1e-4 relative to the tensor scale (north_star),
integers bit-exact."""
import numpy as np
import pytest
import torch

from helpers import O, RTOL, assert_close

import gcn_vae_b200 as K
from gcn_vae_b200 import _lib as L
from gcn_vae_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand_graph(seed, n, e, r):
    rng = np.random.default_rng(seed)
    src = rng.integers(0, n, e)
    dst = rng.integers(0, max(1, n - 3), e)          # the last nodes stay isolated
    et = rng.integers(0, r, e)
    order = np.lexsort((et, src, dst))
    src, dst, et = src[order], dst[order], et[order]
    norm = rng.random(e).astype(np.float32) + 0.1
    return src, dst, et, norm


def _index(src, dst, et, norm, n, r, node_major=False):
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(DEV)
    return ops.graph_index(t(src, torch.int32), t(dst, torch.int32), t(et, torch.int32),
                           t(norm, torch.float32), n, r, node_major=node_major)


# ------------------------------------------------------------------------------ graph (a1)
@pytest.mark.parametrize("n,e,r", [(50, 400, 6), (7, 0, 3), (300, 5000, 40), (5, 64, 1)])
def test_graph_index_integer_exact(n, e, r):
    src, dst, et, norm = _rand_graph(0, n, e, r)
    perm = np.random.default_rng(1).permutation(e)       # hand it over unsorted
    gi = _index(src[perm], dst[perm], et[perm], norm[perm], n, r, node_major=True)
    s_, d_, t_, w_ = src[perm], dst[perm], et[perm], norm[perm]
    for ptr, pack, key, cols in ((gi.row_ptr, gi.fwd_pack, d_, (s_, t_, w_.view(np.int32), d_)),
                                 (gi.col_ptr, gi.bwd_pack, s_, (d_, t_, w_.view(np.int32), np.arange(e))),
                                 (gi.rel_ptr, gi.rel_pack, t_, (s_, d_, t_, w_.view(np.int32)))):
        order = np.argsort(key, kind="stable")
        nbins = r if key is t_ else n
        want_ptr = np.concatenate(([0], np.cumsum(np.bincount(key, minlength=nbins))))
        assert np.array_equal(ptr.cpu().numpy(), want_ptr)
        if e:
            want = np.stack([c[order] for c in cols], axis=1).astype(np.int32)
            assert np.array_equal(pack.cpu().numpy()[:e], want)


@pytest.mark.parametrize("n,t,r", [(40, 300, 5), (1000, 20000, 237), (6, 1, 2)])
def test_graph_build_matches_reference_order(n, t, r):
    rng = np.random.default_rng(2)
    s, o, rel = rng.integers(0, n, t), rng.integers(0, n, t), rng.integers(0, r, t)
    want = O.build_graph_from_triplets(n, r, s, rel, o)
    dv = lambda a: torch.from_numpy(a.astype(np.int32)).to(DEV)
    gi = ops.graph_build(dv(s), dv(rel), dv(o), n, r, node_major=True)
    assert np.array_equal(gi.e_src.cpu().numpy(), want["src"])
    assert np.array_equal(gi.e_dst.cpu().numpy(), want["dst"])
    assert np.array_equal(gi.e_type.cpu().numpy(), want["etype"])
    assert np.array_equal(gi.node_norm.cpu().numpy(), want["norm"])          # bit-exact fp32
    fwd = gi.fwd_pack.cpu().numpy()[:2 * t]
    assert np.array_equal(fwd[:, 0], want["src"]) and np.array_equal(fwd[:, 1], want["etype"])
    assert np.array_equal(fwd[:, 2].view(np.float32), want["edge_norm"].reshape(-1))
    assert np.array_equal(gi.row_ptr.cpu().numpy(),
                          np.concatenate(([0], np.cumsum(np.bincount(want["dst"], minlength=n)))))


# ------------------------------------------------------------------------------ gemm
@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (130, 70, 33), (257, 500, 500), (64, 1000, 20), (500, 100, 3000),
                                   (1, 500, 500), (3, 77, 1000), (8, 1000, 45)])        # last three: the M <= 8 kernel
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_gemm_layouts(M, N, K, ta, tb):
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a = torch.randn((K, M) if ta else (M, K), generator=g)
    b = torch.randn((N, K) if tb else (K, N), generator=g)
    want = (a.t() if ta else a).double() @ (b.t() if tb else b).double()
    out = torch.empty(M, N, device=DEV)
    ops.gemm(a.to(DEV), b.to(DEV), out, trans_a=bool(ta), trans_b=bool(tb))
    assert_close(out, want, 2e-5, f"gemm {M}x{N}x{K} ta={ta} tb={tb}")


def test_gemm_epilogue_and_accumulate():
    g = torch.Generator().manual_seed(0)
    M, N, K = 200, 90, 75
    a, b = torch.randn(M, K, generator=g), torch.randn(K, N, generator=g)
    bias, add = torch.randn(N, generator=g), torch.randn(M, N, generator=g)
    mask = (torch.rand(M, N, generator=g) < 0.8).float() / 0.8
    want = torch.relu(a @ b + bias + add) * mask
    out = torch.empty(M, N, device=DEV)
    ops.gemm(a.to(DEV), b.to(DEV), out, bias=bias.to(DEV), addend=add.to(DEV), relu=True, mask=mask.to(DEV))
    assert_close(out, want, 2e-5, "fused epilogue")
    base = torch.randn(M, N, generator=g)
    out2 = base.to(DEV).clone()
    ops.gemm(a.to(DEV), b.to(DEV), out2, accumulate=True)
    assert_close(out2, base + a @ b, 2e-5, "accumulate")
    # the M <= 8 kernel (first pass of a MADE call: one row, bias + ReLU in the epilogue; flow_network.py:91)
    for tb in (False, True):
        a1, b1 = torch.randn(2, 300, generator=g), torch.randn((N, 300) if tb else (300, N), generator=g)
        add1, mask1 = torch.randn(2, N, generator=g), (torch.rand(2, N, generator=g) < 0.8).float() / 0.8
        base1 = torch.randn(2, N, generator=g)
        out5 = base1.to(DEV).clone()
        ops.gemm(a1.to(DEV), b1.to(DEV), out5, trans_b=tb, bias=bias.to(DEV), addend=add1.to(DEV), relu=True,
                 mask=mask1.to(DEV), accumulate=True)
        assert_close(out5, base1 + torch.relu(a1 @ (b1.t() if tb else b1) + bias + add1) * mask1, 2e-5, "small-M epilogue")
    # K = 0: epilogue only
    out3 = torch.empty(M, N, device=DEV)
    ops.epilogue_only(out3, bias=bias.to(DEV), addend=add.to(DEV))
    assert_close(out3, add + bias, 1e-6, "K=0 epilogue")
    # split-K path with a mask and with accumulate
    a2, b2 = torch.randn(4000, 60, generator=g), torch.randn(4000, 50, generator=g)
    m2 = (torch.rand(60, 50, generator=g) < 0.5).float()
    out4 = torch.ones(60, 50, device=DEV)
    ops.gemm(a2.to(DEV), b2.to(DEV), out4, trans_a=True, mask=m2.to(DEV), accumulate=True)
    assert_close(out4, 1 + (a2.t().double() @ b2.double()).float() * m2, 2e-5, "split-K masked accumulate")


@pytest.mark.parametrize("M,N,K,ta,tb", [(14541, 500, 500, 0, 0), (14541, 500, 1000, 0, 1), (500, 1000, 14541, 1, 0),
                                          (300, 260, 4100, 1, 1), (1000, 500, 700, 0, 1), (129, 257, 200, 0, 0)])
def test_gemm_tensor_core_path(M, N, K, ta, tb):
    """Shapes that run on tcgen05 (two-term fp16 split under one power-of-two scale per matrix, operands read
    K-major or MN-major as stored): fp32-level accuracy against fp64 in all four orientations, with rows of
    different magnitude, the fused epilogue, and split-K.  Contract of the split: an element keeps 22 bits while it
    is within 2^-17 of the matrix maximum, below that its absolute error is 2^-40 of the maximum - so with rows
    spread over 2^16 the error stays at fp32 level relative to |a_m| |b_n|, and with rows spread over 2^24 it is
    bounded relative to the largest rows."""
    assert L.lib().kg_gemm_f32_workspace_bytes(M, N, K) > 0
    g = torch.Generator().manual_seed(M + N + K)
    a0 = torch.randn((K, M) if ta else (M, K), generator=g)
    b0 = torch.randn((N, K) if tb else (K, N), generator=g)
    for spread, tol_row, tol_mat in ((12, 1e-4, 2e-6), (4, 2e-6, 2e-6)):
        ra = torch.exp2(torch.randint(-spread, spread, (M,), generator=g).float())
        rb = torch.exp2(torch.randint(-spread, spread, (N,), generator=g).float())
        a = a0 * (ra.view(1, -1) if ta else ra.view(-1, 1))
        b = b0 * (rb.view(-1, 1) if tb else rb.view(1, -1))
        A64, B64 = (a.t() if ta else a).double(), (b.t() if tb else b).double()
        want = A64 @ B64
        bound = A64.norm(dim=1, keepdim=True) * B64.norm(dim=0, keepdim=True)     # |a_m| |b_n|
        out = torch.empty(M, N, device=DEV)
        ops.gemm(a.to(DEV), b.to(DEV), out, trans_a=bool(ta), trans_b=bool(tb))
        diff = (out.cpu().double() - want).abs()
        err = (diff / bound).max().item()
        assert err < tol_row, (spread, err)         # fp32 FMA chains sit at ~1e-7..1e-6 of |a||b| as well
        assert (diff.max() / bound.max()).item() < tol_mat, (spread, (diff.max() / bound.max()).item())
    bias, add = torch.randn(N, generator=g), torch.randn(M, N, generator=g)
    mask = (torch.rand(M, N, generator=g) < 0.8).float() / 0.8
    base = torch.randn(M, N, generator=g)
    out2 = base.to(DEV).clone()
    ops.gemm(a.to(DEV), b.to(DEV), out2, trans_a=bool(ta), trans_b=bool(tb), bias=bias.to(DEV),
             addend=add.to(DEV), relu=True, mask=mask.to(DEV), accumulate=True)
    term = torch.relu(want + bias.double() + add.double()) * mask.double()
    want2 = base.double() + term
    scale2 = bound + base.double().abs() + term.abs() + bias.double().abs() + add.double().abs()
    err2 = ((out2.cpu().double() - want2).abs() / scale2).max().item()
    assert err2 < 2e-6, err2


def test_gemm_prepared_operands_serve_all_three_layer_products():
    """kg_gemm_prepare / kg_gemm_f32_prepared: x, W and g are split once and reused, in both orientations, by the
    three products of a linear layer (kgvae/flow_network.py:15 and its backward): y = x W^T, dx = g W, dW = g^T x.
    Row slices (ld > cols) and a ragged K (not a multiple of 64) included; bitwise equal to the unprepared call."""
    g = torch.Generator().manual_seed(11)
    n, din, dout = 3001, 500, 1000
    xw = torch.randn(n, din + 12, generator=g).to(DEV)
    x = xw[:, :din]                                           # row pitch 512, 500 columns
    W = (torch.randn(dout, din, generator=g) * 0.05).to(DEV)
    gr = (torch.randn(n, dout, generator=g) * 1e-4).to(DEV)   # gradients are small: the scale is per matrix
    xp = ops.Prepared(x) if x.is_contiguous() else ops.Prepared(x.contiguous())
    Wp, gp = ops.Prepared(W), ops.Prepared(gr)
    xc = x.contiguous()
    y, dx, dW = (torch.empty(n, dout, device=DEV), torch.empty(n, din, device=DEV), torch.empty(dout, din, device=DEV))
    ops.gemm(xp, Wp, y, trans_b=True)
    ops.gemm(gp, Wp, dx)
    ops.gemm(gp, xp, dW, trans_a=True)
    x64, W64, g64 = xc.double().cpu(), W.double().cpu(), gr.double().cpu()
    for got, want, what in ((y, x64 @ W64.t(), "y"), (dx, g64 @ W64, "dx"), (dW, g64.t() @ x64, "dW")):
        assert_close(got, want, 3e-6, f"prepared {what}")
    y2, dW2 = torch.empty_like(y), torch.empty_like(dW)
    ops.gemm(xc, W, y2, trans_b=True)
    ops.gemm(gr, xc, dW2, trans_a=True)
    assert torch.equal(y, y2) and torch.equal(dW, dW2)
    # a strided source is split straight from its rows (no copy): same bits as the contiguous copy
    n_bytes = L.lib().kg_gemm_prep_bytes(n, din)
    b1, b2 = torch.zeros(n_bytes, dtype=torch.uint8, device=DEV), torch.zeros(n_bytes, dtype=torch.uint8, device=DEV)
    L.call("kg_gemm_prepare", x.data_ptr(), x.stride(0), n, din, L.ptr(b1), n_bytes, L.stream())
    L.call("kg_gemm_prepare", L.f32(xc), din, n, din, L.ptr(b2), n_bytes, L.stream())
    assert torch.equal(b1, b2)
    with pytest.raises(RuntimeError, match="below the tensor-core size"):
        L.call("kg_gemm_f32_prepared", L.ptr(b1), 0, L.ptr(b2), 1, L.f32(y), dout, 8, 8, 8, None, None, 0, None, 0,
               None, 0, L.stream())


def test_colsum_and_reductions():
    g = torch.Generator().manual_seed(1)
    for rows, cols in [(1, 1), (300, 37), (14541, 100), (0, 5)]:
        x = torch.randn(rows, cols, generator=g)
        assert_close(ops.colsum(x.to(DEV)), x.double().sum(0), 2e-5, f"colsum {rows}x{cols}")
    x = torch.randn(1_000_003, generator=g)
    assert_close(ops._reduce("kg_sum", x.to(DEV)), x.double().sum(), 1e-4, "sum")
    assert_close(ops._reduce("kg_sum_squares", x.to(DEV)), (x.double() ** 2).sum(), 1e-5, "sumsq")


# ------------------------------------------------------------------------------ embedding (a2)
def test_embedding_fwd_bwd():
    g = torch.Generator().manual_seed(2)
    table = torch.randn(50, 24, generator=g, requires_grad=True)
    ids = torch.tensor([3, 3, 49, 0, 7, 3])
    gout = torch.randn(6, 24, generator=g)
    table[ids].backward(gout)
    t2 = table.detach().to(DEV).requires_grad_(True)
    out = ops.EmbeddingFn.apply(t2, ids.to(torch.int32).to(DEV))
    out.backward(gout.to(DEV))
    assert torch.equal(out.detach().cpu(), table.detach()[ids])
    assert_close(t2.grad, table.grad, 1e-6, "embedding grad")


# ------------------------------------------------------------------------------ bdd layer (a3)
@pytest.mark.parametrize("n,e,r,B,si,so,act", [(60, 500, 6, 4, 5, 5, 1), (60, 500, 6, 4, 5, 10, 0),
                                               (200, 3000, 24, 20, 5, 10, 1), (33, 100, 3, 3, 7, 2, 0),
                                               (10, 0, 2, 2, 4, 4, 1)])
def test_bdd_layer_fwd_bwd(n, e, r, B, si, so, act):
    src, dst, et, norm = _rand_graph(3, n, e, r)
    g = torch.Generator().manual_seed(n + e)
    x = torch.randn(n, B * si, generator=g, requires_grad=True)
    weight = (torch.randn(r, B * si * so, generator=g) * 0.3).requires_grad_(True)
    loop = (torch.randn(B * si, B * so, generator=g) * 0.2).requires_grad_(True)
    bias = torch.randn(B * so, generator=g).requires_grad_(True)
    mask = (torch.rand(n, B * so, generator=g) < 0.8).float() / 0.8
    gout = torch.randn(n, B * so, generator=g)
    graph = {"num_nodes": n, "src": src, "dst": dst, "etype": et, "edge_norm": norm.reshape(-1, 1)}
    want = O.rgcn_bdd_layer(x, graph, weight, bias, loop, B, torch.relu if act else None, mask)
    want.backward(gout)

    gi = _index(src, dst, et, norm, n, r)
    cu = [t.detach().to(DEV).requires_grad_(True) for t in (x, weight, loop, bias)]
    out = ops.BddConvFn.apply(cu[0], cu[1], cu[2], cu[3], gi, B, act, mask.to(DEV))
    out.backward(gout.to(DEV))
    assert_close(out, want, RTOL, "bdd out")
    for name, a, b in zip(("dx", "dW", "dloop", "dbias"), cu, (x, weight, loop, bias)):
        assert_close(a.grad, b.grad, RTOL, f"bdd {name}")


@pytest.mark.parametrize("n,e,r,tile,by_src", [(300, 5000, 40, 64, 0), (300, 5000, 40, 64, 1), (50, 400, 6, 1000, 0),
                                               (1000, 20000, 474, 7, 1), (9, 0, 2, 4, 0)])
def test_graph_rel_tiled_order_integer_exact(n, e, r, tile, by_src):
    """kg_graph_rel_tiled: a permutation of the edges ordered by (node tile, etype), stable."""
    src, dst, et, norm = _rand_graph(5, n, e, r)
    gi = _index(src, dst, et, norm, n, r)
    pack = gi.tiled_rel_pack(by_src, tile).cpu().numpy()[:e]
    key = ((src if by_src else dst) // tile).astype(np.int64) * r + et
    order = np.argsort(key, kind="stable")
    want = np.stack([src[order], dst[order], et[order], norm[order].view(np.int32)], axis=1).astype(np.int32)
    if e:
        assert np.array_equal(pack, want)


@pytest.mark.parametrize("B,si,so", [(100, 5, 5), (100, 5, 10), (50, 10, 10), (24, 4, 4), (16, 8, 8), (8, 5, 5),
                                     (160, 5, 5), (10, 16, 16),
                                     # register-tile kernels (rgcn_bdd_tile.cuh): the WN18-shape blocks, odd
                                     # widths, K-split threads, 512-thread slots
                                     (25, 20, 20), (25, 20, 40), (50, 10, 20), (20, 25, 25), (20, 25, 50),
                                     (10, 50, 50), (10, 50, 100), (4, 20, 40)])
@pytest.mark.parametrize("tiled", [False, True])
def test_bdd_layer_fast_shapes_and_tiled_order(B, si, so, tiled, monkeypatch):
    """The register-resident fast path at the real layer widths (1 and 2 slots per CTA, several
    relation changes per chunk) and the same layer walked in node-tiled order (L2 budget forced
    down so that every matrix counts as larger than L2, streaming hints on)."""
    if tiled:
        monkeypatch.setattr(ops, "L2_TILE_BYTES", 40 * 4 * B * so)
        monkeypatch.setattr(ops, "L2_RESIDENT_BYTES", 0)
        monkeypatch.setattr(ops, "L2_STREAM_BYTES", 0)
    n, e, r = 300, 6000, 11
    src, dst, et, norm = _rand_graph(7, n, e, r)
    g = torch.Generator().manual_seed(B + si)
    x = torch.randn(n, B * si, generator=g, requires_grad=True)
    weight = (torch.randn(r, B * si * so, generator=g) * 0.3).requires_grad_(True)
    loop = torch.randn(B * si, B * so, generator=g) * 0.05
    bias = torch.randn(B * so, generator=g)
    gout = torch.randn(n, B * so, generator=g)
    graph = {"num_nodes": n, "src": src, "dst": dst, "etype": et, "edge_norm": norm.reshape(-1, 1)}
    want = O.rgcn_bdd_layer(x, graph, weight, bias, loop, B, None, None)
    want.backward(gout)
    gi = _index(src, dst, et, norm, n, r)
    cx, cw = x.detach().to(DEV).requires_grad_(True), weight.detach().to(DEV).requires_grad_(True)
    out = ops.BddConvFn.apply(cx, cw, loop.to(DEV), bias.to(DEV), gi, B, 0, None)
    out.backward(gout.to(DEV))
    if tiled:
        assert len(gi._tiled) == 2          # a dst-tiled list (forward) and a src-tiled list (backward)
    assert_close(out, want, RTOL, "bdd out")
    assert_close(cx.grad, x.grad, RTOL, "bdd dx")
    assert_close(cw.grad, weight.grad, RTOL, "bdd dW")


@pytest.mark.parametrize("kind,n,e,r,nb,fin,fout,loop", [("dense", 80, 700, 6, 3, 10, 11, True), ("dense", 80, 700, 5, 5, 16, 8, False),
                                                      ("dense", 50, 400, 9, 4, 300, 70, True), ("ids", 90, 900, 7, 3, 90, 10, True),
                                                      ("ids", 90, 900, 6, 6, 90, 12, False), ("ids", 40, 0, 3, 2, 40, 5, True),
                                                      # ids = arange: the source-tiled kernels (rgcn_basis.cu), incl.
                                                      # ragged last tile, 16 columns, hub nodes (> 512 out-edges)
                                                      ("arange", 90, 900, 7, 3, 90, 10, True),
                                                      ("arange", 333, 6000, 50, 40, 333, 10, False),
                                                      ("arange", 130, 2000, 70, 33, 130, 16, True),
                                                      ("arange_hub", 70, 4000, 9, 4, 70, 10, True),
                                                      ("arange", 40, 0, 3, 2, 40, 5, True)])
def test_basis_layer_fwd_bwd(kind, n, e, r, nb, fin, fout, loop):
    """RelGraphConv("basis") on dense and on integer-id features (kgvae/entity_classify.py:30-43)."""
    src, dst, et, norm = _rand_graph(5, n, e, r)
    if kind == "arange_hub":                    # two hubs own most edges; node 5 keeps a light share
        src = np.where(np.arange(e) % 3 == 0, 69, np.where(np.arange(e) % 3 == 1, 3, src)).astype(src.dtype)
    g = torch.Generator().manual_seed(n + e + nb)
    V = (torch.randn(nb, fin, fout, generator=g) * 0.3).requires_grad_(True)
    wc = torch.randn(r, nb, generator=g).requires_grad_(True) if nb < r else None
    lw = (torch.randn(fin, fout, generator=g) * 0.2).requires_grad_(True) if loop else None
    bias = torch.randn(fout, generator=g).requires_grad_(True)
    mask = (torch.rand(n, fout, generator=g) < 0.8).float() / 0.8
    gout = torch.randn(n, fout, generator=g)
    x = (torch.randperm(n, generator=g) if kind == "ids" else torch.arange(n) if kind.startswith("arange")
         else torch.randn(n, fin, generator=g).requires_grad_(True))
    graph = {"num_nodes": n, "src": src, "dst": dst, "etype": et, "edge_norm": norm.reshape(-1, 1)}
    want = O.rgcn_basis_layer(x, graph, V, wc, bias, lw, torch.relu, mask)
    want.backward(gout)

    layer = K.RelGraphConv(fin, fout, r, "basis", nb, activation=torch.relu, self_loop=loop, dropout=0.0).to(DEV)
    with torch.no_grad():
        layer.weight.copy_(V)
        layer.h_bias.copy_(bias)
        if wc is not None:
            layer.w_comp.copy_(wc)
        if loop:
            layer.loop_weight.copy_(lw)
    layer.dropout_mask = mask.to(DEV)
    gr = K.Graph()
    gr.add_nodes(n)
    gr.add_edges(src, dst)
    xc = x.to(DEV) if kind != "dense" else x.detach().to(DEV).requires_grad_(True)
    out = layer(gr, xc, torch.from_numpy(et).to(DEV), torch.from_numpy(norm.reshape(-1, 1)).to(DEV))
    out.backward(gout.to(DEV))
    assert_close(out, want, RTOL, "basis out")
    assert_close(layer.weight.grad, V.grad, RTOL, "basis dV")
    assert_close(layer.h_bias.grad, bias.grad, RTOL, "basis dbias")
    if wc is not None:
        assert_close(layer.w_comp.grad, wc.grad, RTOL, "basis dw_comp")
    if loop:
        assert_close(layer.loop_weight.grad, lw.grad, RTOL, "basis dloop")
    if kind == "dense":
        assert_close(xc.grad, x.grad, RTOL, "basis dx")


def test_entity_classify_model_runs():
    from gcn_vae_b200 import entity_classify as EC
    data = EC.synthetic_graph("toy", seed=1)
    g = K.Graph()
    g.add_nodes(data.num_nodes)
    g.add_edges(data.edge_src, data.edge_dst)
    torch.manual_seed(0)
    model = EC.EntityClassify(len(g), 10, data.num_classes, data.num_rels, num_bases=4, num_hidden_layers=0,
                              dropout=0.0, use_self_loop=True, use_cuda=True).to(DEV)
    feats = model.create_features()
    et = torch.from_numpy(data.edge_type).to(DEV)
    en = torch.from_numpy(data.edge_norm).unsqueeze(1).to(DEV)
    logits = model(g, feats, et, en)
    loss = torch.nn.functional.cross_entropy(logits[torch.from_numpy(data.train_idx).to(DEV)],
                                             torch.from_numpy(data.labels).to(DEV)[torch.from_numpy(data.train_idx).to(DEV)])
    loss.backward()
    # same model on the oracle
    p = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    graph = {"num_nodes": data.num_nodes, "src": data.edge_src, "dst": data.edge_dst, "etype": data.edge_type,
             "edge_norm": data.edge_norm.reshape(-1, 1)}
    h = O.rgcn_basis_layer(torch.arange(data.num_nodes), graph, p["layers.0.weight"], p["layers.0.w_comp"],
                           p["layers.0.h_bias"], p["layers.0.loop_weight"], torch.relu)
    h = O.rgcn_basis_layer(h, graph, p["layers.1.weight"], p["layers.1.w_comp"], p["layers.1.h_bias"],
                           p["layers.1.loop_weight"], lambda t: torch.softmax(t, dim=1))
    assert_close(logits, h, RTOL, "entity classify logits")
    assert all(q.grad is not None and torch.isfinite(q.grad).all() for q in model.parameters())


def test_relgraphconv_module_matches_shim_semantics():
    """Module-level call with DGL's signature, no self loop / no bias / generic activation."""
    n, e, r, B = 40, 300, 5, 4
    src, dst, et, norm = _rand_graph(4, n, e, r)
    layer = K.RelGraphConv(20, 40, r, "bdd", B, bias=False, activation=torch.tanh, self_loop=False).to(DEV)
    g = K.Graph()
    g.add_nodes(n)
    g.add_edges(src, dst)
    x = torch.randn(n, 20)
    out = layer(g, x.to(DEV), torch.from_numpy(et).to(DEV), torch.from_numpy(norm).view(-1, 1).to(DEV))
    graph = {"num_nodes": n, "src": src, "dst": dst, "etype": et, "edge_norm": norm.reshape(-1, 1)}
    want = torch.tanh(O.rgcn_bdd_layer(x, graph, layer.weight.detach().cpu(), torch.zeros(40),
                                       torch.zeros(20, 40), B))
    assert_close(out, want, RTOL, "RelGraphConv module")
    with pytest.raises(ValueError):
        K.RelGraphConv(500, 500, 36, "bdd", 100)          # DGL: num_bases > num_rels -> num_rels


# ------------------------------------------------------------------------------ latent (a5, a7)
def test_reparam_fwd_bwd():
    g = torch.Generator().manual_seed(5)
    n, h = 70, 36
    h2 = (torch.randn(n, 2 * h, generator=g) * 3).requires_grad_(True)
    h2.data[0, h] = 25.0                                   # softplus threshold branch
    eps = torch.randn(n, h, generator=g)
    m, v = O.gaussian_parameters(h2)
    z = O.sample_gaussian(m, v, eps)
    gz, gm, gv = (torch.randn(n, h, generator=g) for _ in range(3))
    (z * gz + m * gm + v * gv).sum().backward()
    c = h2.detach().to(DEV).requires_grad_(True)
    m2, v2, z2 = ops.ReparamFn.apply(c, eps.to(DEV))
    (z2 * gz.to(DEV) + m2 * gm.to(DEV) + v2 * gv.to(DEV)).sum().backward()
    assert_close(m2, m, 1e-6, "mean")
    assert_close(v2, v, 1e-5, "var")
    assert_close(z2, z, 1e-5, "z")
    assert_close(c.grad, h2.grad, RTOL, "dh2")


@pytest.mark.parametrize("n,h,k", [(50, 20, 3), (130, 100, 10), (9, 500, 16), (40, 33, 1)])
def test_kl_mog_fwd_bwd(n, h, k):
    g = torch.Generator().manual_seed(n + h + k)
    leaf = lambda *s: torch.randn(*s, generator=g).requires_grad_(True)
    z, m = leaf(n, h), leaf(n, h)
    v = (torch.rand(n, h, generator=g) + 0.2).requires_grad_(True)
    z_pre = (torch.randn(1, 2 * k, h, generator=g) * 0.5).requires_grad_(True)
    want = O.kl_term(z, m, v, z_pre, None)
    want.backward()
    cu = [t.detach().to(DEV).requires_grad_(True) for t in (z, m, v, z_pre)]
    got = ops.KlMogFn.apply(*cu)
    got.backward()
    assert_close(got, want, RTOL, "kl")
    for name, a, b in zip(("dz", "dmean", "dvar", "dz_pre"), cu, (z, m, v, z_pre)):
        assert_close(a.grad, b.grad, RTOL, f"kl {name}")


# ------------------------------------------------------------------------------ IAF (a6)
def test_made_module_matches_golden(golden):
    gv = golden("made_block")
    D, nh, N = (int(x) for x in gv["cfg"])
    made = K.MADE(D, D, nh)
    made.load_state_dict({k[len("param/"):]: torch.from_numpy(v) for k, v in gv.items() if k.startswith("param/")})
    made = made.to(DEV)
    perm = K.PermuteLayer(D)
    z = torch.from_numpy(gv["z"]).to(DEV).requires_grad_(True)
    x, log_det = made(z)
    xp, zero = perm(x)
    (xp.pow(2).sum() + log_det.sum()).backward()
    assert_close(x, gv["x"], RTOL, "made x")
    assert_close(log_det, gv["log_det"], RTOL, "made log_det")
    assert_close(xp, gv["x_perm"], RTOL, "permute")
    assert tuple(zero.shape) == (N, 1) and float(zero.abs().sum()) == 0
    assert_close(z.grad, gv["z_grad"], RTOL, "made dz")
    for l in range(nh + 2):
        assert_close(made.net[2 * l].weight.grad, gv[f"grad/net.{2 * l}.weight"], RTOL, f"made dW{l}")
        assert_close(made.net[2 * l].bias.grad, gv[f"grad/net.{2 * l}.bias"], RTOL, f"made db{l}")
    zi, ldi = made.inverse(x.detach())
    assert_close(zi, gv["inv_z"], RTOL, "inverse z")
    assert_close(ldi, gv["inv_log_det"], RTOL, "inverse log_det")


def test_permute_is_involution():
    x = torch.randn(17, 9, device=DEV)
    p = K.PermuteLayer(9)
    assert torch.equal(p(p(x)[0])[0], x)


# ------------------------------------------------------------------------------ decoder (a9)
@pytest.mark.parametrize("n,h,r,S", [(40, 20, 3, 500), (300, 100, 7, 5000), (25, 33, 2, 64), (10, 8, 2, 0),
                                     (2000, 500, 37, 20000), (50, 260, 4, 1000)])
def test_distmult_loss_fwd_bwd(n, h, r, S):
    g = torch.Generator().manual_seed(n + S)
    z = torch.randn(n, h, generator=g).requires_grad_(True)
    w = torch.randn(r, h, generator=g).requires_grad_(True)
    shift = torch.randn((), generator=g).requires_grad_(True)
    rng = np.random.default_rng(S)
    trip = np.stack([rng.integers(0, n, S), rng.integers(0, r, S), rng.integers(0, n, S)], 1).astype(np.int64)
    labels = torch.from_numpy((rng.random(S) < 0.3).astype(np.float32))
    score = O.distmult_score(z, w, trip) + shift
    cu = [t.detach().to(DEV).requires_grad_(True) for t in (z, w, shift)]
    got_score = ops.DistMultScoreFn.apply(cu[0], cu[1], torch.from_numpy(trip).to(torch.int32).to(DEV), cu[2])
    assert_close(got_score, score, RTOL, "score")
    if S == 0:
        return
    want = torch.nn.functional.binary_cross_entropy_with_logits(score, labels)
    want.backward()
    got = ops.BceLogitsFn.apply(got_score, labels.to(DEV))
    got.backward()
    assert_close(got, want, 1e-5, "bce")
    for name, a, b in zip(("dz", "dw", "dshift"), cu, (z, w, shift)):
        assert_close(a.grad, b.grad, RTOL, f"distmult {name}")
    # the fused score + BCE + dw forward used by LinkPredict.get_loss
    fu = [t.detach().to(DEV).requires_grad_(True) for t in (z, w, shift)]
    loss = ops.DistMultBceFn.apply(fu[0], fu[1], torch.from_numpy(trip).to(torch.int32).to(DEV), labels.to(DEV), fu[2])
    (loss * 3.0).backward()
    assert_close(loss, want, 1e-5, "fused bce")
    for name, a, b in zip(("dz", "dw", "dshift"), fu, (z, w, shift)):
        assert_close(a.grad, 3.0 * b.grad, RTOL, f"fused distmult {name}")


def test_distmult_negative_sampled_batch():
    """A batch shaped like the training step's (reference negative_sampling: each positive followed,
    blockwise, by negatives that corrupt its subject or its object): the fused pass walks every
    triplet from the end with the longer (relation, entity) run - objects for subject-corrupted
    negatives - and must give the same loss and gradients whichever end leads."""
    n, h, r, pos = 5000, 64, 9, 3000
    rng = np.random.default_rng(11)
    p = np.stack([rng.integers(0, n, pos), rng.integers(0, r, pos), rng.integers(0, n, pos)], 1).astype(np.int64)
    np.random.seed(5)
    trip, lab = K.utils.negative_sampling(p, n, 10)
    assert len(trip) == 11 * pos >= 1 << 14
    g = torch.Generator().manual_seed(3)
    z = torch.randn(n, h, generator=g).requires_grad_(True)
    w = torch.randn(r, h, generator=g).requires_grad_(True)
    labels = torch.from_numpy(lab.astype(np.float32))
    want = torch.nn.functional.binary_cross_entropy_with_logits(O.distmult_score(z, w, trip), labels)
    want.backward()
    cz, cw = z.detach().to(DEV).requires_grad_(True), w.detach().to(DEV).requires_grad_(True)
    t32 = torch.from_numpy(trip).to(torch.int32).to(DEV)
    loss = ops.DistMultBceFn.apply(cz, cw, t32, labels.to(DEV), None)
    loss.backward()
    assert_close(loss, want, 1e-5, "fused bce")
    assert_close(cz.grad, z.grad, RTOL, "fused dz")
    assert_close(cw.grad, w.grad, RTOL, "fused dw")
    # the orientation really is used: some records lead with the object
    idx = ops.TripletIndex(t32, n, r, entity_index=False)
    rec = idx.rs_rec.cpu().numpy()
    orig = trip[rec[:, 3]]
    swapped = (rec[:, 0] == orig[:, 2]) & (rec[:, 2] == orig[:, 0]) & (orig[:, 0] != orig[:, 2])
    kept = (rec[:, 0] == orig[:, 0]) & (rec[:, 2] == orig[:, 2])
    assert bool(np.all(swapped | kept)) and np.array_equal(rec[:, 1], orig[:, 1])
    assert swapped.sum() > pos                      # subject-corrupted negatives lead with their object
    key = rec[:, 1].astype(np.int64) * n + rec[:, 0]
    assert bool(np.all(np.diff(key) >= 0))          # (relation, leading entity) order
    runs = 1 + int((np.diff(key) != 0).sum())
    plain = len(np.unique(trip[:, 1] * n + trip[:, 0]))
    assert runs < 0.6 * plain                       # far fewer, longer runs than (r, s) order gives


@pytest.mark.parametrize("n,h,r,pos,neg", [(5000, 64, 9, 3000, 10), (300, 500, 5, 400, 3), (40, 20, 3, 60, 0)])
def test_distmult_two_pass_decoder(monkeypatch, n, h, r, pos, neg):
    """The decoder's form for a z that does not fit L2 (kg_triplet_index_trailing + kg_distmult_bce_fwd_lead +
    kg_distmult_bwd_dz_trailing; ops.DECODER_TWO_PASS forces it at test size): same loss and gradients as the oracle's
    calc_score + BCE backward (kgvae/link_predict.py:57-63,74-77), the trailing index lists every triplet once under the
    end that does not lead its rs_rec record, and the gathered gradient is bitwise repeatable (no atomics on that end)."""
    rng = np.random.default_rng(n + pos)
    p = np.stack([rng.integers(0, n, pos), rng.integers(0, r, pos), rng.integers(0, n, pos)], 1).astype(np.int64)
    np.random.seed(7)
    trip, lab = K.utils.negative_sampling(p, n, neg) if neg else (p, (rng.random(pos) < 0.4).astype(np.float32))
    g = torch.Generator().manual_seed(3)
    z = torch.randn(n, h, generator=g).requires_grad_(True)
    w = torch.randn(r, h, generator=g).requires_grad_(True)
    shift = torch.randn((), generator=g).requires_grad_(True)
    labels = torch.from_numpy(np.asarray(lab, dtype=np.float32))
    want = torch.nn.functional.binary_cross_entropy_with_logits(O.distmult_score(z, w, trip) + shift, labels)
    want.backward()
    t32 = torch.from_numpy(trip).to(torch.int32).to(DEV)
    monkeypatch.setattr(ops, "DECODER_TWO_PASS", True)
    grads = []
    for rep in range(2):
        cz, cw, cs = (t.detach().to(DEV).requires_grad_(True) for t in (z, w, shift))
        loss = ops.DistMultBceFn.apply(cz, cw, t32, labels.to(DEV), cs)
        (loss * 2.0).backward()
        assert_close(loss, want, 1e-5, "two-pass bce")
        assert_close(cz.grad, 2.0 * z.grad, RTOL, "two-pass dz")
        assert_close(cw.grad, 2.0 * w.grad, RTOL, "two-pass dw")
        assert_close(cs.grad, 2.0 * shift.grad, RTOL, "two-pass dshift")
        grads.append(cz.grad.clone())
    idx = ops.TripletIndex(t32, n, r, entity_index=False, trailing=True)
    rec, pack, ptr = idx.rs_rec.cpu().numpy(), idx.ent_pack.cpu().numpy(), idx.ent_ptr.cpu().numpy()
    S = len(trip)
    assert pack.shape[0] == S and ptr[0] == 0 and ptr[-1] == S and np.all(np.diff(ptr) >= 0)
    assert np.array_equal(np.sort(pack[:, 2]), np.arange(S))                 # every triplet once
    lead_of = np.empty(S, dtype=np.int64); trail_of = np.empty(S, dtype=np.int64)
    lead_of[rec[:, 3]], trail_of[rec[:, 3]] = rec[:, 0], rec[:, 2]
    owner = np.repeat(np.arange(n), np.diff(ptr))                            # the entity each pack entry is listed under
    assert np.array_equal(owner, trail_of[pack[:, 2]]) and np.array_equal(pack[:, 0], lead_of[pack[:, 2]])
    assert np.array_equal(pack[:, 1], trip[pack[:, 2], 1])
    # rows that are never a leading end receive only gathered contributions: bitwise equal between the two runs
    never_lead = np.setdiff1d(np.arange(n), rec[:, 0])
    if len(never_lead):
        assert torch.equal(grads[0][never_lead], grads[1][never_lead])


def test_mean_square():
    x = torch.randn(300, 50).requires_grad_(True)
    x.pow(2).mean().backward()
    c = x.detach().to(DEV).requires_grad_(True)
    got = ops.MeanSquareFn.apply(c)
    got.backward()
    assert_close(got, x.detach().pow(2).mean(), 1e-5, "mean square")
    assert_close(c.grad, x.grad, 1e-6, "mean square grad")


# ------------------------------------------------------------------------------ ranks (a10)
def _oracle_ranks(emb, w, a, r, b, shift):
    score = O.eval_scores(emb, w, torch.as_tensor(a), torch.as_tensor(r), shift)
    return O.rank_of_target(score, torch.as_tensor(b)), O.rank_interval(score, torch.as_tensor(b)), score


def test_rank_exact_fixture_bit_exact(golden):
    gv = golden("rank_exact")
    emb, w = torch.from_numpy(gv["emb"]), torch.from_numpy(gv["w"])
    t = torch.from_numpy(gv["test_triples"])
    _, ranks = K.utils.calc_mrr(emb.to(DEV), w.to(DEV), t.to(DEV), eval_bz=32, verbose=False, return_ranks=True)
    _, _, want = O.calc_mrr(emb, w, t, eval_bz=32, policy="stable", apply_sigmoid=False)
    assert torch.equal(ranks.cpu(), want)
    # and inside the tie interval of the reference's own (sigmoid, unstable-sort) ranks
    s, r, o = t[:, 0], t[:, 1], t[:, 2]
    lo_s, hi_s = O.rank_interval(torch.sigmoid(O.eval_scores(emb, w, o, r)), s)
    lo_o, hi_o = O.rank_interval(torch.sigmoid(O.eval_scores(emb, w, s, r)), o)
    lo, hi = torch.cat([lo_s, lo_o]), torch.cat([hi_s, hi_o])
    got0 = ranks.cpu() - 1
    assert bool(((got0 >= lo) & (got0 <= hi)).all())
    ref = torch.from_numpy(gv["ref_ranks"])
    untied = lo == hi
    assert torch.equal(got0[untied], ref[untied])


@pytest.mark.parametrize("V,h,M", [(96, 16, 80), (1000, 100, 300), (14541, 500, 48), (130, 20, 1)])
def test_rank_dyadic_inputs_bit_exact(V, h, M):
    """Inputs on a coarse dyadic grid: every partial sum is exact in fp32, so ranks do not
    depend on accumulation order and must equal the oracle's bit for bit (ties included)."""
    rng = np.random.default_rng(V + M)
    emb = torch.from_numpy(rng.integers(-4, 5, size=(V, h)).astype(np.float32) / 4)
    w = torch.from_numpy(rng.integers(-4, 5, size=(7, h)).astype(np.float32) / 4)
    a, r, b = rng.integers(0, V, M), rng.integers(0, 7, M), rng.integers(0, V, M)
    shift = 0.375
    want, _, _ = _oracle_ranks(emb, w, a, r, b, shift)
    dv = lambda x: torch.from_numpy(x.astype(np.int32)).to(DEV)
    got = ops.distmult_rank(emb.to(DEV), w.to(DEV), dv(a), dv(r), dv(b), shift=shift)
    assert torch.equal(got.cpu().long(), want)
    # entity shards add up (multi-GPU evaluation)
    parts = [ops.distmult_rank(emb.to(DEV), w.to(DEV), dv(a), dv(r), dv(b), shift=shift, cand_range=(lo, hi))
             for lo, hi in ((0, V // 3), (V // 3, V // 3 + 1), (V // 3 + 1, V))]
    assert torch.equal(sum(p.long() for p in parts).cpu(), want)


def test_rank_random_floats_within_tolerance_interval():
    rng = np.random.default_rng(9)
    V, h, M = 2000, 500, 100
    emb = torch.from_numpy(rng.standard_normal((V, h)).astype(np.float32))
    w = torch.from_numpy(rng.standard_normal((11, h)).astype(np.float32))
    a, r, b = rng.integers(0, V, M), rng.integers(0, 11, M), rng.integers(0, V, M)
    dv = lambda x: torch.from_numpy(x.astype(np.int32)).to(DEV)
    got = ops.distmult_rank(emb.to(DEV), w.to(DEV), dv(a), dv(r), dv(b)).cpu().long()
    score = O.eval_scores(emb.double(), w.double(), torch.as_tensor(a), torch.as_tensor(r))
    st = score.gather(1, torch.as_tensor(b).view(-1, 1))
    tol = 1e-4 * score.abs().max()
    lo = (score > st + tol).sum(1)
    hi = (score >= st - tol).sum(1) - 1
    assert bool(((got >= lo) & (got <= hi)).all())
    exact = O.rank_of_target(score, torch.as_tensor(b))
    assert int((got != exact).sum()) <= M // 20


@pytest.mark.parametrize("kind", ["gaussian", "positive", "tiny_rows"])
def test_rank_filter_margin(kind):
    """The tensor-core (two-term fp16 split) score that the rank kernel uses as a filter must stay
    far inside the band mu*|q|*|e| (mu = 2^-15) that is re-scored in fp32, and the ranks must
    equal the fp64 ranks except for candidates closer to the target than fp32 can resolve."""
    rng = np.random.default_rng(21)
    V, h, M = 3000, 500, 300
    emb = rng.standard_normal((V, h)).astype(np.float32)
    w = rng.standard_normal((5, h)).astype(np.float32)
    if kind == "positive":                      # all terms of one sign: worst case for accumulation error
        emb, w = np.abs(emb), np.abs(w)
    if kind == "tiny_rows":                     # rows of very different magnitude: per-row scaling
        emb *= np.exp2(rng.integers(-40, 20, size=(V, 1))).astype(np.float32)
    emb, w = torch.from_numpy(emb), torch.from_numpy(w)
    a, r, b = rng.integers(0, V, M), rng.integers(0, 5, M), rng.integers(0, V, M)
    dv = lambda x: torch.from_numpy(x.astype(np.int32)).to(DEV)
    tc = torch.full((M, V), float("nan"), device=DEV)
    got = ops.distmult_rank(emb.to(DEV), w.to(DEV), dv(a), dv(r), dv(b), tc_scores=tc).cpu().long()
    q = (emb[a] * w[r])
    exact = q.double() @ emb.double().T
    scale = q.double().norm(dim=1, keepdim=True) * emb.double().norm(dim=1).view(1, -1)
    dev_tc = ((tc.cpu().double() - exact).abs() / scale).max().item()
    assert dev_tc < 2.0 ** -15 / 10, dev_tc
    st = exact.gather(1, torch.as_tensor(b).view(-1, 1))
    tol = 2.0 ** -20 * scale                    # what an fp32 dot product can resolve
    lo = (exact > st + tol).sum(1)
    hi = (exact >= st - tol).sum(1) - 1
    assert bool(((got >= lo) & (got <= hi)).all())


def test_rank_filtered():
    rng = np.random.default_rng(10)
    V, h, M = 400, 32, 60
    emb = torch.from_numpy(rng.integers(-4, 5, size=(V, h)).astype(np.float32) / 4)
    w = torch.from_numpy(rng.integers(-4, 5, size=(3, h)).astype(np.float32) / 4)
    a, r, b = rng.integers(0, V, M), rng.integers(0, 3, M), rng.integers(0, V, M)
    known = [sorted(set(rng.integers(0, V, rng.integers(0, 40)).tolist()) | {int(b[i])}) for i in range(M)]
    score = O.eval_scores(emb, w, torch.as_tensor(a), torch.as_tensor(r))
    want = O.filtered_ranks(score, b, known)
    ptr = np.concatenate(([0], np.cumsum([len(x) for x in known]))).astype(np.int32)
    idx = np.concatenate(known).astype(np.int32)
    dv = lambda x: torch.from_numpy(x.astype(np.int32)).to(DEV)
    got = ops.distmult_rank(emb.to(DEV), w.to(DEV), dv(a), dv(r), dv(b), filt_ptr=dv(ptr), filt_idx=dv(idx))
    assert torch.equal(got.cpu().long(), want)


# ------------------------------------------------------------------------------ host -> device staging
def test_device_prefetcher_double_buffering():
    """utils.DevicePrefetcher: each take() returns the tensors of the matching submit(), also when the
    host buffers are rewritten between steps and the consumer is still busy with the previous set."""
    pf = K.utils.DevicePrefetcher(DEV)
    host = {"a": torch.zeros(1 << 20, dtype=torch.int32).pin_memory(), "b": torch.zeros(7, 3).pin_memory()}
    sums = []
    host["a"].fill_(0)
    pf.submit(host)
    for i in range(6):
        t = pf.take()
        torch.cuda.current_stream().synchronize()       # the copy of step i has landed: the host buffer may change
        if i + 1 < 6:
            host["a"].fill_(i + 1)
            host["b"].fill_(float(i + 1))
            pf.submit(host)
        x = t["a"].float()
        for _ in range(20):                             # keep the consumer busy while the next copy flies
            x = x * 1.0000001
        sums.append((int(t["a"][123]), float(t["b"][2, 1]), x))
    torch.cuda.synchronize()
    assert [s[0] for s in sums] == list(range(6))
    assert [s[1] for s in sums] == [float(i) for i in range(6)]


@pytest.mark.parametrize("B,si,so", [(100, 5, 5), (100, 5, 10), (25, 20, 40)])
@pytest.mark.parametrize("tiled", [False, True])
def test_bdd_layer_weight_gradient_only(B, si, so, tiled, monkeypatch):
    """The layer input does not require a gradient (dx = NULL at the C boundary): the input-gradient warps
    retire at once and the weight-gradient warps gather for themselves - independent and paired variants."""
    if tiled:
        monkeypatch.setattr(ops, "L2_TILE_BYTES", 40 * 4 * B * so)
        monkeypatch.setattr(ops, "L2_RESIDENT_BYTES", 0)
        monkeypatch.setattr(ops, "L2_STREAM_BYTES", 0)
    n, e, r = 300, 6000, 11
    src, dst, et, norm = _rand_graph(9, n, e, r)
    g = torch.Generator().manual_seed(B + so)
    x = torch.randn(n, B * si, generator=g)
    weight = (torch.randn(r, B * si * so, generator=g) * 0.3).requires_grad_(True)
    loop = torch.randn(B * si, B * so, generator=g) * 0.05
    bias = torch.randn(B * so, generator=g)
    gout = torch.randn(n, B * so, generator=g)
    graph = {"num_nodes": n, "src": src, "dst": dst, "etype": et, "edge_norm": norm.reshape(-1, 1)}
    want = O.rgcn_bdd_layer(x, graph, weight, bias, loop, B, None, None)
    want.backward(gout)
    gi = _index(src, dst, et, norm, n, r)
    cw = weight.detach().to(DEV).requires_grad_(True)
    out = ops.BddConvFn.apply(x.to(DEV), cw, loop.to(DEV), bias.to(DEV), gi, B, 0, None)
    out.backward(gout.to(DEV))
    assert_close(out, want, RTOL, "bdd out")
    assert_close(cw.grad, weight.grad, RTOL, "bdd dW")


@pytest.mark.parametrize("rows,cols,act,masked", [(1000, 500, 1, True), (77, 1000, 1, False), (300, 11, 1, True),
                                                  (64, 8, 0, True), (1, 4, 1, False)])
def test_act_dropout_bwd_with_fused_column_sums(rows, cols, act, masked):
    """kg_act_dropout_bwd_colsum = kg_act_dropout_bwd followed by kg_colsum (fused when cols % 4 == 0)."""
    g = torch.Generator().manual_seed(rows + cols)
    go = torch.randn(rows, cols, generator=g)
    out = torch.relu(torch.randn(rows, cols, generator=g))
    mask = (torch.rand(rows, cols, generator=g) < 0.8).float() / 0.8 if masked else None
    want = go * (mask if masked else 1.0)
    if act == 1:
        want = want * (out > 0).float()
    gp, db = ops.act_dropout_bwd(go.to(DEV), out.to(DEV), None if mask is None else mask.to(DEV), act, want_colsum=True)
    assert torch.equal(gp.cpu(), want)
    assert_close(db, want.double().sum(0).float(), 1e-5, "fused column sums")


# ------------------------------------------------------------------------------ device sampler (SURVEY 8f, N2)
def test_device_sampler_structure_and_train_step():
    """utils.generate_sampled_graph_and_labels_device follows the reference's sampling procedure
    (kgvae/utils.py:85-124,158-171) on the GPU: checked structurally (it does not reproduce numpy's
    random stream - the host sampler does), then one training step runs on its outputs."""
    n_ent, n_rel, B, rate = 500, 12, 600, 4
    data = K.datasets.synthetic_kg("toy", seed=1)
    tri = torch.from_numpy(data.train).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(5)
    g, node_id, etype, enorm, samples, labels = K.utils.generate_sampled_graph_and_labels_device(
        tri, B, 0.5, n_rel, rate, generator=gen)
    n, E = node_id.shape[0], etype.numel()
    nid = node_id.view(-1).cpu()
    assert torch.equal(nid, torch.unique(nid)) and len(g) == n          # ascending, duplicate-free relabelling
    pos = samples[:B].cpu().long()
    orig = torch.stack([nid[pos[:, 0]], pos[:, 1], nid[pos[:, 2]]], 1)    # back to entity ids
    train_set = {tuple(r) for r in data.train.tolist()}
    assert all(tuple(r) in train_set for r in orig.tolist())
    assert len({tuple(r) for r in orig.tolist()}) >= B - 5               # without replacement (toy data has few duplicates)
    assert labels.shape[0] == B * (rate + 1) and float(labels[:B].min()) == 1.0 and float(labels[B:].max()) == 0.0
    neg = samples[B:].cpu().long().view(rate, B, 3)
    same_s, same_o = neg[:, :, 0] == pos[:, 0], neg[:, :, 2] == pos[:, 2]
    assert bool((neg[:, :, 1] == pos[:, 1]).all()) and bool((same_s | same_o).all())      # exactly one end is redrawn
    assert 0.3 < float((~same_s).float().mean()) < 0.7                   # subject / object about evenly
    assert int(samples[:, [0, 2]].max()) < n and int(samples[:, [0, 2]].min()) >= 0
    # graph: B/2 kept edges + their reverses, (dst, src, rel) order, 1 / in-degree norms
    assert E == 2 * int(B * 0.5)
    src, dst = (t.cpu().long() for t in g._dev_edges[torch.device(DEV)])
    et = etype.cpu().long()
    key = (dst * n + src) * (2 * n_rel) + et
    assert bool((key[1:] >= key[:-1]).all())
    half = {(int(s), int(r), int(d)) for s, r, d in zip(src, et, dst) if r < n_rel}
    assert half <= {tuple(r) for r in pos.tolist()}
    assert {(d, r + n_rel, s) for s, r, d in half} == {(int(s), int(r), int(d)) for s, r, d in zip(src, et, dst) if r >= n_rel}
    deg = torch.bincount(dst, minlength=n).float()
    assert_close(enorm.view(-1), (1.0 / deg)[dst], 1e-6, "edge norm")
    # one training step on the sampled batch
    torch.manual_seed(0)
    model = K.LinkPredict(K.KGVAE, n_ent, 40, n_rel, num_bases=8, dropout=0.2, use_cuda=True, reg_param=0.01,
                          kl_param=1e-3, k=4, n_flows=1).to(DEV)
    embed = model(g, node_id, etype, enorm)
    loss, _, _, _ = model.get_loss(g, embed, samples, labels)
    loss.backward()
    assert torch.isfinite(loss) and torch.isfinite(model.w_relation.grad).all()


# ------------------------------------------------------------------------------ top-k tails (N3)
@pytest.mark.parametrize("V,h,M,k", [(96, 16, 80, 1), (1000, 100, 300, 3), (14541, 500, 200, 10), (130, 20, 1, 5),
                                     (300, 64, 50, 1)])
def test_topk_dyadic_inputs_bit_exact(V, h, M, k):
    """utils.generate's argmax generalised to top-k (kgvae/utils.py:245-288): on dyadic inputs every partial sum
    is exact, so the k best tails (ties by ascending id) and their scores must equal the oracle's exactly -
    massive ties included (few distinct score values)."""
    rng = np.random.default_rng(V * 3 + k)
    emb = torch.from_numpy(rng.integers(-4, 5, size=(V, h)).astype(np.float32) / 4)
    w = torch.from_numpy(rng.integers(-4, 5, size=(7, h)).astype(np.float32) / 4)
    a, r = rng.integers(0, V, M), rng.integers(0, 7, M)
    shift = -0.25
    want_idx, want_sc = O.topk_tails(emb, w, torch.as_tensor(a), torch.as_tensor(r), k, shift)
    dv = lambda x: torch.from_numpy(x.astype(np.int32)).to(DEV)
    idx, sc = ops.distmult_topk(emb.to(DEV), w.to(DEV), dv(a), dv(r), k=k, shift=shift)
    assert torch.equal(idx.cpu().long(), want_idx)
    assert torch.equal(sc.cpu(), want_sc)


def test_topk_random_floats_and_generate(tmp_path):
    rng = np.random.default_rng(21)
    V, h, M, k = 3000, 500, 150, 5
    emb = torch.from_numpy(rng.standard_normal((V, h)).astype(np.float32))
    w = torch.from_numpy(rng.standard_normal((11, h)).astype(np.float32))
    trip = np.stack([rng.integers(0, V, M), rng.integers(0, 11, M), rng.integers(0, V, M)], 1)
    score = O.eval_scores(emb.double(), w.double(), torch.as_tensor(trip[:, 0]), torch.as_tensor(trip[:, 1]))
    want_sc, want_idx = torch.topk(score, k, dim=1)
    out = tmp_path / "result.txt"
    tails, sc = K.utils.generate(emb.to(DEV), w.to(DEV), torch.from_numpy(trip).to(DEV), topk=k, out_path=str(out))
    # scores agree to fp32 accuracy; indices agree wherever the fp64 gap to the next candidate exceeds that accuracy
    assert float((sc.cpu().double() - want_sc).abs().max()) <= 1e-4 * float(score.abs().max())
    kth_gap = (want_sc[:, :-1] - want_sc[:, 1:]).min(1)[0]
    clear = kth_gap > 1e-4 * score.abs().max()
    assert torch.equal(tails.cpu()[clear], want_idx[clear])
    lines = out.read_text().splitlines()
    assert len(lines) >= M and lines[0].count(" - ") == 2


# ------------------------------------------------------------------------------ single-product mode
def test_single_product_mode_is_reported_separately():
    """kg_set_tc_terms(1): one fp16 product instead of the three-term split (north_star: reduced-precision GEMM
    variants, reported separately with their tolerance).  Default mode restored afterwards; the default result
    stays fp32-accurate, the single-product one is within 2^-9 of |a||b| per entry."""
    gen = torch.Generator(device=DEV).manual_seed(5)
    M, N, Kd = 4096, 512, 500
    a = torch.randn(M, Kd, device=DEV, generator=gen)
    b = torch.randn(Kd, N, device=DEV, generator=gen)
    want = a.double() @ b.double()
    bound = (a.double().norm(dim=1).view(-1, 1) * b.double().norm(dim=0).view(1, -1))
    full = ops.gemm(a, b, torch.empty(M, N, device=DEV))
    with ops.tensor_core_terms(1):
        single = ops.gemm(a, b, torch.empty(M, N, device=DEV))
    again = ops.gemm(a, b, torch.empty(M, N, device=DEV))
    assert torch.equal(full, again)                                   # mode restored
    e_full = float(((full.double() - want).abs() / bound).max())
    e_single = float(((single.double() - want).abs() / bound).max())
    assert e_full < 4e-6 and 1e-6 < e_single < 2.0 ** -9, (e_full, e_single)
    # ranks: identical wherever the exact decision margin is wider than the single product's rounding
    V, h, Mq = 4000, 500, 512
    emb = torch.randn(V, h, device=DEV, generator=gen)
    w = torch.randn(9, h, device=DEV, generator=gen)
    qa = torch.randint(0, V, (Mq,), device=DEV, generator=gen, dtype=torch.int32)
    qr = torch.randint(0, 9, (Mq,), device=DEV, generator=gen, dtype=torch.int32)
    qb = torch.randint(0, V, (Mq,), device=DEV, generator=gen, dtype=torch.int32)
    exact = ops.distmult_rank(emb, w, qa, qr, qb)
    with ops.tensor_core_terms(1):
        approx = ops.distmult_rank(emb, w, qa, qr, qb)
    # 4000 Gaussian candidates are ~0.014 apart in score around a typical target, the single product is off by
    # ~0.01: neighbours swap, nothing more (that is the tolerance this mode is reported with)
    diff = (exact.long() - approx.long()).abs()
    assert float(diff.float().mean()) < 2.0 and int(diff.max()) <= 8


# ------------------------------------------------------------------------------ bdd layer by column chunks
@pytest.mark.parametrize("n,e,r,B,so", [(300, 6000, 30, 100, 5), (300, 6000, 30, 100, 10), (64, 700, 5, 8, 5), (64, 700, 5, 8, 10)])
def test_bdd_column_chunks_match_the_full_layer(n, e, r, B, so):
    """kg_bdd_rel_fwd_cols / kg_bdd_rel_bwd_cols (column chunks for the pipelined all-gather / reduce-scatter of
    destination-partitioned training): running the layer chunk by chunk on compact column slices of x gives the
    same messages, source gradients and weight gradients as the one-launch form."""
    si = 5
    src, dst, et, norm = _rand_graph(11, n, e, r)
    gen = torch.Generator(device=DEV).manual_seed(B + so)
    x = torch.randn(n, B * si, device=DEV, generator=gen)
    weight = torch.randn(r, B * si * so, device=DEV, generator=gen) * 0.3
    dagg = torch.randn(n, B * so, device=DEV, generator=gen)
    gi = _index(src, dst, et, norm, n, r)
    agg = torch.zeros(n, B * so, device=DEV)
    L.call("kg_bdd_rel_fwd", L.f32(x), None, 0, L.i32(gi.rel_pack), e, L.f32(weight), None, B, si, so, L.f32(agg), 0, L.stream())
    dx, dw = torch.zeros_like(x), torch.zeros_like(weight)
    L.call("kg_bdd_rel_bwd", L.f32(x), None, 0, L.f32(dagg), L.i32(gi.rel_pack), e, L.f32(weight), None, B, si, so,
           L.f32(dx), L.f32(dw), 0, L.stream())
    chunks = ops._block_chunks(B, si, so, 2)
    assert len(chunks) == 2 and chunks[0][0] == 0 and chunks[-1][1] == B
    agg_c, dw_c, dx_parts = torch.zeros_like(agg), torch.zeros_like(dw), []
    for b0, b1 in chunks:
        xc = x[:, b0 * si:b1 * si].contiguous()
        L.call("kg_bdd_rel_fwd_cols", L.f32(xc), L.i32(gi.rel_pack), e, L.f32(weight), b0, b1 - b0, B, si, so,
               L.f32(agg_c), 0, L.stream())
        dxc = torch.zeros_like(xc)
        L.call("kg_bdd_rel_bwd_cols", L.f32(xc), L.f32(dagg), L.i32(gi.rel_pack), e, L.f32(weight), b0, b1 - b0, B, si, so,
               L.f32(dxc), L.f32(dw_c), 0, L.stream())
        dx_parts.append(dxc)
    assert_close(agg_c, agg, 1e-5, "chunked messages")
    assert_close(torch.cat(dx_parts, 1), dx, 1e-5, "chunked source gradients")
    assert_close(dw_c, dw, 1e-5, "chunked weight gradients")
