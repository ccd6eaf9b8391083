"""Entity-sharded top-k tails (kg_distmult_topk_shard): the lists of the shards [0, b1), [b1, b2), ... merged with
parallel.merge_topk in one process equal the unsharded kg_distmult_topk bit for bit, raw and filtered, and one shard's
raw output equals a brute-force fp32 oracle restricted to that shard."""
import numpy as np
import pytest
import torch

from helpers import O

import gcn_vae_b200 as K

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ops = K.ops


def _dyadic(rng, V, h, n_rel, levels):
    emb = torch.from_numpy(rng.integers(-levels, levels + 1, size=(V, h)).astype(np.float32) / 4)
    w = torch.from_numpy(rng.integers(-levels, levels + 1, size=(n_rel, h)).astype(np.float32) / 4)
    return emb, w


def _csr(lists):
    ptr = np.concatenate(([0], np.cumsum([len(x) for x in lists]))).astype(np.int32)
    idx = np.concatenate([np.asarray(x, dtype=np.int64) for x in lists] + [np.zeros(0, np.int64)]).astype(np.int32)
    return torch.from_numpy(ptr).to(DEV), torch.from_numpy(idx).to(DEV)


def _dv(x):
    return torch.from_numpy(np.asarray(x).astype(np.int32)).to(DEV)


def _merged(emb, w, a, r, k, shift, bounds, fp=None, fi=None):
    """Top-k of every shard [bounds[i], bounds[i+1]), merged as the ranks of a sharded generation merge them."""
    parts = [ops.distmult_topk(emb, w, a, r, k=k, shift=shift, filt_ptr=fp, filt_idx=fi, cand_range=(lo, hi))
             for lo, hi in zip(bounds[:-1], bounds[1:])]
    for (idx, sc), lo, hi in zip(parts, bounds[:-1], bounds[1:]):
        ok = idx >= 0
        assert bool(((idx >= lo) & (idx < hi))[ok].all()), (lo, hi)          # global ids of the shard only
        assert bool(torch.isneginf(sc[~ok]).all())
    return K.parallel.merge_topk(torch.cat([p[0] for p in parts], 1), torch.cat([p[1] for p in parts], 1), k)


def _oracle_shard(emb, w, a, r, k, shift, lo, hi, lists=None):
    """Dense fp32 scores of the candidates [lo, hi) (listed ids removed), stable sort: -1 / -inf past the end."""
    score = O.eval_scores(emb, w, torch.as_tensor(a), torch.as_tensor(r), shift)
    if lists is not None:
        for i, lst in enumerate(lists):
            if len(lst):
                score[i, torch.as_tensor(lst)] = -float("inf")
    score = score[:, lo:hi]
    order = torch.sort(-score, dim=1, stable=True)[1][:, :k]
    sc = score.gather(1, order)
    if sc.shape[1] < k:
        pad = k - sc.shape[1]
        sc = torch.cat([sc, torch.full((sc.shape[0], pad), -float("inf"))], 1)
        order = torch.cat([order, torch.zeros((order.shape[0], pad), dtype=order.dtype)], 1)
    return torch.where(torch.isinf(sc), torch.full_like(order, -1), order + lo), sc


def _bounds(V):
    """A one-entity shard, an empty one, boundaries off the 256-wide tiles, and a shard narrower than k."""
    return [0, 1, 1, 300, 557, V - 5, V]


@pytest.mark.parametrize("V,h,M,k,levels", [(700, 16, 160, 1, 1), (1000, 100, 160, 3, 4), (3000, 64, 120, 10, 4),
                                            (600, 8, 160, 10, 1)])
@pytest.mark.parametrize("filtered", [False, True])
def test_sharded_topk_merges_to_unsharded_on_dyadic_inputs(V, h, M, k, levels, filtered):
    """Dyadic inputs (levels = 1: massive ties): every partial sum is exact.  Filter query kinds: empty list, random
    list, the 300 best-scored entities plus random ones, and all but k - 1 entities (every shard then holds fewer
    than k unlisted entities)."""
    rng = np.random.default_rng(V + 7 * k + int(filtered))
    emb, w = _dyadic(rng, V, h, 7, levels)
    a, r = rng.integers(0, V, M), rng.integers(0, 7, M)
    shift = 0.75
    lists = fp = fi = None
    if filtered:
        dense = O.eval_scores(emb, w, torch.as_tensor(a), torch.as_tensor(r), shift)
        best = torch.sort(-dense, dim=1, stable=True)[1]
        lists = []
        for i in range(M):
            kind = i % 4
            if kind == 0:
                lst = []
            elif kind == 1:
                lst = rng.integers(0, V, rng.integers(1, 60)).tolist()
            elif kind == 2:
                lst = best[i, :300].tolist() + rng.integers(0, V, 40).tolist()
            else:
                lst = np.delete(np.arange(V), rng.choice(V, k - 1, replace=False)).tolist()
            lists.append(sorted(set(lst)))
        fp, fi = _csr(lists)
    e, wd, ad, rd = emb.to(DEV), w.to(DEV), _dv(a), _dv(r)
    want_idx, want_sc = ops.distmult_topk(e, wd, ad, rd, k=k, shift=shift, filt_ptr=fp, filt_idx=fi)
    idx, sc = _merged(e, wd, ad, rd, k, shift, _bounds(V), fp, fi)
    assert torch.equal(idx, want_idx) and torch.equal(sc, want_sc)
    o_idx, o_sc = _oracle_shard(emb, w, a, r, k, shift, 0, V, lists)
    assert torch.equal(want_idx.cpu().long(), o_idx) and torch.equal(want_sc.cpu(), o_sc)
    if filtered:
        assert bool((want_idx[3::4, -1] == -1).all())
    # every shard on its own against the brute-force oracle restricted to it
    for lo, hi in zip(_bounds(V)[:-1], _bounds(V)[1:]):
        s_idx, s_sc = ops.distmult_topk(e, wd, ad, rd, k=k, shift=shift, filt_ptr=fp, filt_idx=fi, cand_range=(lo, hi))
        o_idx, o_sc = _oracle_shard(emb, w, a, r, k, shift, lo, hi, lists)
        assert torch.equal(s_idx.cpu().long(), o_idx), (lo, hi)
        assert torch.equal(s_sc.cpu(), o_sc), (lo, hi)


@pytest.mark.parametrize("filtered", [False, True])
def test_sharded_topk_random_floats_fb15k237_width(filtered):
    """V = 14 541, h = 500 Gaussian inputs: each score is the canonical fp32 value whichever shard computes it, so the
    merge is bit-equal to the unsharded call even where fp32 ties and near-ties decide."""
    rng = np.random.default_rng(31 + int(filtered))
    V, h, M, k = 14541, 500, 200, 10
    emb = torch.from_numpy(rng.standard_normal((V, h)).astype(np.float32)).to(DEV)
    w = torch.from_numpy(rng.standard_normal((11, h)).astype(np.float32)).to(DEV)
    a, r = _dv(rng.integers(0, V, M)), _dv(rng.integers(0, 11, M))
    fp = fi = None
    if filtered:
        fp, fi = _csr([sorted(set(rng.integers(0, V, 150).tolist())) for _ in range(M)])
    want = ops.distmult_topk(emb, w, a, r, k=k, shift=0.5, filt_ptr=fp, filt_idx=fi)
    for bounds in (_bounds(V), [K.parallel.entity_shard(V, p, 8)[0] for p in range(8)] + [V]):
        idx, sc = _merged(emb, w, a, r, k, 0.5, bounds, fp, fi)
        assert torch.equal(idx, want[0]) and torch.equal(sc, want[1])


def test_sharded_topk_rejects_a_bad_range():
    emb = torch.ones(10, 8, device=DEV)
    w = torch.ones(2, 8, device=DEV)
    a = r = torch.zeros(3, dtype=torch.int32, device=DEV)
    for rng in ((5, 3), (-1, 4), (0, 11)):
        with pytest.raises(RuntimeError, match="candidate shard"):
            ops.distmult_topk(emb, w, a, r, k=2, cand_range=rng)
