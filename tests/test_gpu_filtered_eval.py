"""Filtered evaluation and filtered generation on the GPU (an extension: the reference is raw-only,
kgvae/link_predict.py:7): the device filter lists against utils.build_filter, filtered ranks through calc_mrr against
the oracle, filtered top-k tails against a dense brute-force oracle, and the driver's --filtered flag."""
import os
import re

import numpy as np
import pytest
import torch

from helpers import O

import gcn_vae_b200 as K

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ops = K.ops


def _assert_lists_match(known, num_nodes, num_rels, qa, qr):
    """FilterIndex.lists equals utils.build_filter bit for bit, in both directions."""
    fi = K.utils.FilterIndex(known, num_nodes, num_rels, DEV)
    for direction in ("object", "subject"):
        want_ptr, want_idx = K.utils.build_filter(known, qa, qr, num_rels, direction, "cpu")
        ptr, idx = fi.lists(torch.as_tensor(qa).to(DEV), torch.as_tensor(qr).to(DEV), direction)
        assert ptr.dtype == torch.int32 and idx.dtype == torch.int32
        assert torch.equal(ptr.cpu(), want_ptr), direction
        assert torch.equal(idx.cpu(), want_idx), direction
    return fi


def test_filter_lists_toy_with_duplicates_repeats_empty_lists_and_last_ids():
    d = K.datasets.synthetic_kg("toy", seed=4)
    N, R = d.num_nodes, d.num_rels
    known = np.concatenate([d.train, d.valid, d.test])
    rng = np.random.default_rng(0)
    dup = known[rng.integers(0, len(known), 500)]                       # duplicated triples
    last = np.array([[N - 1, R - 1, N - 1], [N - 1, R - 1, 0], [0, R - 1, N - 1], [N - 1, 0, 7], [N - 1, R - 1, 3]])
    known = np.concatenate([known, dup, last, last])[rng.permutation(len(known) + 500 + 10)]
    q = np.concatenate([d.test[:, [0, 1]], d.test[:40, [0, 1]], d.test[:40, [2, 1]],     # repeated queries
                        [[N - 1, R - 1], [0, R - 1], [N - 1, 0], [N - 1, R - 1]],          # ids at N-1 / R-1
                        np.stack([rng.integers(0, N, 200), rng.integers(0, R, 200)], 1)])  # mostly empty lists
    _assert_lists_match(known, N, R, q[:, 0], q[:, 1])
    ptr, _ = K.utils.build_filter(known, q[:, 0], q[:, 1], R, "object", "cpu")
    assert int((ptr[1:] == ptr[:-1]).sum()) > 50                        # the fixture has empty lists


def test_filter_lists_fb15k237_skewed_test_set():
    d = K.datasets.synthetic_kg("FB15k-237", seed=1, skew=1.0)
    known = np.concatenate([d.train, d.valid, d.test])
    q = np.concatenate([d.test[:, [0, 1]], d.test[:, [2, 1]]])
    _assert_lists_match(known, d.num_nodes, d.num_rels, q[:, 0], q[:, 1])
    ptr, _ = K.utils.build_filter(known, q[:, 0], q[:, 1], d.num_rels, "object", "cpu")
    assert int((ptr[1:] - ptr[:-1]).max()) >= 200                      # lists run to hundreds of entries


def test_filter_lists_wikikg2_key_width():
    """2 bits(N) + bits(R) = 54 at the wikikg2 entity and relation counts, at a reduced triple count."""
    d = K.datasets.synthetic_kg("wikikg2", seed=2, scale=0.01)
    known = np.concatenate([d.train, d.valid, d.test,
                            [[d.num_nodes - 1, d.num_rels - 1, d.num_nodes - 1], [5, d.num_rels - 1, d.num_nodes - 1]]])
    q = np.concatenate([d.test[:, [0, 1]], [[d.num_nodes - 1, d.num_rels - 1], [5, d.num_rels - 1]]])
    _assert_lists_match(known, d.num_nodes, d.num_rels, q[:, 0], q[:, 1])


def test_filter_lists_empty_inputs():
    fi = _assert_lists_match(np.zeros((0, 3), dtype=np.int64), 50, 4, [1, 2, 3], [0, 1, 3])
    ptr, idx = fi.lists(torch.zeros(0, dtype=torch.int32, device=DEV), torch.zeros(0, dtype=torch.int32, device=DEV),
                        "object")
    assert ptr.tolist() == [0] and idx.numel() == 0


def _dyadic(rng, V, h, n_rel, levels=4):
    emb = torch.from_numpy(rng.integers(-levels, levels + 1, size=(V, h)).astype(np.float32) / 4)
    w = torch.from_numpy(rng.integers(-levels, levels + 1, size=(n_rel, h)).astype(np.float32) / 4)
    return emb, w


def test_calc_mrr_filtered_ranks_equal_the_oracle():
    rng = np.random.default_rng(11)
    V, h, R = 400, 32, 3
    emb, w = _dyadic(rng, V, h, R)
    # few (a, r) pairs with many known ends, so that lists are long and many candidates are taken out
    heads = rng.integers(0, V, 30)
    known = np.stack([heads[rng.integers(0, 30, 4000)], rng.integers(0, R, 4000), rng.integers(0, V, 4000)], 1)
    known = np.concatenate([known, known[:, ::-1]])                   # (o, r, s) too: long subject lists
    test = known[rng.choice(len(known), 80, replace=False)]
    fi = K.utils.FilterIndex(known, V, R, DEV)
    test_d = torch.from_numpy(test).to(DEV)
    _, raw = K.utils.calc_mrr(emb.to(DEV), w.to(DEV), test_d, verbose=False, return_ranks=True)
    _, got = K.utils.calc_mrr(emb.to(DEV), w.to(DEV), test_d, verbose=False, return_ranks=True, filter_index=fi)
    kset = {tuple(t) for t in known.tolist()}
    s, r, o = (torch.as_tensor(test[:, i]) for i in range(3))
    lists_s = [[c for c in range(V) if (c, int(r[i]), int(o[i])) in kset] for i in range(len(test))]
    lists_o = [[c for c in range(V) if (int(s[i]), int(r[i]), c) in kset] for i in range(len(test))]
    want = torch.cat([O.filtered_ranks(O.eval_scores(emb, w, o, r), s, lists_s),
                      O.filtered_ranks(O.eval_scores(emb, w, s, r), o, lists_o)]) + 1
    assert torch.equal(got.cpu(), want)
    assert bool((got <= raw).all()) and bool((got < raw).any())
    # periodic validation ranks only the first eval_bz queries of each direction
    _, part = K.utils.calc_mrr(emb.to(DEV), w.to(DEV), test_d, eval_bz=25, all_batches=False, verbose=False,
                               return_ranks=True, filter_index=fi)
    assert torch.equal(part.cpu(), torch.cat([want[:25], want[80:105]]))


def _oracle_filtered_topk(emb, w, a, r, k, shift, lists):
    """Dense scores with the listed ids removed, then a stable sort (ties by ascending id); -1 / -inf past the end."""
    score = O.eval_scores(emb, w, torch.as_tensor(a), torch.as_tensor(r), shift)
    for i, lst in enumerate(lists):
        if len(lst):
            score[i, torch.as_tensor(lst)] = -float("inf")
    order = torch.sort(-score, dim=1, stable=True)[1][:, :k]
    sc = score.gather(1, order)
    return torch.where(torch.isinf(sc), torch.full_like(order, -1), order), sc


def _csr(lists):
    ptr = np.concatenate(([0], np.cumsum([len(x) for x in lists]))).astype(np.int32)
    idx = np.concatenate([np.asarray(x, dtype=np.int64) for x in lists] + [np.zeros(0, np.int64)]).astype(np.int32)
    return torch.from_numpy(ptr).to(DEV), torch.from_numpy(idx).to(DEV)


@pytest.mark.parametrize("V,h,M,k,levels", [(700, 16, 160, 1, 1), (1000, 100, 160, 3, 4), (3000, 64, 120, 10, 4),
                                            (600, 8, 160, 10, 1)])
def test_filtered_topk_dyadic_inputs_bit_exact(V, h, M, k, levels):
    """Dyadic inputs: every partial sum is exact, so tails and scores must equal the oracle's.  levels = 1: massive
    ties.  Query kinds: empty list, random list, a list of the 300 best-scored entities (longer than a 256-wide tile)
    plus random ones, and all but k - 1 entities listed (trailing -1)."""
    rng = np.random.default_rng(V + 7 * k)
    emb, w = _dyadic(rng, V, h, 7, levels)
    a, r = rng.integers(0, V, M), rng.integers(0, 7, M)
    shift = 0.75
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
    want_idx, want_sc = _oracle_filtered_topk(emb, w, a, r, k, shift, lists)
    fp, fi = _csr(lists)
    dv = lambda x: torch.from_numpy(x.astype(np.int32)).to(DEV)
    idx, sc = ops.distmult_topk(emb.to(DEV), w.to(DEV), dv(a), dv(r), k=k, shift=shift, filt_ptr=fp, filt_idx=fi)
    assert torch.equal(idx.cpu().long(), want_idx)
    assert torch.equal(sc.cpu(), want_sc)
    assert bool((want_idx[3::4, -1] == -1).all())                     # fewer than k unlisted entities
    # an empty filter changes nothing
    plain = ops.distmult_topk(emb.to(DEV), w.to(DEV), dv(a), dv(r), k=k, shift=shift)
    assert torch.equal(idx[0::4], plain[0][0::4]) and torch.equal(sc[0::4], plain[1][0::4])


def test_filtered_topk_random_floats_fb15k237_width():
    """V = 14 541, h = 500 Gaussian inputs against an fp64 reference: scores within fp32 accuracy, tails equal
    wherever the fp64 gaps around the k best (including the one to the (k+1)-th) exceed that accuracy."""
    rng = np.random.default_rng(23)
    V, h, M, k = 14541, 500, 200, 10
    emb = torch.from_numpy(rng.standard_normal((V, h)).astype(np.float32))
    w = torch.from_numpy(rng.standard_normal((11, h)).astype(np.float32))
    a, r = rng.integers(0, V, M), rng.integers(0, 11, M)
    score = O.eval_scores(emb.double(), w.double(), torch.as_tensor(a), torch.as_tensor(r))
    top = torch.topk(score, 40, dim=1)[1]
    lists = [sorted(set(top[i, : 5 * (i % 8)].tolist() + rng.integers(0, V, 100).tolist())) for i in range(M)]
    filt = score.clone()
    for i, lst in enumerate(lists):
        filt[i, torch.as_tensor(lst)] = -float("inf")
    want_sc, want_idx = torch.topk(filt, k + 1, dim=1)
    fp, fi = _csr(lists)
    dv = lambda x: torch.from_numpy(x.astype(np.int32)).to(DEV)
    idx, sc = ops.distmult_topk(emb.to(DEV), w.to(DEV), dv(a), dv(r), k=k, filt_ptr=fp, filt_idx=fi)
    tol = 1e-4 * float(score.abs().max())
    assert float((sc.cpu().double() - want_sc[:, :k]).abs().max()) <= tol
    clear = (want_sc[:, :-1] - want_sc[:, 1:]).min(1)[0] > tol
    assert int(clear.sum()) > M // 2
    assert torch.equal(idx.cpu().long()[clear], want_idx[clear, :k])
    listed = set((i, c) for i, lst in enumerate(lists) for c in lst)
    assert not any((i, c) in listed for i, row in enumerate(idx.cpu().tolist()) for c in row)


# ------------------------------------------------------------------------------ driver --filtered
def _args(tmp_path, *extra):
    argv = ["-d", "toy", "--gpu", "0", "--n-hidden", "40", "--n-bases", "8", "--graph-batch-size", "600",
            "--negative-sample", "4", "--n-epochs", "2", "--evaluate-every", "2", "--eval-batch-size", "64",
            "--mog-k", "4", "--n-flows", "1", "--kl-param", "1e-3",
            "--model-state-file", os.path.join(str(tmp_path), "model_state.pth"), *extra]
    return K.link_predict.build_parser().parse_args(argv)


def _metric(out, name):
    return [float(x) for x in re.findall(re.escape(name) + r": ([0-9.]+)", out)]


def test_driver_filtered_validation_and_test_mode(tmp_path, capsys):
    np.random.seed(4)
    torch.manual_seed(4)
    K.link_predict.main(_args(tmp_path, "--filtered"))
    out = capsys.readouterr().out
    assert "start eval" in out and len(_metric(out, "MRR (raw)")) == 1 and len(_metric(out, "MRR (filtered)")) == 1
    mrr = K.link_predict.main(_args(tmp_path, "--test-mode", "1", "--filtered"))
    out = capsys.readouterr().out
    raw, filt = _metric(out, "MRR (raw)"), _metric(out, "MRR (filtered)")
    assert len(raw) == 1 and len(filt) == 1 and out.index("MRR (raw)") < out.index("MRR (filtered)")
    assert "Hits (filtered) @ 10" in out
    assert abs(mrr - raw[0]) < 1e-6 and filt[0] >= raw[0]


def test_driver_filtered_generation_writes_only_unseen_tails(tmp_path, capsys, monkeypatch):
    np.random.seed(5)
    torch.manual_seed(5)
    K.link_predict.main(_args(tmp_path))
    monkeypatch.chdir(tmp_path)
    tails = K.link_predict.main(_args(tmp_path, "--test-mode", "1", "--generate", "1", "--filtered"))
    assert "generated tails" in capsys.readouterr().out
    d = K.datasets.load_data("toy")
    known = {tuple(t) for t in np.concatenate([d.train, d.valid, d.test]).tolist()}
    gen = [tuple(int(x[1:]) for x in line.split(" = ")) for line in (tmp_path / "result.txt").read_text().splitlines()
           if " = " in line]
    assert len(gen) == len(d.test) and not any(t in known for t in gen)
    assert not any((int(s), int(r), int(c)) in known for (s, r, _), c in zip(d.test.tolist(), tails[:, 0].tolist()))
