"""Host logic of the multi-GPU link-prediction driver, on CPU.

* ``parallel.merge_topk`` with the gloo backend at world size 2 and 3: every rank holds the top-k lists of its own
  entity shard, and the merged lists must equal a full sort of all candidates by (score desc, id asc).  The scores
  are small integers, so ties are everywhere, including across shard boundaries; some candidates are ineligible
  (filtered), some shards hold fewer than k of them or none at all.
* ``link_predict.rank_seeds``: identically seeded processes leave with distinct numpy and torch streams, derived as
  its docstring says; one process leaves both streams untouched."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gcn_vae_b200 import link_predict, parallel

KS = (1, 3, 10)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _problem(case):
    """(scores fp32 [M, V], eligible bool [M, V]) of one case, the same in every process."""
    rng = np.random.default_rng(case)
    M, V = 9, int(rng.integers(5, 40))
    scores = rng.integers(-2, 3, size=(M, V)).astype(np.float32)
    eligible = rng.random((M, V)) < 0.8
    eligible[0] = False                       # a query with no candidate at all
    eligible[1] = np.arange(V) < 2            # a query with fewer than k candidates
    return torch.from_numpy(scores), torch.from_numpy(eligible)


def _top(scores, eligible, lo, hi, k):
    """Top-k of the candidates [lo, hi) by full sort: (idx int32 [M, k] global ids or -1, score fp32 [M, k])."""
    M = scores.shape[0]
    idx = torch.full((M, k), -1, dtype=torch.int32)
    sc = torch.full((M, k), float("-inf"), dtype=torch.float32)
    for m in range(M):
        cand = sorted((-float(scores[m, j]), j) for j in range(lo, hi) if eligible[m, j])[:k]
        for i, (s, j) in enumerate(cand):
            idx[m, i], sc[m, i] = j, -s
    return idx, sc


def _bounds(V, world, how):
    if how == "block":
        return [parallel.entity_shard(V, p, world) for p in range(world)]
    cuts = [0, 0] + [min(V, 3 + 5 * p) for p in range(world - 2)] + [V]        # rank 0's shard is empty
    return [(cuts[p], cuts[p + 1]) for p in range(world)]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = {}
        for case in range(6):
            scores, eligible = _problem(case)
            V = scores.shape[1]
            for how in ("block", "empty-first"):
                lo, hi = _bounds(V, world, how)[rank]
                for k in KS:
                    idx, sc = _top(scores, eligible, lo, hi, k)
                    res[(case, how, k)] = parallel.merge_topk(idx, sc, k)
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_merge_topk_equals_full_sort(world):
    port = _free_port()
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
        res = [dict(out[r]) for r in range(world)]
    checked = 0
    for (case, how, k), (idx, sc) in res[0].items():
        scores, eligible = _problem(case)
        want_idx, want_sc = _top(scores, eligible, 0, scores.shape[1], k)
        assert idx.dtype == torch.int32 and sc.dtype == torch.float32 and idx.shape == (scores.shape[0], k)
        assert torch.equal(idx, want_idx), (case, how, k, idx, want_idx)
        assert torch.equal(sc, want_sc), (case, how, k)
        assert (idx[0] == -1).all() and (idx[1, 2:] == -1).all()          # padding
        for r in range(1, world):                                         # every rank returns the same lists
            assert torch.equal(res[r][(case, how, k)][0], idx) and torch.equal(res[r][(case, how, k)][1], sc)
        checked += 1
    assert checked == 6 * 2 * len(KS)


def test_merge_topk_without_process_group_sorts_one_list():
    idx = torch.tensor([[4, -1, 2, 7]], dtype=torch.int32)
    sc = torch.tensor([[1.0, 5.0, 1.0, 3.0]])
    got_idx, got_sc = parallel.merge_topk(idx, sc, 5)
    assert got_idx.tolist() == [[7, 2, 4, -1, -1]]
    assert got_sc.tolist() == [[3.0, 1.0, 1.0, float("-inf"), float("-inf")]]


def _draws():
    return np.random.rand(4).tolist(), torch.rand(4).tolist()


@pytest.mark.parametrize("world", [2, 3])
def test_rank_seeds_give_identically_seeded_ranks_distinct_streams(world):
    draws = []
    for rank in range(world):
        np.random.seed(7)
        torch.manual_seed(11)
        torch.rand(3)                                  # the model's initialisation consumes the torch stream
        link_predict.rank_seeds(rank, world)
        got = _draws()
        # the derivation the docstring states
        np.random.seed(7)
        base = int(np.random.randint(0, 2**31 - world))
        np.random.seed(base + rank)
        torch.manual_seed(11 + rank)
        assert got == _draws(), rank
        draws.append(got)
    for a in range(world):
        for b in range(a + 1, world):
            assert draws[a][0] != draws[b][0] and draws[a][1] != draws[b][1], (a, b)


def test_rank_seeds_single_process_changes_nothing():
    np.random.seed(3)
    torch.manual_seed(5)
    torch.rand(2)
    link_predict.rank_seeds(0, 1)
    got = _draws()
    np.random.seed(3)
    torch.manual_seed(5)
    torch.rand(2)
    assert got == _draws()
