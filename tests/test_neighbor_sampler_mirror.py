"""The neighbourhood-expansion sampler's specification (tests/neighbor_mirror.py) against the exact law of the
reference's rule (kgvae/utils.py:33-76), and its invariants at the FB15k-237 shape.  CPU only."""
import numpy as np
import pytest

import gcn_vae_b200 as K
import neighbor_mirror as M

DRAWS = 4000
P_MIN = 1e-3


@pytest.mark.parametrize("case", M.tiny_graphs(), ids=lambda c: c[0])
def test_enumeration_is_a_distribution_over_distinct_picks(case):
    _, tri, n, B = case
    probs = M.sequence_probabilities(tri, n, B)
    assert abs(sum(probs.values()) - 1.0) < 1e-12
    assert all(len(set(s)) == B and p > 0 for s, p in probs.items())


@pytest.mark.parametrize("case", M.tiny_graphs(), ids=lambda c: c[0])
def test_reference_sampler_follows_the_enumeration(case):
    """utils.sample_edge_neighborhood (numpy's random stream, the reference's calls) against the exact law: this
    validates the enumeration itself."""
    name, tri, n, B = case
    probs = M.sequence_probabilities(tri, n, B)
    adj, deg = K.utils.get_adj_and_degrees(n, np.asarray(tri))
    np.random.seed(11)
    seqs = [K.utils.sample_edge_neighborhood(adj, deg, len(tri), B) for _ in range(DRAWS)]
    assert M.chi_square_p(probs, seqs) > P_MIN, name


@pytest.mark.parametrize("tries", [M.TRIES, 0], ids=["tries", "scan-only"])
@pytest.mark.parametrize("case", M.tiny_graphs(), ids=lambda c: c[0])
def test_mirror_follows_the_enumeration(case, tries):
    """The mirror on random words against the exact law; with R = 0 every pick goes through the unpicked-entry scan
    (step 4), which must give the same law on its own."""
    name, tri, n, B = case
    probs = M.sequence_probabilities(tri, n, B)
    rng = np.random.default_rng(5)
    words = M.random_words(rng, B, DRAWS)
    seqs = []
    fallbacks = 0
    for w in words:
        out, st = M.neighbor_sample(tri, n, w, tries=tries, return_state=True)
        seqs.append(out)
        fallbacks += st["fallbacks"]
    if tries == 0:
        assert fallbacks == DRAWS * B
    assert M.chi_square_p(probs, seqs) > P_MIN, name


def test_two_components_use_the_unseen_draw():
    """Once the first component is used up, no seen entity has an unpicked edge: the draw falls back to [cnt > 0]."""
    _, tri, n, B = M.tiny_graphs()[3]
    rng = np.random.default_rng(0)
    hit = False
    for w in M.random_words(rng, B, 200):
        out, st = M.neighbor_sample(tri, n, w, return_state=True)
        if out[0] == 0:                        # (0, 0, 1) first: its component is exhausted at once
            assert not st["seen_draw"][1]
            hit = True
    assert hit


def _check_invariants(tri, n, picks, state):
    tri = np.asarray(tri)
    B = len(picks)
    assert len(np.unique(picks)) == B
    deg = np.bincount(tri[:, [0, 2]].reshape(-1), minlength=n)
    cnt = deg.copy()
    seen = np.zeros(n, dtype=bool)
    for i, e in enumerate(picks):
        s, o = tri[e, 0], tri[e, 2]
        if i > 0 and not (seen[s] or seen[o]):
            # only when no seen entity has an unpicked edge
            assert not (cnt[seen] > 0).any(), i
        cnt[s] -= 1
        cnt[o] -= 1
        seen[s] = seen[o] = True
    inc = np.bincount(tri[picks][:, [0, 2]].reshape(-1), minlength=n)
    assert np.array_equal(state["cnt"], deg - inc) and np.array_equal(state["cnt"], cnt)
    assert np.array_equal(state["seen"], seen)
    assert state["picked"].sum() == B and state["picked"][picks].all()


@pytest.mark.parametrize("skew", [0.0, 1.0])
def test_mirror_invariants_at_fb15k237_shape(skew):
    data = K.datasets.synthetic_kg("FB15k-237", seed=0, skew=skew)
    B = 1500
    words = M.random_words(np.random.default_rng(1), B)
    picks, state = M.neighbor_sample(data.train, data.num_nodes, words, return_state=True)
    _check_invariants(data.train, data.num_nodes, picks, state)


def test_mirror_adjacency_is_get_adj_and_degrees():
    data = K.datasets.synthetic_kg("toy", seed=4)
    tri = data.train.copy()
    tri[7] = (9, 0, 9)                                          # a self-loop appears twice, subject end first
    ptr, eid, other = M.adjacency(tri, data.num_nodes)
    adj, deg = K.utils.get_adj_and_degrees(data.num_nodes, tri)
    assert np.array_equal(np.diff(ptr), deg)
    for v in range(data.num_nodes):
        got = np.stack([eid[ptr[v]:ptr[v + 1]], other[ptr[v]:ptr[v + 1]]], 1)
        assert np.array_equal(got, adj[v].reshape(-1, 2))


def test_mirror_rejects_bad_sizes():
    tri = [(0, 0, 1), (1, 0, 2)]
    with pytest.raises(ValueError):
        M.neighbor_sample(tri, 3, np.zeros((3, M.WORDS), dtype=np.uint32))


@pytest.mark.parametrize("args", [(0, 5, 1), (5, 0, 1), (5, 4, 0), (5, 4, 5)],
                         ids=["no-entities", "no-triples", "B=0", "B>T"])
def test_device_plan_rejects_bad_sizes(args):
    """kg_neighbor_sample_plan refuses empty graphs and sample sizes outside 1..T before touching the device."""
    import ctypes
    handle = K._lib.lib()
    k, ws = ctypes.c_int(), ctypes.c_size_t()
    assert handle.kg_neighbor_sample_plan(*args, ctypes.byref(k), ctypes.byref(ws)) == -1
    assert b"neighbor_sample" in handle.kg_last_error()
