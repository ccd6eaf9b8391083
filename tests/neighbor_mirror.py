"""numpy restatement of the device neighbourhood-expansion edge sampler (csrc/neighbor_sampler.cu), pick for pick.

It is the specification the kernel is tested against.  The procedure is the reference's ``sample_edge_neighborhood``
(kgvae/utils.py:33-76, ``utils.sample_edge_neighborhood``) driven by caller-given uniform 32-bit words instead of
numpy's random stream:

* adjacency: for each entity v its entries (edge id, other end) in the order of ``utils.get_adj_and_degrees`` -
  ascending edge id, the subject end first for a self-loop, which appears twice; ``deg[v]`` entries;
* state: ``cnt = deg``, ``seen = 0``, ``picked = 0``;
* pick i uses the words ``w[i, 0..WORDS-1]``:
  1. weights ``cnt * seen``, or ``[cnt > 0]`` when those sum to 0; W their sum;
  2. ``r = (w0 W) >> 32``; v = the first entity whose inclusive prefix sum of the weights exceeds r; ``seen[v] = 1``;
  3. for t = 1..R: ``j = (w_t deg[v]) >> 32``; take entry j if its edge is not picked;
  4. if no try succeeded: ``k = (w_{R+1} cnt[v]) >> 32``; take the k-th unpicked entry of v's list, in list order;
  5. ``picked[e] = 1``, ``cnt[v] -= 1``, ``cnt[other] -= 1`` (a self-loop loses 2), ``seen[other] = 1``.

``cnt[v]`` is always the number of unpicked entries of v, so step 4 is the conditional law of the reference's
rejection loop and the whole procedure is the reference's up to the 2^-32 granularity of the integer mapping.
"""
import numpy as np

WORDS, TRIES = 8, 6            # KG_NEIGHBOR_WORDS, KG_NEIGHBOR_TRIES


def adjacency(triplets, num_nodes):
    """(ptr [N+1], eid [2T], other [2T]): the lists of utils.get_adj_and_degrees in CSR form."""
    tri = np.asarray(triplets, dtype=np.int64)
    ends = tri[:, [0, 2]].reshape(-1)
    order = np.argsort(ends, kind="stable")
    deg = np.bincount(ends, minlength=num_nodes)
    return np.concatenate(([0], np.cumsum(deg))), order // 2, tri[:, [2, 0]].reshape(-1)[order]


def neighbor_sample(triplets, num_nodes, words, tries=TRIES, return_state=False):
    """The picks (int64 [B]) for ``words`` (uint32 [B, WORDS]).  ``tries``: R (0 forces step 4 on every pick).
    ``return_state``: also return a dict with the final ``cnt`` / ``seen`` / ``picked``, the number of step-4 picks
    ``fallbacks`` and, per pick, the vertex ``v`` and whether the seen-weighted draw was used (``seen_draw``)."""
    ptr, eid, other = adjacency(triplets, num_nodes)
    T = len(eid) // 2
    words = np.asarray(words, dtype=np.uint64)
    B = words.shape[0]
    if not 1 <= B <= T:
        raise ValueError(f"sample size must be in 1 .. {T}")
    cnt = np.diff(ptr).astype(np.int64)
    seen = np.zeros(num_nodes, dtype=bool)
    picked = np.zeros(T, dtype=bool)
    out = np.empty(B, dtype=np.int64)
    verts, seen_draw, fallbacks = np.empty(B, dtype=np.int64), np.empty(B, dtype=bool), 0
    for i in range(B):
        w = [int(x) for x in words[i]]
        weights = cnt * seen
        W = int(weights.sum())
        seen_draw[i] = W > 0
        if W == 0:
            weights = (cnt > 0).astype(np.int64)
            W = int(weights.sum())
        r = (w[0] * W) >> 32
        v = int(np.searchsorted(np.cumsum(weights), r, side="right"))
        seen[v] = True
        lo, d = int(ptr[v]), int(ptr[v + 1] - ptr[v])
        j = None
        for t in range(1, tries + 1):
            jt = lo + ((w[t] * d) >> 32)
            if not picked[eid[jt]]:
                j = jt
                break
        if j is None:
            fallbacks += 1
            k = (w[tries + 1] * int(cnt[v])) >> 32
            j = lo + int(np.flatnonzero(~picked[eid[lo:lo + d]])[k])
        e, o = int(eid[j]), int(other[j])
        picked[e] = True
        cnt[v] -= 1
        cnt[o] -= 1
        seen[o] = True
        out[i] = e
        verts[i] = v
    if return_state:
        return out, dict(cnt=cnt, seen=seen, picked=picked, fallbacks=fallbacks, v=verts, seen_draw=seen_draw)
    return out


def random_words(rng, B, n_samples=None):
    shape = (B, WORDS) if n_samples is None else (n_samples, B, WORDS)
    return rng.integers(0, 2 ** 32, size=shape, dtype=np.uint64).astype(np.uint32)


def sequence_probabilities(triplets, num_nodes, B):
    """Exact probability of every ordered sequence of B picks under the reference's rule (a vertex ~ cnt * seen, or
    ~ [cnt > 0] when that sums to 0, then an entry uniform among its unpicked entries).  dict tuple -> float."""
    ptr, eid, other = adjacency(triplets, num_nodes)
    T = len(eid) // 2
    probs = {}

    def walk(prefix, p, cnt, seen, picked):
        if len(prefix) == B:
            probs[tuple(prefix)] = probs.get(tuple(prefix), 0.0) + p
            return
        weights = cnt * seen
        if weights.sum() == 0:
            weights = (cnt > 0).astype(np.int64)
        W = weights.sum()
        for v in np.flatnonzero(weights):
            pv = p * weights[v] / W
            lo, hi = ptr[v], ptr[v + 1]
            for j in range(lo, hi):
                e, o = eid[j], other[j]
                if picked[e]:
                    continue
                c2, s2, k2 = cnt.copy(), seen.copy(), picked.copy()
                k2[e] = True
                c2[v] -= 1
                c2[o] -= 1
                s2[v] = s2[o] = True
                walk(prefix + [int(e)], pv / cnt[v], c2, s2, k2)

    walk([], 1.0, np.diff(ptr).astype(np.int64), np.zeros(num_nodes, dtype=bool), np.zeros(T, dtype=bool))
    return probs


def chi_square_p(probs, sequences, min_expected=5.0):
    """p-value of a chi-square goodness-of-fit test of the observed ``sequences`` (iterable of tuples) against
    ``probs``; categories with expected counts below ``min_expected`` are pooled into one."""
    from scipy import stats
    seqs = [tuple(int(x) for x in s) for s in sequences]
    n = len(seqs)
    counts = {}
    for s in seqs:
        if s not in probs:
            raise AssertionError(f"sequence {s} has probability 0")
        counts[s] = counts.get(s, 0) + 1
    keys = sorted(probs, key=lambda k: -probs[k])
    obs, exp, pool_o, pool_e = [], [], 0, 0.0
    for k in keys:
        if probs[k] * n >= min_expected:
            obs.append(counts.get(k, 0))
            exp.append(probs[k] * n)
        else:
            pool_o += counts.get(k, 0)
            pool_e += probs[k] * n
    if pool_e > 0:
        obs.append(pool_o)
        exp.append(pool_e)
    exp = np.asarray(exp) * (n / np.sum(exp))
    return float(stats.chisquare(obs, exp).pvalue)


def tiny_graphs():
    """(name, triplets, num_nodes, B) of the enumeration cases."""
    path = [(0, 0, 1), (1, 0, 2), (2, 1, 3), (3, 0, 4)]
    star = [(0, 0, 1), (0, 1, 2), (3, 0, 0), (0, 2, 4), (5, 0, 0)]
    # a triangle with a self-loop on 1 and the triple (0, 0, 1) twice
    tri_loop = [(0, 0, 1), (1, 1, 2), (2, 0, 0), (1, 2, 1), (0, 0, 1)]
    # two components: once the first is exhausted no seen entity has an unpicked edge -> the [cnt > 0] draw
    two = [(0, 0, 1), (2, 0, 3), (3, 1, 4)]
    # entity ids 0, 2, 5, 6 unused
    unused = [(1, 0, 3), (3, 1, 4), (4, 0, 1), (7, 0, 3)]
    return [("path", path, 5, 3), ("star", star, 6, 3), ("triangle-selfloop-dup", tri_loop, 3, 3),
            ("two-components", two, 5, 3), ("unused-ids", unused, 8, 3)]

