"""The device neighbourhood-expansion edge sampler (kg_neighbor_sample, ``--edge-sampler neighbor``): bit-exact against
its numpy specification (tests/neighbor_mirror.py) on the same words, its law on the device, the bank that feeds the
training steps eagerly and inside a CUDA graph, the sampler's output and the driver."""
import os

import numpy as np
import pytest
import torch

import gcn_vae_b200 as K
import neighbor_mirror as M

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _device_words(words):
    return torch.from_numpy(np.ascontiguousarray(words).view(np.int32)).to(DEV)


def _launch(tri, n, words):
    """picks [K, B] and fallbacks [K] of one launch on ``words`` (uint32 [K, B, 8])."""
    t = torch.as_tensor(np.asarray(tri), device=DEV)
    adj_ptr, adj = K.ops.neighbor_adjacency(t, n)
    fb = torch.full((words.shape[0],), -1, dtype=torch.int32, device=DEV)
    picks = K.ops.neighbor_sample(adj_ptr, adj, n, words.shape[1], _device_words(words), fallbacks=fb)
    return picks.cpu().numpy(), fb.cpu().numpy()


def _expect_mirror(tri, n, words, picks, fallbacks, rows):
    for s in rows:
        ref, st = M.neighbor_sample(tri, n, words[s], return_state=True)
        assert np.array_equal(picks[s], ref), f"sample {s}: first difference at pick {np.argmax(picks[s] != ref)}"
        assert fallbacks[s] == st["fallbacks"], s


def _hub_graph(seed=0):
    """Entity 0 with degree > 1024, self-loops on it and on a few others, and a sparse rest."""
    rng = np.random.default_rng(seed)
    n = 300
    hub = np.stack([np.zeros(1000, int), rng.integers(0, 5, 1000), rng.integers(1, n, 1000)], 1)
    hub[::2, [0, 2]] = hub[::2, [2, 0]]                         # the hub at either end
    loops = np.array([[0, 1, 0]] * 40 + [[7, 2, 7], [9, 0, 9]])
    rest = np.stack([rng.integers(1, n, 400), rng.integers(0, 5, 400), rng.integers(1, n, 400)], 1)
    tri = np.concatenate([hub, loops, rest])[rng.permutation(1000 + 42 + 400)]
    assert np.bincount(tri[:, [0, 2]].reshape(-1))[0] > 1024
    return tri, n


# ---------------------------------------------------------------------------------------------------------------
# bit-exact against the mirror
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", M.tiny_graphs(), ids=lambda c: c[0])
def test_kernel_equals_mirror_on_tiny_graphs(case):
    _, tri, n, B = case
    for b in (1, B, len(tri)):
        words = M.random_words(np.random.default_rng(b), b, 64)
        picks, fb = _launch(tri, n, words)
        _expect_mirror(tri, n, words, picks, fb, range(64))


@pytest.mark.parametrize("B", ["1", "T/2", "T"])
def test_kernel_equals_mirror_on_the_toy_graph(B):
    data = K.datasets.synthetic_kg("toy", seed=1)
    T = len(data.train)
    b = {"1": 1, "T/2": T // 2, "T": T}[B]
    words = M.random_words(np.random.default_rng(3), b, 3)
    picks, fb = _launch(data.train, data.num_nodes, words)
    _expect_mirror(data.train, data.num_nodes, words, picks, fb, range(3))
    if b == T:
        assert all(np.array_equal(np.sort(p), np.arange(T)) for p in picks)


def test_kernel_equals_mirror_on_a_hub_with_self_loops():
    """A hub of degree > 1024 (the unpicked-entry scan walks more than 32 chunks) with 40 self-loops."""
    tri, n = _hub_graph()
    T = len(tri)
    for b in (T // 2, T):
        words = M.random_words(np.random.default_rng(b), b, 4)
        picks, fb = _launch(tri, n, words)
        _expect_mirror(tri, n, words, picks, fb, range(4))
        assert fb.min() > 0


def test_kernel_equals_mirror_on_every_sample_of_a_full_bank():
    data = K.datasets.synthetic_kg("toy", seed=2)
    B = 64
    k, _ = K.ops.neighbor_sample_plan(data.num_nodes, len(data.train), B)
    assert k >= 148
    words = M.random_words(np.random.default_rng(4), B, k)
    picks, fb = _launch(data.train, data.num_nodes, words)
    _expect_mirror(data.train, data.num_nodes, words, picks, fb, range(k))


@pytest.mark.parametrize("shape", [("FB15k-237", 0.0, 1.0, 20000), ("FB15k-237", 1.0, 1.0, 20000),
                                   ("wn18", 0.0, 1.0, 20000), ("wikikg2", 0.0, 0.001, 300)],
                         ids=["FB15k-237", "FB15k-237-skew1", "wn18", "wikikg2-global"])
def test_kernel_equals_mirror_at_benchmark_shapes(shape):
    """A whole bank at each shape; the first and the last sample are checked against the mirror.  The wikikg2
    entity count does not fit shared memory: its state lives in per-warp slabs of the workspace."""
    name, skew, scale, B = shape
    data = K.datasets.synthetic_kg(name, seed=0, skew=skew, scale=scale)
    T, n = len(data.train), data.num_nodes
    k, ws = K.ops.neighbor_sample_plan(n, T, B)
    assert (ws > 0) == (name == "wikikg2"), ws
    words = M.random_words(np.random.default_rng(7), B, k)
    picks, fb = _launch(data.train, n, words)
    _expect_mirror(data.train, n, words, picks, fb, [0, k - 1])
    assert all(len(np.unique(p)) == B for p in picks[:: max(1, k // 8)])


def test_two_launches_on_the_same_words_give_the_same_bits():
    data = K.datasets.synthetic_kg("FB15k-237", seed=0, skew=1.0)
    B = 5000
    k, _ = K.ops.neighbor_sample_plan(data.num_nodes, len(data.train), B)
    words = M.random_words(np.random.default_rng(8), B, k)
    a, fa = _launch(data.train, data.num_nodes, words)
    b, fb = _launch(data.train, data.num_nodes, words)
    assert np.array_equal(a, b) and np.array_equal(fa, fb)


def test_kernel_follows_the_exact_law():
    """One launch of more samples than one wave holds (the warps loop over samples) on a tiny graph, against the
    exact probability of every pick sequence under the reference's rule."""
    _, tri, n, B = M.tiny_graphs()[2]
    draws = 20000
    words = M.random_words(np.random.default_rng(9), B, draws)
    picks, fb = _launch(tri, n, words)
    assert M.chi_square_p(M.sequence_probabilities(tri, n, B), picks) > 1e-3
    _expect_mirror(tri, n, words, picks, fb, [0, draws - 1])


def test_bad_sizes_are_rejected():
    tri = torch.tensor([[0, 0, 1], [1, 0, 2]], device=DEV)
    adj_ptr, adj = K.ops.neighbor_adjacency(tri, 3)
    for b in (0, 3):
        with pytest.raises(RuntimeError, match="sample_size"):
            K.ops.neighbor_sample(adj_ptr, adj, 3, b, torch.zeros(1, b, 8, dtype=torch.int32, device=DEV))


# ---------------------------------------------------------------------------------------------------------------
# the bank
# ---------------------------------------------------------------------------------------------------------------
def _wn18_bank(B=16):
    data = K.datasets.synthetic_kg("wn18", seed=0)
    bank = K.utils.NeighborEdgeBank(torch.from_numpy(data.train).to(DEV), data.num_nodes, B)
    return data, bank


def test_bank_eager_consumes_rows_in_order_and_refills():
    data, bank = _wn18_bank()
    K_ = bank.K
    snaps, rows = [], []
    for i in range(2 * K_ + 3):
        before = bank.refills
        rows.append(bank.next().clone())
        if bank.refills != before:
            snaps.append(bank.bank.clone())
        assert bank.consumed == int(bank.cursor) == i % K_ + 1
    assert bank.refills == 3 and len(snaps) == 3
    expect = torch.cat(snaps)[:len(rows)]
    assert torch.equal(torch.stack(rows), expect)
    assert len({tuple(r.tolist()) for r in rows}) == len(rows)


def test_bank_inside_a_cuda_graph_replayed_past_the_bank():
    data, bank = _wn18_bank()
    K_ = bank.K
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        first = bank.next().clone()                 # eager warm-up: refill, row 0
    torch.cuda.current_stream().wait_stream(side)
    snaps = [bank.bank.clone()]
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        row = bank.next()
    assert bank.consumed == 1 and int(bank.cursor) == 1     # the capture ran nothing
    rows = [first]
    for _ in range(2 * K_ + 5):
        before = bank.refills
        bank.before_replay()
        if bank.refills != before:
            snaps.append(bank.bank.clone())
        graph.replay()
        rows.append(row.clone())
        assert bank.consumed == int(bank.cursor)
    assert bank.refills == 3
    expect = torch.cat(snaps)[:len(rows)]
    assert torch.equal(torch.stack(rows), expect)
    assert len({tuple(r.tolist()) for r in rows}) == len(rows)


# ---------------------------------------------------------------------------------------------------------------
# SampledDeviceSampler(edge_sampler="neighbor")
# ---------------------------------------------------------------------------------------------------------------
def test_sampled_sampler_with_neighbor_picks():
    """Relabelling, negatives, labels, split and n_valid are those of the bank row the sample consumed."""
    data = K.datasets.synthetic_kg("toy", seed=3)
    train, n_rel, B, rate = data.train, data.num_rels, 600, 5
    sm = K.utils.SampledDeviceSampler(torch.from_numpy(train).to(DEV), B, 0.5, n_rel, rate, edge_sampler="neighbor")
    with pytest.raises(ValueError):
        K.utils.SampledDeviceSampler(torch.from_numpy(train).to(DEV), B, 0.5, n_rel, rate, edge_sampler="other")
    torch.manual_seed(0)
    for _ in range(3):
        a = sm.sample()
        picked = sm.bank.bank[sm.bank.consumed - 1].cpu().numpy()
        assert len(np.unique(picked)) == B
        tri = train[picked]
        uniq, inv = np.unique(np.concatenate([tri[:, 0], tri[:, 2]]), return_inverse=True)
        n = int(a["n_valid"])
        node_id = a["node_id"].cpu().numpy().reshape(-1)
        smp = a["samples"].cpu().numpy()
        assert n == len(uniq) and np.array_equal(node_id[:n], uniq)
        assert np.array_equal(node_id[n:], np.arange(n, sm.n))
        pos = smp[:B]
        assert np.array_equal(pos, np.stack([inv[:B], tri[:, 1], inv[B:]], 1))
        neg = smp[B:].reshape(rate, B, 3)
        same_s, same_o = neg[:, :, 0] == pos[None, :, 0], neg[:, :, 2] == pos[None, :, 2]
        assert (same_s | same_o).all() and np.array_equal(neg[:, :, 1], np.broadcast_to(pos[None, :, 1], (rate, B)))
        assert smp[:, [0, 2]].min() >= 0 and smp[:, [0, 2]].max() < n
        lab = a["labels"].cpu().numpy()
        assert lab[:B].min() == 1 and lab[B:].max() == 0
        src, dst, et = (a[k].cpu().numpy() for k in ("src", "dst", "etype"))
        E = len(src) // 2
        assert E == B // 2 and np.array_equal(src[:E], dst[E:]) and np.array_equal(et[E:], et[:E] + n_rel)
        pos_set = {tuple(p) for p in pos}
        assert all((s, r, o) in pos_set for s, r, o in zip(src[:E], et[:E], dst[:E]))
        assert np.bincount(dst, minlength=sm.n)[n:].sum() == 0


# ---------------------------------------------------------------------------------------------------------------
# the driver
# ---------------------------------------------------------------------------------------------------------------
def _args(tmp_path, *extra):
    argv = ["--gpu", "0", "--n-hidden", "40", "--n-bases", "8", "--graph-batch-size", "600", "--negative-sample", "4",
            "--eval-batch-size", "64", "--mog-k", "4", "--n-flows", "0", "--kl-param", "1e-3", "--lr", "1e-2",
            "--edge-sampler", "neighbor", "--device-sampler",
            "--model-state-file", os.path.join(str(tmp_path), "model_state.pth"), *extra]
    return K.link_predict.build_parser().parse_args(argv)


def _losses(out):
    return [float(line.split("Loss")[1].split("|")[0]) for line in out.splitlines() if line.startswith("Epoch")]


def test_driver_eager_device_neighbor_sampler(tmp_path, capsys, monkeypatch):
    """--device-sampler --edge-sampler neighbor draws on the GPU: the host sampler is never called."""
    def no_host(*a, **k):
        raise AssertionError("host neighbour sampler called")
    monkeypatch.setattr(K.utils, "sample_edge_neighborhood", no_host)
    np.random.seed(0)
    torch.manual_seed(0)
    best = K.link_predict.main(_args(tmp_path, "-d", "toy", "--n-epochs", "6", "--evaluate-every", "3"))
    losses = _losses(capsys.readouterr().out)
    assert len(losses) == 6 and all(np.isfinite(losses)) and 0.0 < best <= 1.0


def test_driver_capture_step_with_the_device_neighbor_sampler(tmp_path, capsys):
    """--capture-step --device-sampler --edge-sampler neighbor on the wn18 shape: more iterations than one bank
    holds, so the bank refills between replays; training, validation and checkpoints as in the eager loop."""
    data = K.datasets.synthetic_kg("wn18", seed=0)
    k, _ = K.ops.neighbor_sample_plan(data.num_nodes, len(data.train), 600)
    epochs = k + 12
    np.random.seed(0)
    torch.manual_seed(0)
    args = _args(tmp_path, "-d", "wn18", "--capture-step", "--n-epochs", str(epochs), "--evaluate-every",
                 str(epochs // 2))
    best = K.link_predict.main(args)
    out = capsys.readouterr().out
    losses = _losses(out)
    assert len(losses) == epochs - 1 and all(np.isfinite(losses))
    assert "start eval" in out and "training done" in out and 0.0 <= best <= 1.0
    assert torch.load(args.model_state_file, map_location="cpu")["epoch"] in (epochs // 2 * 1, epochs // 2 * 2)
    with pytest.raises(ValueError):
        K.link_predict.main(_args(tmp_path, "-d", "toy", "--capture-step", "--edge-sampler", "other"))
