"""link_predict.main on two GPUs, as ``torchrun --nproc-per-node 2`` runs it: the driver joins the process group the
environment describes, trains one replica per GPU on distinct batches, shards validation, --test-mode and --generate
over the entities and tears the group down.  Needs 2 CUDA devices (skipped otherwise); NCCL over NVLink.

Each spawned rank records what ``forward`` / ``get_loss`` receive (as tests/test_gpu_driver_batches.py does), the
embeddings and results of the evaluation calls and every checkpoint write; the checks run in the ranks (against a
sequence rebuilt from the seed derivation of ``link_predict.rank_seeds``) and here (against single-GPU calls)."""
import builtins
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
WORLD, SEED, EPOCHS = 2, 0, 3


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _args(K, tmp, *extra):
    argv = ["-d", "toy", "--n-hidden", "40", "--n-bases", "8", "--graph-batch-size", "600",
            "--negative-sample", "4", "--n-epochs", str(EPOCHS), "--evaluate-every", "1000", "--eval-batch-size", "64",
            "--mog-k", "4", "--n-flows", "1", "--kl-param", "1e-3",
            "--model-state-file", os.path.join(tmp, "model_state.pth"), *extra]
    return K.link_predict.build_parser().parse_args(argv)


MODES = {"host-uniform": (), "device-uniform": ("--device-sampler",),
         "device-neighbor": ("--device-sampler", "--edge-sampler", "neighbor"),
         "capture-full": ("--capture-step", "--graph-batch-size", "1000000"),
         "capture-sampled": ("--capture-step", "--device-sampler")}


class _Recorder:
    """Wraps the driver's entry points inside one rank: the train-step inputs, the encoder noise, the first
    parameters, the evaluation / generation calls, checkpoint writes and result.txt opens."""

    def __init__(self, K):
        self.K, self.saved = K, []
        LP, U = K.link_predict, K.utils
        self.orig = {"forward": LP.LinkPredict.forward, "get_loss": LP.LinkPredict.get_loss,
                     "reparam": K.ops.ReparamFn.apply, "calc_mrr": U.calc_mrr, "generate": U.generate,
                     "save": torch.save, "open": builtins.open}
        rec = self

        def forward(self_, g, h, r, norm):
            rec.model = self_
            if self_.training and not torch.cuda.is_current_stream_capturing():
                if rec.init is None:
                    rec.init = {k: v.detach().cpu().clone() for k, v in self_.state_dict().items()}
                src, dst = g.device_edges(h.device)
                rec.batches.append({"node_id": h.cpu(), "etype": r.cpu(), "norm": norm.cpu(), "src": src.cpu(),
                                    "dst": dst.cpu(), "n": g.number_of_nodes()})
            return rec.orig["forward"](self_, g, h, r, norm)

        def get_loss(self_, g, embed, triplets, labels):
            if self_.training and not torch.cuda.is_current_stream_capturing():
                nv = getattr(g, "n_valid", None)
                rec.batches[-1].update(samples=triplets.cpu(), labels=labels.cpu(),
                                       n_valid=None if nv is None else nv.cpu())
            return rec.orig["get_loss"](self_, g, embed, triplets, labels)

        def reparam(x, eps):
            if torch.is_grad_enabled() and not torch.cuda.is_current_stream_capturing():
                rec.eps.append(eps.cpu())
            return rec.orig["reparam"](x, eps)

        def calc_mrr(embedding, w, test_triplets, **kw):
            kw["return_ranks"] = True
            mrr, ranks = rec.orig["calc_mrr"](embedding, w, test_triplets, **kw)
            shift = kw.get("flow_log_prob")
            rec.evals.append({"emb": embedding.cpu(), "w": w.detach().cpu(), "test": test_triplets.cpu(),
                              "shift": None if shift is None else shift.detach().cpu().reshape(()),
                              "eval_bz": kw["eval_bz"], "all_batches": kw["all_batches"],
                              "filtered": kw.get("filter_index") is not None, "sharded": kw.get("sharded"),
                              "ranks": ranks.cpu(), "mrr": mrr})
            return mrr

        def generate(embedding, w, test_triplets, **kw):
            tails, score = rec.orig["generate"](embedding, w, test_triplets, **kw)
            shift = kw.get("flow_log_prob")
            rec.gens.append({"emb": embedding.cpu(), "w": w.detach().cpu(), "test": test_triplets.cpu(),
                             "shift": None if shift is None else shift.detach().cpu().reshape(()),
                             "filtered": kw.get("filter_index") is not None, "tails": tails.cpu(),
                             "score": score.cpu()})
            return tails, score

        def save(obj, f, *a, **kw):
            rec.saved.append(str(f))
            return rec.orig["save"](obj, f, *a, **kw)

        def open_(file, mode="r", *a, **kw):
            if str(file).endswith("result.txt") and "w" in mode:
                rec.result_opens += 1
            return rec.orig["open"](file, mode, *a, **kw)

        self.repl = {(LP.LinkPredict, "forward"): forward, (LP.LinkPredict, "get_loss"): get_loss,
                     (K.ops.ReparamFn, "apply"): reparam, (U, "calc_mrr"): calc_mrr, (U, "generate"): generate,
                     (torch, "save"): save, (builtins, "open"): open_}

    def run(self, args):
        self.batches, self.eps, self.evals, self.gens, self.init, self.model = [], [], [], [], None, None
        self.result_opens = 0
        saved = {key: getattr(*key) for key in self.repl}
        for (obj, name), fn in self.repl.items():
            setattr(obj, name, fn)
        try:
            np.random.seed(SEED)
            torch.manual_seed(SEED)
            return self.K.link_predict.main(args)
        finally:
            for (obj, name), fn in saved.items():
                setattr(obj, name, fn)


def _rebuilt_batches(K, args, data, dev, rank):
    """The batches rank ``rank`` must draw: the samplers called directly after the seed derivation of rank_seeds."""
    np.random.seed(SEED)
    torch.manual_seed(SEED)
    model = K.LinkPredict(K.KGVAE, data.num_nodes, args.n_hidden, data.num_rels, num_bases=args.n_bases,
                          num_hidden_layers=args.n_layers, dropout=args.dropout, use_cuda=True,
                          reg_param=args.regularization, kl_param=args.kl_param, mmd_param=args.mmd_param,
                          k=args.mog_k, n_flows=args.n_flows).to(dev).train()
    K.link_predict.rank_seeds(rank, WORLD)
    train = torch.from_numpy(np.asarray(data.train)).to(dev)
    out = []
    if args.capture_step:
        if args.graph_batch_size >= len(data.train):
            s = K.utils.FullBatchDeviceSampler(train, data.num_rels, args.negative_sample, args.graph_split_size)
        else:
            s = K.utils.SampledDeviceSampler(train, args.graph_batch_size, args.graph_split_size, data.num_rels,
                                             args.negative_sample, edge_sampler=args.edge_sampler)
        t = s.sample()
        return [{"node_id": t["node_id"].cpu(), "etype": t["etype"].cpu(), "samples": t["samples"].cpu()}]
    if not args.device_sampler:
        adj_list, degrees = K.utils.get_adj_and_degrees(data.num_nodes, data.train)
        for _ in range(EPOCHS):
            g, node_id, etype, node_norm, samples, labels = K.utils.generate_sampled_graph_and_labels(
                data.train, args.graph_batch_size, args.graph_split_size, data.num_rels, adj_list, degrees,
                args.negative_sample, args.edge_sampler)
            out.append({"node_id": torch.from_numpy(node_id).view(-1, 1).long(), "etype": torch.from_numpy(etype),
                        "samples": torch.from_numpy(samples)})
        return out
    bank = None
    if args.edge_sampler == "neighbor":
        bank = K.utils.NeighborEdgeBank(train, data.num_nodes, args.graph_batch_size)
    for _ in range(EPOCHS):
        g, node_id, etype, norm, samples, labels = K.utils.generate_sampled_graph_and_labels_device(
            train, args.graph_batch_size, args.graph_split_size, data.num_rels, args.negative_sample,
            picked=None if bank is None else bank.next())
        out.append({"node_id": node_id.cpu(), "etype": etype.cpu(), "samples": samples.cpu()})
        with torch.no_grad():                     # the forward pass draws noise and dropout masks between samples
            model(g, node_id, etype, norm)
        model.release_graph()
    return out


def _same(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)


def _worker(rank, ports, tmp, out):
    import gcn_vae_b200 as K
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    os.chdir(tmp)
    rec = _Recorder(K)
    data = K.datasets.load_data("toy")
    res = {}
    port = iter(ports)

    def launch(args):
        """main as under torchrun: the driver creates (and must destroy) the process group."""
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(next(port)), WORLD_SIZE=str(WORLD),
                          RANK=str(rank), LOCAL_RANK=str(rank))
        try:
            return rec.run(args)
        finally:
            assert not dist.is_initialized()

    # sampling modes: distinct per rank, and the documented derivation
    for mode, extra in MODES.items():
        args = _args(K, tmp, *extra)
        launch(args)
        got = rec.batches
        want = _rebuilt_batches(K, args, data, dev, rank)
        assert len(got) == len(want), (mode, len(got), len(want))
        for i, (a, b) in enumerate(zip(got, want)):
            for key, ref in b.items():
                assert _same(a[key], ref), (mode, i, key)
        res[mode] = [{k: b[k] for k in ("node_id", "samples")} for b in got]

    # parameters after EPOCHS steps (no dropout): the recorded inputs and noise replay on one GPU in the test
    args = _args(K, tmp, "--device-sampler", "--dropout", "0")
    launch(args)
    res["train"] = {"init": rec.init, "batches": rec.batches, "eps": rec.eps,
                    "final": {k: v.detach().cpu() for k, v in rec.model.state_dict().items()}}

    # validation (raw and filtered) with checkpoints, then --test-mode and --generate
    launch(_args(K, tmp, "--evaluate-every", "1", "--filtered"))
    res["valid"] = rec.evals
    res["saved"] = rec.saved
    launch(_args(K, tmp, "--test-mode", "1", "--filtered"))
    res["test"] = rec.evals
    for extra in ((), ("--filtered",)):
        tails = launch(_args(K, tmp, "--test-mode", "1", "--generate", "1", *extra))
        res["gen" + "".join(extra)] = (rec.gens, tails.cpu(), rec.result_opens)

    # main raising inside its process group: the group is still destroyed (launch asserts it)
    try:
        launch(_args(K, tmp, "--edge-sampler", "bogus"))
        res["raised"] = False
    except ValueError:
        res["raised"] = True

    # a caller's process group is used and left alive
    for k in ("WORLD_SIZE", "RANK", "LOCAL_RANK"):
        os.environ.pop(k, None)
    os.environ["MASTER_PORT"] = str(next(port))
    dist.init_process_group("nccl", rank=rank, world_size=WORLD, device_id=dev)
    try:
        mrr = rec.run(_args(K, tmp, "--n-epochs", "1", "--evaluate-every", "1"))
        res["caller_group_alive"] = dist.is_initialized()
        res["caller_mrr"] = mrr
    finally:
        dist.destroy_process_group()
    out[rank] = res


def test_driver_on_two_gpus(tmp_path):
    if torch.cuda.device_count() < WORLD:
        pytest.skip("needs 2 GPUs")
    import gcn_vae_b200 as K
    from helpers import rel_err
    ports = [_free_port() for _ in range(16)]
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(ports, str(tmp_path), out), nprocs=WORLD, join=True)
        res = [dict(out[r]) for r in range(WORLD)]
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)

    # the two ranks train on different batches
    for mode in MODES:
        a, b = res[0][mode], res[1][mode]
        assert all(not (_same(x["node_id"], y["node_id"]) and _same(x["samples"], y["samples"]))
                   for x, y in zip(a, b)), mode

    # parameters: identical on both ranks, and a one-process replay that averages the ranks' gradients
    t0, t1 = res[0]["train"], res[1]["train"]
    for k, v in t0["final"].items():
        assert _same(v, t1["final"][k]), k
    for k, v in t0["init"].items():
        assert _same(v, t1["init"][k]), k
    args = _args(K, str(tmp_path), "--device-sampler", "--dropout", "0")
    data = K.datasets.load_data("toy")
    ref = K.LinkPredict(K.KGVAE, data.num_nodes, args.n_hidden, data.num_rels, num_bases=args.n_bases,
                        num_hidden_layers=args.n_layers, dropout=0.0, use_cuda=True, reg_param=args.regularization,
                        kl_param=args.kl_param, mmd_param=args.mmd_param, k=args.mog_k, n_flows=args.n_flows).to(dev)
    ref.load_state_dict({k: v.to(dev) for k, v in t0["init"].items()})
    ref.train()
    opt = torch.optim.Adam(ref.parameters(), lr=args.lr, fused=True)
    buckets = ref.grad_buckets()
    assert len(t0["batches"]) == len(t1["batches"]) == EPOCHS and len(t0["eps"]) == EPOCHS
    for i in range(EPOCHS):
        grads = []
        for t in (t0, t1):
            b = t["batches"][i]
            buckets.zero()
            ref.encoder.preset_eps = t["eps"][i].to(dev)
            g = K.Graph.from_device_edges(b["n"], b["src"].to(dev), b["dst"].to(dev))
            embed = ref(g, b["node_id"].to(dev), b["etype"].to(dev), b["norm"].to(dev))
            loss = ref.get_loss(g, embed, b["samples"].to(dev), b["labels"].to(dev))[0]
            loss.backward()
            ref.release_graph()
            grads.append(buckets.flat.clone())
        buckets.flat.copy_((grads[0] + grads[1]) / 2)
        buckets.clip_(args.grad_norm)
        opt.step()
    for name, p in ref.state_dict().items():
        assert rel_err(t0["final"][name].to(dev), p) <= 1e-5, name

    # sharded ranks equal single-GPU calc_mrr on the broadcast embedding; every rank agrees
    fi = K.utils.FilterIndex(np.concatenate([data.train, data.valid, data.test]), data.num_nodes, data.num_rels, dev)
    for key, n_calls in (("valid", 2 * EPOCHS), ("test", 2)):
        ev0, ev1 = res[0][key], res[1][key]
        assert len(ev0) == len(ev1) == n_calls and [e["filtered"] for e in ev0] == [False, True] * (n_calls // 2)
        for e0, e1 in zip(ev0, ev1):
            assert e0["sharded"] and _same(e0["emb"], e1["emb"]) and _same(e0["ranks"], e1["ranks"])
            assert e0["mrr"] == e1["mrr"]
            _, want = K.utils.calc_mrr(e0["emb"].to(dev), e0["w"].to(dev), e0["test"].to(dev), eval_bz=e0["eval_bz"],
                                       all_batches=e0["all_batches"], verbose=False, return_ranks=True,
                                       flow_log_prob=None if e0["shift"] is None else e0["shift"].to(dev),
                                       filter_index=fi if e0["filtered"] else None)
            assert torch.equal(e0["ranks"], want.cpu()), key

    # generation: bit-equal to single-GPU generate, result.txt written once
    for key in ("gen", "gen--filtered"):
        (g0, tails0, opens0), (g1, tails1, opens1) = res[0][key], res[1][key]
        assert opens0 == 1 and opens1 == 0 and _same(tails0, tails1)
        e = g0[0]
        assert _same(e["emb"], g1[0]["emb"]) and _same(e["score"], g1[0]["score"])
        want_t, want_s = K.utils.generate(e["emb"].to(dev), e["w"].to(dev), e["test"].to(dev),
                                          flow_log_prob=None if e["shift"] is None else e["shift"].to(dev),
                                          filter_index=fi if e["filtered"] else None)
        assert torch.equal(e["tails"], want_t.cpu()) and torch.equal(e["score"], want_s.cpu()), key
    assert (tmp_path / "result.txt").exists()

    # checkpoints: rank 0 only; teardown on an exception; a caller's group stays alive
    assert res[0]["saved"] and not res[1]["saved"]
    assert res[0]["raised"] and res[1]["raised"]
    assert res[0]["caller_group_alive"] and res[1]["caller_group_alive"]
    assert res[0]["caller_mrr"] == res[1]["caller_mrr"]
