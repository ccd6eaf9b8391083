"""link_predict.main trains on the batches its sampling flags select, drawn in the order the samplers themselves draw
them.  For each mode the inputs of every train step (what ``forward`` and ``get_loss`` receive) are recorded and
compared bit for bit with a sequence rebuilt here from the same seeds by calling the sampler functions directly.
Under --capture-step only the warm-up step runs outside the CUDA graph: its draw is compared, and the losses, gradients
and parameters after the replays are compared with CapturedTrainStep driven directly."""
import os

import numpy as np
import pytest
import torch

import gcn_vae_b200 as K
from helpers import rel_err

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
SEED, EPOCHS = 0, 4


def _args(tmp_path, *extra):
    argv = ["-d", "toy", "--gpu", "0", "--n-hidden", "40", "--n-bases", "8", "--graph-batch-size", "600",
            "--negative-sample", "4", "--n-epochs", str(EPOCHS), "--evaluate-every", "1000", "--eval-batch-size", "64",
            "--mog-k", "4", "--n-flows", "1", "--kl-param", "1e-3",
            "--model-state-file", os.path.join(str(tmp_path), "model_state.pth"), *extra]
    return K.link_predict.build_parser().parse_args(argv)


@pytest.fixture
def run_main(monkeypatch):
    """``run_main(args)`` seeds numpy and torch, runs ``main`` and returns (batches, model, losses): the inputs of every
    train step that ran outside a CUDA-graph capture, the model ``main`` trained, and the loss of every replay."""
    LP = K.link_predict

    def run(args):
        batches, models, losses = [], [], []
        forward, get_loss, step = LP.LinkPredict.forward, LP.LinkPredict.get_loss, LP.CapturedTrainStep.step

        def rec_forward(self, g, h, r, norm):
            models[:] = [self]
            if self.training and not torch.cuda.is_current_stream_capturing():
                batches.append({"node_id": h.cpu(), "etype": r.cpu(), "norm": norm.cpu()})
            return forward(self, g, h, r, norm)

        def rec_get_loss(self, g, embed, triplets, labels):
            if not torch.cuda.is_current_stream_capturing():
                nv = getattr(g, "n_valid", None)
                batches[-1].update(samples=triplets.cpu(), labels=labels.cpu(),
                                   n_valid=None if nv is None else nv.cpu())
            return get_loss(self, g, embed, triplets, labels)

        def rec_step(self, **tensors):
            loss = step(self, **tensors)
            losses.append(float(loss))
            return loss

        with monkeypatch.context() as m:
            m.setattr(LP.LinkPredict, "forward", rec_forward)
            m.setattr(LP.LinkPredict, "get_loss", rec_get_loss)
            m.setattr(LP.CapturedTrainStep, "step", rec_step)
            np.random.seed(SEED)
            torch.manual_seed(SEED)
            LP.main(args)
        return batches, models[0], losses

    return run


def _record(node_id, etype, norm, samples, labels, n_valid=None):
    cpu = lambda t: None if t is None else t.detach().cpu()
    return {"node_id": cpu(node_id), "etype": cpu(etype), "norm": cpu(norm), "samples": cpu(samples),
            "labels": cpu(labels), "n_valid": cpu(n_valid)}


def _assert_same_batches(got, want):
    assert len(got) == len(want), (len(got), len(want))
    for i, (a, b) in enumerate(zip(got, want)):
        assert set(a) == set(b), (i, set(a), set(b))
        for key, ref in b.items():
            if ref is None:
                assert a[key] is None, (i, key)
            else:
                t = a[key]
                assert t.dtype == ref.dtype and t.shape == ref.shape and torch.equal(t, ref), (i, key)


def _model(args, data):
    """The model ``main`` builds for these arguments."""
    return K.LinkPredict(K.KGVAE, data.num_nodes, args.n_hidden, data.num_rels, num_bases=args.n_bases,
                         num_hidden_layers=args.n_layers, dropout=args.dropout, use_cuda=True,
                         reg_param=args.regularization, kl_param=args.kl_param, mmd_param=args.mmd_param,
                         k=args.mog_k, n_flows=args.n_flows).to(DEV).train()


def _host_batches(args, data):
    """utils.generate_sampled_graph_and_labels once per epoch on numpy's global stream."""
    np.random.seed(SEED)
    adj_list, degrees = K.utils.get_adj_and_degrees(data.num_nodes, data.train)
    out = []
    for _ in range(EPOCHS):
        g, node_id, etype, node_norm, samples, labels = K.utils.generate_sampled_graph_and_labels(
            data.train, args.graph_batch_size, args.graph_split_size, data.num_rels, adj_list, degrees,
            args.negative_sample, args.edge_sampler)
        out.append(_record(torch.from_numpy(node_id).view(-1, 1).long(), torch.from_numpy(etype),
                           K.node_norm_to_edge_norm(g, torch.from_numpy(node_norm).view(-1, 1)),
                           torch.from_numpy(samples), torch.from_numpy(labels)))
    return out


def _device_batches(args, data):
    """utils.generate_sampled_graph_and_labels_device once per epoch, the neighbourhood sampler's picks from a
    NeighborEdgeBank.  Each step's forward pass draws its dropout masks and noise from the same device generator
    between two samples, so the forward pass runs here too (its draws depend on the shapes only)."""
    torch.manual_seed(SEED)
    model = _model(args, data)
    train = torch.from_numpy(np.asarray(data.train)).to(DEV)
    bank = None
    if args.edge_sampler == "neighbor" and args.graph_batch_size < len(data.train):
        bank = K.utils.NeighborEdgeBank(train, data.num_nodes, args.graph_batch_size)
    out = []
    for _ in range(EPOCHS):
        g, node_id, etype, norm, samples, labels = K.utils.generate_sampled_graph_and_labels_device(
            train, args.graph_batch_size, args.graph_split_size, data.num_rels, args.negative_sample,
            picked=None if bank is None else bank.next())
        out.append(_record(node_id, etype, norm, samples, labels))
        with torch.no_grad():
            model(g, node_id, etype, norm)
        model.release_graph()
    return out


def _capturable_sampler(args, data):
    train = torch.from_numpy(np.asarray(data.train)).to(DEV)
    if args.graph_batch_size >= len(data.train):
        return K.utils.FullBatchDeviceSampler(train, data.num_rels, args.negative_sample, args.graph_split_size)
    return K.utils.SampledDeviceSampler(train, args.graph_batch_size, args.graph_split_size, data.num_rels,
                                        args.negative_sample, edge_sampler=args.edge_sampler)


EAGER = {"host-uniform": (), "host-neighbor": ("--edge-sampler", "neighbor"),
         "device-uniform": ("--device-sampler",),
         "device-neighbor": ("--device-sampler", "--edge-sampler", "neighbor")}     # batch 600 of 4000 triples


@pytest.mark.parametrize("mode", list(EAGER))
def test_eager_driver_trains_on_the_sampler_sequence(mode, tmp_path, run_main):
    args = _args(tmp_path, *EAGER[mode])
    data = K.datasets.load_data(args.dataset)
    assert args.graph_batch_size < len(data.train)
    batches, _, losses = run_main(args)
    assert losses == []
    want = _device_batches(args, data) if args.device_sampler else _host_batches(args, data)
    _assert_same_batches(batches, want)


CAPTURED = {"capture-full": ("--capture-step", "--graph-batch-size", "1000000"),
            "capture-sampled": ("--capture-step", "--device-sampler")}


@pytest.mark.parametrize("mode", list(CAPTURED))
def test_captured_driver_trains_on_the_sampler_sequence(mode, tmp_path, run_main):
    args = _args(tmp_path, *CAPTURED[mode])
    data = K.datasets.load_data(args.dataset)
    batches, model, losses = run_main(args)

    torch.manual_seed(SEED)
    t = _capturable_sampler(args, data).sample()
    _assert_same_batches(batches, [_record(t["node_id"], t["etype"], t["norm"], t["samples"], t["labels"],
                                           t.get("n_valid"))])
    assert (batches[0]["n_valid"] is None) == (mode == "capture-full")

    # the warm-up step is epoch 1, every later epoch one replay
    np.random.seed(SEED)
    torch.manual_seed(SEED)
    ref = _model(args, data)
    opt = torch.optim.Adam(ref.parameters(), lr=args.lr, fused=True, capturable=True)
    sampler = _capturable_sampler(args, data)
    cap = K.link_predict.CapturedTrainStep(ref, opt, None, sampler.n, buckets=ref.grad_buckets(),
                                           grad_norm=args.grad_norm, warmup=1, sampler=sampler)
    ref_losses = [float(cap.step()) for _ in range(EPOCHS - 1)]
    cap.close()
    assert len(losses) == EPOCHS - 1 and np.allclose(losses, ref_losses, rtol=1e-5), (losses, ref_losses)
    for (name, p), q in zip(model.named_parameters(), ref.parameters()):
        if p.requires_grad:
            assert rel_err(p.grad, q.grad) < 1e-3, name
        # Adam normalises the update: an element whose gradient is fp32 reduction noise moves by up to lr either way
        assert rel_err(p, q) < 1e-3, name
