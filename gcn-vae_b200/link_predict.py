"""Link prediction head and training driver with the reference's surface (kgvae/link_predict.py).

``LinkPredict`` keeps the constructor, ``forward`` / ``calc_score`` / ``regularization_loss`` /
``get_loss`` and the ``w_relation`` parameter.  ``main`` keeps the reference's flags and loop;
evaluation stays on the GPU (the reference moves the model to the CPU for it).
"""
import argparse
import time

import numpy as np
import torch
import torch.nn as nn

from . import datasets, ops, utils
from .model import KGVAE, RGCN


class LinkPredict(nn.Module):
    def __init__(self, model_class, in_dim, h_dim, num_rels, num_bases=-1, num_hidden_layers=1,
                 dropout=0, use_cuda=True, reg_param=0, kl_param=0, mmd_param=0, k=1, n_flows=0):
        super().__init__()
        kwargs = dict(num_nodes=in_dim, h_dim=h_dim, out_dim=h_dim, num_rels=num_rels * 2,
                      num_bases=num_bases, num_hidden_layers=num_hidden_layers, dropout=dropout,
                      use_self_loop=use_cuda, use_cuda=use_cuda)
        if model_class is KGVAE:          # the reference passes k/n_flows to RGCN too and crashes
            kwargs.update(k=k, n_flows=n_flows)
        self.encoder = model_class(**kwargs)
        self.reg_param, self.kl_param, self.mmd_param = reg_param, kl_param, mmd_param
        self.w_relation = nn.Parameter(torch.Tensor(num_rels, h_dim))
        self.use_cuda, self.k, self.n_flows = use_cuda, k, n_flows
        nn.init.xavier_uniform_(self.w_relation, gain=nn.init.calculate_gain("relu"))

    def grad_buckets(self, group=None, average=True, sharded=()):
        """parallel.GradBuckets over this model's parameters, cut in the order backward produces the gradients:
        decoder / prior / flows first, then the second and the first RelGraphConv, the entity embedding last
        (its gradient is complete only at the very end of backward).  ``sharded``: parameters that are NOT
        replicated (destination-partitioned training shards the embedding table) and are left out."""
        from . import parallel
        skip = {id(p) for p in sharded}
        enc = self.encoder
        named = dict(self.named_parameters())
        pick = lambda prefix: [p for n, p in named.items() if n.startswith(prefix) and p.requires_grad and id(p) not in skip]
        head = [p for n, p in named.items() if p.requires_grad and id(p) not in skip and
                not n.startswith(("encoder.rconv_layer_", "encoder.input_layer", "encoder.layers"))]
        order = [head, pick("encoder.rconv_layer_2"), pick("encoder.rconv_layer_1"), pick("encoder.layers"),
                 pick("encoder.input_layer")]
        params = [p for p in self.parameters() if p.requires_grad and id(p) not in skip]
        return parallel.GradBuckets(params, buckets=[b for b in order if b], group=group, average=average)

    def release_graph(self):
        """Detach the tensors the encoder caches between ``forward`` and ``get_loss`` (``z_mean``, ``z_sigma``, the
        flow's log-determinants - the reference keeps them as attributes, kgvae/model.py:113-123).  They hold the
        whole autograd graph of the last forward alive, and with it the parameters' gradient-accumulation nodes,
        which are bound to the stream they were created on."""
        enc = self.encoder
        for name in ("z_mean", "z_sigma", "log_det_sum", "flow_log_prob"):
            v = getattr(enc, name, None)
            if isinstance(v, torch.Tensor) and v.grad_fn is not None:
                setattr(enc, name, v.detach())

    def _flow_shift(self):
        if self.n_flows > 0 and isinstance(self.encoder, KGVAE):
            return self.encoder.get_flow_log_prob()
        return None

    def calc_score(self, embedding, triplets, shift=None):
        """DistMult score of each (s, r, o) row (link_predict.py:57-63)."""
        trip = ops.as_i32(triplets, embedding.device)
        return ops.DistMultScoreFn.apply(embedding, self.w_relation, trip, shift)

    def forward(self, g, h, r, norm):
        return self.encoder.forward(g, h, r, norm)

    def regularization_loss(self, embedding, n_valid=None):
        """``n_valid``: the mean over the first n_valid rows of ``embedding`` only (a padded node set)."""
        return ops.MeanSquareFn.apply(embedding, n_valid) + ops.MeanSquareFn.apply(self.w_relation)

    def get_loss(self, g, embed, triplets, labels):
        """(loss, predict_loss, kl, mmd) as in link_predict.py:71-92.  When ``g.n_valid`` is set (a sampled subgraph
        padded to a fixed node budget) the per-node terms - regulariser, KL, MMD - cover the valid rows only and the
        padding rows of z get exactly zero gradient."""
        if getattr(g, "partition", None) is not None:
            return self._get_loss_partitioned(g.partition, embed, triplets, labels)
        trip = ops.as_i32(triplets, embed.device)
        lab = torch.as_tensor(labels, dtype=torch.float32, device=embed.device)
        zero = lambda: torch.zeros(1, device=embed.device)
        enc = self.encoder
        nv = getattr(g, "n_valid", None)
        if isinstance(enc, KGVAE) and (embed.requires_grad or nv is not None):
            # pred + reg + KL in one autograd node: their gradients wrt z are combined in a single pass
            flp = enc.flow_log_prob if enc.n_flows > 0 else None
            head, predict_loss, reg_loss, kl_core = ops.LossHeadFn.apply(
                embed, enc.z_mean, enc.z_sigma, enc.z_pre, self.w_relation, trip, lab, self._flow_shift(),
                self.reg_param, self.kl_param, nv)
            # the reference adds None here when n_flows == 0 and crashes (SURVEY F5); None -> 0
            kl = (kl_core if flp is None else kl_core + flp) if self.kl_param > 0 else zero()
            mmd = enc.get_mmd(embed, nv) if self.mmd_param > 0 else zero()
            loss = head
            if self.kl_param > 0 and flp is not None:
                loss = loss + self.kl_param * flp
            if self.mmd_param > 0:
                loss = loss + self.mmd_param * mmd
            return loss, predict_loss, kl, mmd
        predict_loss = ops.DistMultBceFn.apply(embed, self.w_relation, trip, lab, self._flow_shift())
        reg_loss = self.regularization_loss(embed, nv)
        kl = self.encoder.get_kl(embed) if self.kl_param > 0 else zero()
        mmd = self.encoder.get_mmd(embed) if self.mmd_param > 0 else zero()
        loss = predict_loss + self.reg_param * reg_loss + self.kl_param * kl + self.mmd_param * mmd
        return loss, predict_loss, kl, mmd


    def _get_loss_partitioned(self, part, embed, triplets, labels):
        """Destination-partitioned form: ``embed`` holds this rank's rows of z, ``triplets`` (global
        ids) / ``labels`` are this rank's share of the scored triplets.  Every term is scaled so
        that the SUM over ranks of the returned loss is the reference's loss; gradients of
        replicated parameters are then summed over ranks (parallel.allreduce_sum_grads)."""
        from . import parallel
        dev = embed.device
        trip = ops.as_i32(triplets, dev)
        lab = torch.as_tensor(labels, dtype=torch.float32, device=dev)
        counts = torch.tensor([float(trip.shape[0])], device=dev)
        torch.distributed.all_reduce(counts, group=part.group)
        # the all-gather of z runs while the local terms (regulariser, KL) are computed; the reduce-scatter of dz is
        # started inside the decoder's forward pass (the fused kernel has the gradient then) and waited for in backward
        pending_z = parallel.allgather_rows_start(embed.detach(), part)
        frac = part.n_local / part.n_global
        reg_loss = ops.MeanSquareFn.apply(embed) * frac + ops.MeanSquareFn.apply(self.w_relation) / part.world_size
        zero = lambda: torch.zeros(1, device=dev)
        if self.kl_param > 0:
            kl = ops.KlMogFn.apply(embed, self.encoder.z_mean, self.encoder.z_sigma, self.encoder.z_pre) * frac
            if self.encoder.flow_log_prob is not None:
                kl = kl + self.encoder.flow_log_prob / part.world_size
        else:
            kl = zero()
        predict_loss = ops.PartitionedDistMultBceFn.apply(embed, self.w_relation, trip, lab, self._flow_shift(),
                                                          part, pending_z)
        predict_loss = predict_loss * (float(trip.shape[0]) / counts).reshape(())      # device scalar: no host sync
        if self.mmd_param > 0:            # every rank evaluates the same term on the same 200 + 200 rows
            mmd = self.encoder.get_mmd_partitioned(embed, part) / part.world_size
        else:
            mmd = zero()
        loss = predict_loss + self.reg_param * reg_loss + self.kl_param * kl + self.mmd_param * mmd
        return loss, predict_loss, kl, mmd


class CapturedTrainStep:
    """The train step of kgvae/link_predict.py:217-228 - edge index, forward, ``get_loss``, backward,
    ``clip_grad_norm_``, ``optimizer.step()`` - for inputs of FIXED shape (full-graph training, or any fixed
    number of nodes / edges / scored triplets), captured once into a CUDA graph and replayed.

    An eager step is ~150 kernel launches issued through autograd and ctypes; at 4-5 ms of GPU work per step
    the host cannot stay ahead of the device, and the GPU idles between kernels.  A replay is one launch: the
    step then costs what its kernels cost.  Everything in the step is stream-ordered device work (no host
    read-back, device-resident Adam step counters, Philox offsets advanced per replay by PyTorch), so the replay
    computes exactly what the eager step computes on the tensors in ``inputs``.

    ``example``: dict of device tensors ``node_id [n,1]``, ``src``/``dst``/``etype [E]`` (int32), ``norm [E,1]``,
    ``samples [S,3]`` (int32), ``labels [S]`` - their shapes are the captured shapes.  The optimizer must be
    ``capturable`` (``torch.optim.Adam(..., fused=True, capturable=True)``).  The ``warmup`` eager steps that
    precede the capture ARE train steps on ``example``.  ``step(**tensors)`` copies new inputs of the same shapes
    into place (device-to-device or from pinned host memory, stream-ordered), replays, and returns the loss
    tensor (device; read it with ``float()`` when needed).

    ``sampler``: an object whose ``sample()`` returns that dict with fixed shapes using only stream-ordered device
    work (``utils.FullBatchDeviceSampler``, ``utils.SampledDeviceSampler``): the draw is then captured too and
    ``step()`` - no arguments - is the whole iteration of the reference's loop (kgvae/link_predict.py:200-236): fresh
    edge sample (SampledDeviceSampler), fresh negatives, fresh graph split, edge index, forward, loss, backward, clip,
    Adam, in one replay (``example`` may be ``None``).  A sample with an ``n_valid`` entry (a node set padded to a
    fixed budget) sets ``Graph.n_valid``, which keeps the padding rows out of the loss.  A sampler with a
    ``before_replay()`` method has it called before every replay (the neighbourhood sampler refills its bank of edge
    samples there)."""

    FIELDS = ("node_id", "src", "dst", "etype", "norm", "samples", "labels")

    def __init__(self, model, optimizer, example, num_nodes, buckets=None, grad_norm=1.0, warmup=3, sampler=None):
        from . import _lib
        from .graph import Graph
        if not all(g.get("capturable", False) for g in optimizer.param_groups):
            raise RuntimeError("CapturedTrainStep: the optimizer must be constructed with capturable=True")
        dev = example["src"].device if example is not None else next(model.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("kgvae_b200: CapturedTrainStep needs CUDA tensors (no CPU fallback)")
        self._Graph = Graph
        self.model, self.optimizer, self.num_nodes, self.grad_norm = model, optimizer, int(num_nodes), grad_norm
        self.buckets = buckets if buckets is not None else model.grad_buckets()
        self.sampler = sampler
        self.inputs = None if sampler is not None else {k: example[k].clone() for k in self.FIELDS}
        self.predict_loss = self.kl = self.mmd = None
        # Warm-up and capture run on ONE side stream, and no autograd graph of an earlier step may be alive: a
        # parameter's gradient-accumulation node runs on the stream it was created on, and one left over from an
        # eager step on the default stream would make that stream wait on the capture (illegal).
        model.release_graph()
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        before, prof = _lib.launches, _lib.profile
        _lib.profile = None                   # no timing events inside a capture
        try:
            with torch.cuda.stream(side):     # lazy initialisation, optimizer state and allocator warm-up
                for _ in range(max(int(warmup), 1)):
                    self._eager()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            before = _lib.launches
            with torch.cuda.graph(self.graph, stream=side):
                self.loss = self._eager()
        finally:
            _lib.profile = prof
        self.launches_per_step = _lib.launches - before      # kernels of this library inside one replay

    def _eager(self):
        t = self.inputs if self.sampler is None else self.sampler.sample()
        g = self._Graph.from_device_edges(self.num_nodes, t["src"], t["dst"])
        g.n_valid = t.get("n_valid")
        self.buckets.zero()
        embed = self.model(g, t["node_id"], t["etype"], t["norm"])
        loss, self.predict_loss, self.kl, self.mmd = self.model.get_loss(g, embed, t["samples"], t["labels"])
        loss.backward()
        self.buckets.finish()
        self.buckets.clip_(self.grad_norm)
        self.optimizer.step()
        self.model.release_graph()
        return loss.detach()

    def close(self):
        """Release the captured graph and its memory pool (required before the process group is destroyed when the
        capture contains NCCL kernels)."""
        if self.graph is not None:
            torch.cuda.synchronize()
            self.graph.reset()
            self.graph = None

    def load(self, **tensors):
        if self.inputs is None:
            raise RuntimeError("CapturedTrainStep: this step draws its own inputs (sampler=...)")
        for k, v in tensors.items():
            self.inputs[k].copy_(v.view_as(self.inputs[k]), non_blocking=True)

    def step(self, **tensors):
        if tensors:
            self.load(**tensors)
        before = getattr(self.sampler, "before_replay", None)
        if before is not None:            # e.g. a bank of edge samples that refills between replays
            before()
        self.graph.replay()
        return self.loss

    __call__ = step


def node_norm_to_edge_norm(g, node_norm):
    """edge_norm[e] = node_norm[dst[e]] (link_predict.py:95-100)."""
    g = g.local_var()
    g.ndata["norm"] = node_norm
    g.apply_edges(lambda edges: {"norm": edges.dst["norm"]})
    return g.edata["norm"]


def _graph_inputs(graph, rel, norm, num_nodes, device):
    node_id = torch.arange(0, num_nodes, dtype=torch.long).view(-1, 1).to(device)
    rel_t = torch.from_numpy(rel).to(device)
    edge_norm = node_norm_to_edge_norm(graph, torch.from_numpy(norm).view(-1, 1)).to(device)
    return node_id, rel_t, edge_norm


def _validate(model, args, epoch, best_mrr, val_graph, val_node_id, val_rel, val_norm, valid_t):
    """Periodic validation with checkpoints (kgvae/link_predict.py:238-259); returns the best MRR so far."""
    model.eval()
    print("start eval")
    torch.save({"state_dict": model.state_dict(), "epoch": epoch}, args.model_state_file)
    with torch.no_grad():
        embed = model(val_graph, val_node_id, val_rel, val_norm)
    mrr = utils.calc_mrr(embed, model.w_relation, valid_t, hits=[1, 3, 10],
                         eval_bz=args.eval_batch_size, all_batches=False,
                         flow_log_prob=model._flow_shift())
    model.release_graph()
    if mrr < best_mrr:
        torch.save({"state_dict": model.state_dict(), "epoch": epoch}, args.model_state_file + "_latest")
    else:
        best_mrr = mrr
        torch.save({"state_dict": model.state_dict(), "epoch": epoch}, args.model_state_file)
    return best_mrr


def main(args):
    data = datasets.load_data(args.dataset)
    num_nodes, num_rels = data.num_nodes, data.num_rels
    train_data, valid_data, test_data = data.train, data.valid, data.test
    if not torch.cuda.is_available():
        raise RuntimeError("kgvae_b200 needs a CUDA device (no CPU fallback)")
    device = torch.device("cuda", max(args.gpu, 0))
    torch.cuda.set_device(device)

    model_class = KGVAE if args.model_class == "KGVAE" else RGCN
    model = LinkPredict(model_class=model_class, in_dim=num_nodes, h_dim=args.n_hidden,
                        num_rels=num_rels, num_bases=args.n_bases, num_hidden_layers=args.n_layers,
                        dropout=args.dropout, use_cuda=True, reg_param=args.regularization,
                        kl_param=args.kl_param, mmd_param=args.mmd_param, k=args.mog_k,
                        n_flows=args.n_flows).to(device)

    valid_t = torch.LongTensor(valid_data)
    val_graph, val_rel, val_norm = utils.build_test_graph(num_nodes, num_rels, valid_t)
    val_node_id, val_rel, val_norm = _graph_inputs(val_graph, val_rel, val_norm, num_nodes, device)
    adj_list, degrees = utils.get_adj_and_degrees(num_nodes, train_data)
    capture = bool(getattr(args, "capture_step", False))
    optimizer = torch.optim.Adam(model.parameters(), lr=args.lr, fused=True, capturable=capture)
    # gradients live in one flat buffer: zeroing is one memset, clipping one norm + one scale
    # (same arithmetic as optimizer.zero_grad() / clip_grad_norm_ of kgvae/link_predict.py:227,236)
    buckets = model.grad_buckets()
    forward_time, backward_time = [], []

    if args.test_mode:
        print("\nstart testing:")
        checkpoint = torch.load(args.model_state_file, map_location=device)
        test_t = torch.LongTensor(test_data)
        test_graph, test_rel, test_norm = utils.build_test_graph(num_nodes, num_rels, test_t)
        test_node_id, test_rel, test_norm = _graph_inputs(test_graph, test_rel, test_norm, num_nodes, device)
        model.eval()
        model.load_state_dict(checkpoint["state_dict"])
        print("Using best epoch: {}".format(checkpoint["epoch"]))
        with torch.no_grad():
            embed = model(test_graph, test_node_id, test_rel, test_norm)
        if args.generate:             # kgvae/link_predict.py:181-184: generation instead of ranking
            tails, scores = utils.generate(embed, model.w_relation, test_t, flow_log_prob=model._flow_shift(),
                                           out_path="result.txt")
            print(f"generated tails for {len(tails)} test queries -> result.txt")
            return tails
        return utils.calc_mrr(embed, model.w_relation, test_t, hits=[1, 3, 10],
                              eval_bz=args.eval_batch_size, all_batches=True,
                              flow_log_prob=model._flow_shift())

    print("start training...")
    epoch, best_mrr = 0, 0
    if args.load:
        print(f"Loading checkpoint file {args.model_state_file} for training")
        checkpoint = torch.load(args.model_state_file, map_location=device)
        model.load_state_dict(checkpoint["state_dict"])
        epoch = checkpoint["epoch"]

    train_dev = None
    captured = None
    bank = None                          # eager --device-sampler --edge-sampler neighbor: a bank of edge samples
    if capture:
        # full-graph training: every iteration scores all training triples with fresh negatives on a fresh graph
        # split - fixed shapes, so sampler + step are captured once and every iteration is one CUDA-graph replay.
        # Sampled subgraphs (--device-sampler): the node set is padded to a fixed budget, so their shapes are fixed too
        # Both edge samplers select every triple when B >= T, so FullBatchDeviceSampler serves both there
        full = args.graph_batch_size >= len(train_data)
        sampled = getattr(args, "device_sampler", False)
        if args.edge_sampler not in ("uniform", "neighbor"):
            raise ValueError("Sampler type must be either 'uniform' or 'neighbor'.")
        if not (full or sampled):
            raise RuntimeError("--capture-step needs full-batch sampling (--graph-batch-size >= the number of "
                               f"training triples, {len(train_data)}) or --device-sampler")
        model.train()
        train_dev = torch.from_numpy(np.asarray(train_data)).to(device)
        if full:
            sampler = utils.FullBatchDeviceSampler(train_dev, num_rels, args.negative_sample, args.graph_split_size)
        else:
            sampler = utils.SampledDeviceSampler(train_dev, args.graph_batch_size, args.graph_split_size, num_rels,
                                                 args.negative_sample, edge_sampler=args.edge_sampler)
        captured = CapturedTrainStep(model, optimizer, None, sampler.n, buckets=buckets, grad_norm=args.grad_norm,
                                     warmup=1, sampler=sampler)
        epoch += 1                       # the warm-up step that precedes the capture is a training step
    while True:
        model.train()
        epoch += 1
        if captured is not None:
            torch.cuda.synchronize()
            t0 = time.time()
            loss = captured.step()
            torch.cuda.synchronize()
            forward_time.append(time.time() - t0)          # the replay is forward + backward + update in one
            backward_time.append(0.0)
            print("Epoch {:04d} | Loss {:.4f} | Best MRR {:.4f} | pred_loss {:.4f} | kl {:.4f} | mmd {:.4f}".format(
                epoch, loss.item(), best_mrr, captured.predict_loss.item(), captured.kl.item(), captured.mmd.item()))
            if epoch % args.evaluate_every == 0:
                best_mrr = _validate(model, args, epoch, best_mrr, val_graph, val_node_id, val_rel, val_norm, valid_t)
            if epoch >= args.n_epochs:
                break
            continue
        if getattr(args, "device_sampler", False) and args.edge_sampler in ("uniform", "neighbor"):
            # opt-in: the same sampling procedure drawn on the GPU (not numpy's random stream)
            if train_dev is None:
                train_dev = torch.from_numpy(np.asarray(train_data)).to(device)
            picked = None
            if args.edge_sampler == "neighbor" and args.graph_batch_size < len(train_data):
                if bank is None:
                    bank = utils.NeighborEdgeBank(train_dev, num_nodes, args.graph_batch_size)
                picked = bank.next()
            g, node_id, edge_type, edge_norm, batch, labels = utils.generate_sampled_graph_and_labels_device(
                train_dev, args.graph_batch_size, args.graph_split_size, num_rels, args.negative_sample,
                picked=picked)
        else:
            g, node_id, edge_type, node_norm, batch, labels = utils.generate_sampled_graph_and_labels(
                train_data, args.graph_batch_size, args.graph_split_size, num_rels, adj_list, degrees,
                args.negative_sample, args.edge_sampler)
            node_id = torch.from_numpy(node_id).view(-1, 1).long().to(device)
            edge_type = torch.from_numpy(edge_type).to(device)
            edge_norm = node_norm_to_edge_norm(g, torch.from_numpy(node_norm).view(-1, 1)).to(device)
            batch, labels = torch.from_numpy(batch).to(device), torch.from_numpy(labels).to(device)

        torch.cuda.synchronize()
        t0 = time.time()
        embed = model(g, node_id, edge_type, edge_norm)
        loss, pred_loss, kl, mmd = model.get_loss(g, embed, batch, labels)
        torch.cuda.synchronize()
        t1 = time.time()
        loss.backward()
        buckets.finish()
        buckets.clip_(args.grad_norm)
        optimizer.step()
        torch.cuda.synchronize()
        t2 = time.time()
        forward_time.append(t1 - t0)
        backward_time.append(t2 - t1)
        print("Epoch {:04d} | Loss {:.4f} | Best MRR {:.4f} | pred_loss {:.4f} | kl {:.4f} | mmd {:.4f}".format(
            epoch, loss.item(), best_mrr, pred_loss.item(), kl.item(), mmd.item()))
        buckets.zero()

        if epoch % args.evaluate_every == 0:
            best_mrr = _validate(model, args, epoch, best_mrr, val_graph, val_node_id, val_rel, val_norm, valid_t)
        if epoch >= args.n_epochs:
            break

    print("training done")
    print("Mean forward time: {:4f}s".format(np.mean(forward_time)))
    print("Mean Backward time: {:4f}s".format(np.mean(backward_time)))
    return best_mrr


def build_parser():
    p = argparse.ArgumentParser(description="Link Prediction")
    p.add_argument("--dropout", type=float, default=0.2)
    p.add_argument("--n-hidden", type=int, default=500)
    p.add_argument("--gpu", type=int, default=-1)
    p.add_argument("--lr", type=float, default=1e-3)
    p.add_argument("--n-bases", type=int, default=100)
    p.add_argument("--n-layers", type=int, default=2)
    p.add_argument("--n-epochs", type=int, default=int(1e5))
    p.add_argument("-d", "--dataset", type=str, required=True)
    p.add_argument("--eval-batch-size", type=int, default=400)
    p.add_argument("--regularization", type=float, default=0.01)
    p.add_argument("--kl-param", type=float, default=1e-5)
    p.add_argument("--mmd-param", type=float, default=0)
    p.add_argument("--mog-k", type=int, default=10)
    p.add_argument("--n-flows", type=int, default=0)
    p.add_argument("--grad-norm", type=float, default=1.0)
    p.add_argument("--graph-batch-size", type=int, default=20000)
    p.add_argument("--graph-split-size", type=float, default=0.5)
    p.add_argument("--negative-sample", type=int, default=10)
    p.add_argument("--evaluate-every", type=int, default=200)
    p.add_argument("--edge-sampler", type=str, default="uniform")
    p.add_argument("--test-mode", type=bool, default=False)
    p.add_argument("--model-state-file", type=str, default="model_state.pth")
    p.add_argument("--model-class", type=str, default="KGVAE")
    p.add_argument("--load", type=bool, default=False)
    p.add_argument("--generate", type=bool, default=False)
    p.add_argument("--capture-step", action="store_true",
                   help="(new) full-graph training (--graph-batch-size >= the number of training triples), or sampled "
                        "subgraphs with --device-sampler (nodes padded to min(2 B, entities)): edge sample, negatives, "
                        "graph split, edge index, forward, loss, backward, clipping and Adam are captured once into a "
                        "CUDA graph and every iteration is one replay; one warm-up iteration precedes the capture")
    p.add_argument("--device-sampler", action="store_true",
                   help="(new) draw the edge sample (--edge-sampler uniform or neighbor), the negatives and the "
                        "graph split on the GPU; same procedure as the reference's host sampler, not its numpy random "
                        "stream.  The neighbour sampler draws a bank of samples per kernel launch")
    return p


if __name__ == "__main__":
    parsed = build_parser().parse_args()
    print(parsed)
    main(parsed)
