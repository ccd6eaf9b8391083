"""Encoders with the reference's module surface (kgvae/model.py), running on sm_100a kernels.

``KGVAE`` keeps the constructor, the attributes callers read (``z_mean``, ``z_sigma``,
``flow_log_prob``, ``node_id``), the methods (``forward``, ``get_kl``, ``get_mmd``,
``get_flow_log_prob``, ``sample_z``) and the state-dict keys of the reference, so it drops in
behind ``LinkPredict`` and loads reference checkpoints.
"""
import random

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops, utils
from .flow_network import MADE, PermuteLayer
from .nn import RelGraphConv


class EmbeddingLayer(nn.Module):
    """Entity embedding lookup (kgvae/model.py:185-191)."""

    def __init__(self, num_nodes, h_dim):
        super().__init__()
        self.embedding = nn.Embedding(num_nodes, h_dim)

    def forward(self, g, h, r, norm):
        ids = ops.as_i32(h.reshape(-1), self.embedding.weight.device)
        return ops.EmbeddingFn.apply(self.embedding.weight, ids)


class KGVAE(nn.Module):
    """Embedding -> 2 x RelGraphConv(bdd, self-loop) -> mean/variance heads -> reparameterised
    sample -> optional IAF flow (kgvae/model.py:13-124)."""

    def __init__(self, num_nodes, h_dim, out_dim, num_rels, num_bases, num_hidden_layers=1,
                 dropout=0, use_self_loop=False, use_cuda=True, k=10, n_flows=0):
        super().__init__()
        self.num_nodes, self.h_dim, self.out_dim, self.num_rels = num_nodes, h_dim, out_dim, num_rels
        self.num_bases = None if num_bases < 0 else num_bases
        self.num_hidden_layers = num_hidden_layers
        self.dropout = dropout
        self.use_self_loop, self.use_cuda = use_self_loop, use_cuda
        self.k = k
        self.flow_log_prob = None
        self.preset_eps = None        # parity hook: noise to use instead of torch.randn
        self.build_encoder()
        self.z_pre = nn.Parameter(torch.randn(1, 2 * k, h_dim) / np.sqrt(k * h_dim))
        self.pi = nn.Parameter(torch.ones(k) / k, requires_grad=False)
        self.n_flows = n_flows
        if n_flows > 0:
            self.build_iaf()

    def build_iaf(self):
        blocks = []
        for _ in range(self.n_flows):
            blocks += [MADE(self.h_dim, self.h_dim, self.n_flows), PermuteLayer(self.h_dim)]
        self.nf = nn.Sequential(*blocks)

    def build_encoder(self):
        self.input_layer = EmbeddingLayer(self.num_nodes, self.h_dim)
        self.rconv_layer_1 = RelGraphConv(self.h_dim, self.h_dim, self.num_rels, "bdd",
                                          self.num_bases, activation=nn.ReLU(), self_loop=True,
                                          dropout=self.dropout)
        self.rconv_layer_2 = RelGraphConv(self.h_dim, self.h_dim * 2, self.num_rels, "bdd",
                                          self.num_bases, activation=nn.Identity(), self_loop=True,
                                          dropout=self.dropout)

    # ---- hot path ------------------------------------------------------------------------
    def forward(self, g, h, r, norm):
        self.node_id = h.squeeze()
        x = self.input_layer(g, h, r, norm)
        x = self.rconv_layer_1(g, x, r, norm)
        x = self.rconv_layer_2(g, x, r, norm)
        eps = self.preset_eps
        if eps is None:
            part = getattr(g, "partition", None)
            # partitioned: replicated parameters need the same seed on every rank, so the rows of different
            # ranks would otherwise draw identical noise - each rank samples from its own generator
            gen = None if part is None else part.noise_generator(x.device)
            eps = torch.randn((x.shape[0], self.h_dim), device=x.device, generator=gen)
        self.z_mean, self.z_sigma, z = ops.ReparamFn.apply(x, eps)
        if self.n_flows > 0:
            log_det_sum = None
            for flow in self.nf:
                z, log_det = flow.forward(z)
                if isinstance(flow, MADE):      # PermuteLayer contributes zeros
                    log_det_sum = log_det if log_det_sum is None else log_det_sum + log_det
            self.log_det_sum = log_det_sum
            part = getattr(g, "partition", None)
            n_valid = getattr(g, "n_valid", None)
            if n_valid is not None:   # a padded node set: the mean over the valid rows
                keep = ops.valid_rows(log_det_sum.shape[0], n_valid, log_det_sum.device)
                self.flow_log_prob = torch.where(keep, log_det_sum, 0.0).sum() / n_valid.reshape(()).to(torch.float32)
            elif part is None:
                self.flow_log_prob = torch.mean(log_det_sum)
            else:                     # mean over ALL nodes: local sums, summed over the ranks
                from . import parallel
                self.flow_log_prob = parallel.AllReduceSumFn.apply(log_det_sum.sum(), part.group) / part.n_global
        return z

    def get_kl(self, z):
        kl = ops.KlMogFn.apply(z, self.z_mean, self.z_sigma, self.z_pre)
        # the reference adds None here when n_flows == 0 and crashes (SURVEY F5); None -> 0
        return kl if self.flow_log_prob is None else kl + self.flow_log_prob

    def get_flow_log_prob(self):
        return self.flow_log_prob

    # ---- cold paths (plain tensor ops, as in the reference) ---------------------------------
    def compute_kernel(self, x, y):
        d = x.size(1)
        diff = x.unsqueeze(1) - y.unsqueeze(0)
        return torch.exp(-diff.pow(2).mean(2) / float(d))

    def get_mmd(self, z, n_valid=None):
        """``n_valid`` (device int32 [1], optional): only the first n_valid rows of z are nodes (a padded sampled
        subgraph); the 200 posterior rows are then distinct valid rows drawn on the device (kept in ``mmd_rows``),
        with no host read-back, so the term can be captured in a CUDA graph.  Like the unpadded path, which raises
        through ``random.sample``, it needs 200 nodes: fewer than 200 rows raise, and a draw with n_valid < 200 makes
        the term NaN (the host never reads n_valid, so the failure shows in the loss instead)."""
        m_mix, s_mix = utils.gaussian_parameters(self.z_pre, dim=1)
        num_sample = 200
        z_pri = utils.sample_gaussian(m_mix, s_mix, repeat=num_sample // self.k)
        if self.n_flows > 0:
            for flow in self.nf:
                z_pri, _ = flow.forward(z_pri)
        if n_valid is None:
            z_post = z[random.sample(range(z.shape[0]), num_sample)]
        else:                         # the first 200 of a random order of the valid rows (padding keys sort last)
            if z.shape[0] < num_sample:
                raise ValueError(f"get_mmd: {z.shape[0]} node rows, the MMD term needs {num_sample}")
            keys = torch.where(ops.valid_rows(z.shape[0], n_valid, z.device), torch.rand(z.shape[0], device=z.device),
                               2.0)
            self.mmd_rows = torch.argsort(keys)[:num_sample]
            z_post = z[self.mmd_rows]
        mmd = (self.compute_kernel(z_pri, z_pri).mean() + self.compute_kernel(z_post, z_post).mean()
               - 2 * self.compute_kernel(z_pri, z_post).mean())
        if n_valid is not None:       # padding rows entered z_post: no value rather than a wrong one
            mmd = torch.where(n_valid.reshape(()) >= num_sample, mmd, float("nan"))
        return mmd

    def get_mmd_partitioned(self, z_local, part):
        """get_mmd for destination-partitioned training (kgvae/model.py:89-102): the 200 posterior rows are
        drawn among ALL nodes (rank 0 draws, everyone receives the ids), each rank contributes the rows it
        owns and a differentiable sum over the ranks assembles them everywhere; the 200 prior samples use
        noise broadcast from rank 0, so every rank computes the same value (the caller divides by the world
        size: losses are summed over the ranks)."""
        import torch.distributed as dist
        from . import parallel
        num_sample = 200
        dev = z_local.device
        src_rank = dist.get_global_rank(part.group, 0) if part.group is not None else 0
        ids = torch.tensor(random.sample(range(part.n_global), num_sample), dtype=torch.int64, device=dev)
        dist.broadcast(ids, src=src_rank, group=part.group)
        mine = (ids >= part.lo) & (ids < part.hi)
        rows = torch.zeros((num_sample, z_local.shape[1]), dtype=z_local.dtype, device=dev)
        rows = rows.index_put((torch.nonzero(mine).reshape(-1),), z_local[(ids[mine] - part.lo)])
        z_post = parallel.AllReduceSumFn.apply(rows, part.group)
        m_mix, s_mix = utils.gaussian_parameters(self.z_pre, dim=1)
        repeat = num_sample // self.k
        sd = torch.cat([torch.sqrt(s_mix.squeeze())] * repeat, dim=0) if repeat > 1 else torch.sqrt(s_mix)
        mean = torch.cat([m_mix.squeeze()] * repeat, dim=0) if repeat > 1 else m_mix
        noise = torch.randn_like(sd)
        dist.broadcast(noise, src=src_rank, group=part.group)
        z_pri = mean + noise * sd
        if self.n_flows > 0:
            for flow in self.nf:
                z_pri, _ = flow.forward(z_pri)
        return (self.compute_kernel(z_pri, z_pri).mean() + self.compute_kernel(z_post, z_post).mean()
                - 2 * self.compute_kernel(z_pri, z_post).mean())

    def sample_z(self, batch):
        m, v = utils.gaussian_parameters(self.z_pre.squeeze(0), dim=0)
        idx = torch.distributions.categorical.Categorical(self.pi).sample((batch,))
        x = utils.sample_gaussian(m[idx], v[idx])
        if self.n_flows > 0:
            for flow in self.nf[::-1]:
                x, _ = flow.inverse(x)
        return x


class BaseRGCN(nn.Module):
    """Layer-stack base class (kgvae/model.py:134-182); base of EntityClassify (config 4)."""

    def __init__(self, num_nodes, h_dim, out_dim, num_rels, num_bases, num_hidden_layers=1,
                 dropout=0, use_self_loop=False, use_cuda=False):
        super().__init__()
        self.num_nodes, self.h_dim, self.out_dim, self.num_rels = num_nodes, h_dim, out_dim, num_rels
        self.num_bases = None if num_bases < 0 else num_bases
        self.num_hidden_layers, self.dropout = num_hidden_layers, dropout
        self.use_self_loop, self.use_cuda = use_self_loop, use_cuda
        self.build_model()

    def build_model(self):
        self.layers = nn.ModuleList()
        first = self.build_input_layer()
        if first is not None:
            self.layers.append(first)
        for idx in range(self.num_hidden_layers):
            self.layers.append(self.build_hidden_layer(idx))
        last = self.build_output_layer()
        if last is not None:
            self.layers.append(last)

    def build_input_layer(self):
        return None

    def build_hidden_layer(self, idx):
        raise NotImplementedError

    def build_output_layer(self):
        return None

    def forward(self, g, h, r, norm):
        for layer in self.layers:
            h = layer(g, h, r, norm)
        return h

    def get_kl(self, z):
        return torch.zeros(1, device=z.device)


class RGCN(BaseRGCN):
    """Non-variational RGCN encoder (kgvae/model.py:203-211)."""

    def build_input_layer(self):
        return EmbeddingLayer(self.num_nodes, self.h_dim)

    def build_hidden_layer(self, idx):
        act = F.relu if idx < self.num_hidden_layers - 1 else None
        return RelGraphConv(self.h_dim, self.h_dim, self.num_rels, "bdd", self.num_bases,
                            activation=act, self_loop=True, dropout=self.dropout)
