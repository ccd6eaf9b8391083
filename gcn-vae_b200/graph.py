"""Graph container with the slice of the ``dgl.DGLGraph`` surface the reference uses.

Call sites being served (reference): ``g = dgl.DGLGraph(); g.add_nodes(n); g.add_edges(src, dst)``
(kgvae/utils.py:141-148), ``g.in_degrees(range(n))`` (:129, link_predict.py:216),
``g.local_var()``, ``g.ndata[...]``, ``g.apply_edges(lambda edges: {...: edges.dst[...]})``,
``g.edata[...]`` (link_predict.py:95-100), ``g.number_of_nodes()``, ``len(g)``.

Beyond that surface the graph owns the device-side edge orderings (ops.GraphIndex) that the
message-passing kernels consume; they are built on first use for a given (etypes, norm) pair
and reused by both RelGraphConv layers and their backward passes.

``n_valid`` (default None): an int32 device tensor [1] when only the first n_valid nodes are real and the rest pad
a sampled subgraph to a fixed node budget (utils.SampledDeviceSampler); the loss terms then average over the valid
rows only.
"""
import numpy as np
import torch

from . import ops


class _EdgeView:
    def __init__(self, g):
        self.src = _Lazy(g.ndata, g._src_t)
        self.dst = _Lazy(g.ndata, g._dst_t)
        self.data = g.edata


class _Lazy:
    """edges.src[...] / edges.dst[...]: node data gathered at the edge end-points."""

    def __init__(self, frame, index_fn):
        self._frame, self._index_fn = frame, index_fn

    def __getitem__(self, key):
        val = self._frame[key]
        return val[self._index_fn(val.device)]


class Graph:
    def __init__(self):
        self._n = 0
        self._src = np.zeros(0, dtype=np.int64)
        self._dst = np.zeros(0, dtype=np.int64)
        self.ndata, self.edata = {}, {}
        self._dev_edges = {}     # device -> (src int32, dst int32)
        self._index = None       # (key, ops.GraphIndex)
        self.n_valid = None      # device int32 [1]: nodes past it are padding

    @classmethod
    def from_device_edges(cls, num_nodes, src, dst):
        """A graph whose edge list already lives on the GPU (int32 ``src`` / ``dst``): nothing is copied; the
        host-side queries pull the edges over on first use."""
        g = cls()
        g._n = int(num_nodes)
        g._dev_edges[src.device] = (src, dst)
        return g

    # ---- DGLGraph construction surface -------------------------------------------------
    def add_nodes(self, n):
        self._n += int(n)

    def add_edges(self, src, dst):
        to_np = lambda a: a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        self._src = np.concatenate([self._src, to_np(src).astype(np.int64).reshape(-1)])
        self._dst = np.concatenate([self._dst, to_np(dst).astype(np.int64).reshape(-1)])
        self._dev_edges.clear()
        self._index = None

    # ---- DGLGraph query surface ----------------------------------------------------------
    def _ensure_host(self):
        """Graphs built on the device (utils.generate_sampled_graph_and_labels_device, bench) carry only
        device edge lists: the host-side queries below pull them over once instead of answering for an
        empty graph."""
        if self._src.shape[0] == 0 and self._dev_edges:
            src, dst = next(iter(self._dev_edges.values()))
            self._src = src.detach().cpu().numpy().astype(np.int64)
            self._dst = dst.detach().cpu().numpy().astype(np.int64)

    def number_of_nodes(self):
        return self._n

    def number_of_edges(self):
        if self._src.shape[0] == 0 and self._dev_edges:
            return int(next(iter(self._dev_edges.values()))[0].numel())
        return int(self._src.shape[0])

    def __len__(self):
        return self._n

    def in_degrees(self, v=None):
        self._ensure_host()
        deg = torch.from_numpy(np.bincount(self._dst, minlength=self._n))
        return deg if v is None else deg[torch.as_tensor(list(v), dtype=torch.long)]

    def edges(self):
        self._ensure_host()
        return torch.from_numpy(self._src), torch.from_numpy(self._dst)

    def local_var(self):
        self._ensure_host()
        g = Graph.__new__(Graph)
        g._n, g._src, g._dst = self._n, self._src, self._dst
        g.ndata, g.edata = dict(self.ndata), dict(self.edata)
        g._dev_edges, g._index = self._dev_edges, self._index
        g.n_valid = self.n_valid
        return g

    def apply_edges(self, func):
        self.edata.update(func(_EdgeView(self)))

    # ---- device side --------------------------------------------------------------------
    def _src_t(self, device):
        return torch.from_numpy(self._src).to(device)

    def _dst_t(self, device):
        return torch.from_numpy(self._dst).to(device)

    def device_edges(self, device):
        device = torch.device(device)
        if device not in self._dev_edges:
            pin = lambda a: torch.from_numpy(a.astype(np.int32))
            self._dev_edges[device] = (pin(self._src).to(device, non_blocking=True),
                                       pin(self._dst).to(device, non_blocking=True))
        return self._dev_edges[device]

    def index_for(self, etypes, norm, num_etypes, node_major=False):
        """ops.GraphIndex for this edge list with the given per-edge types and norms
        (``node_major``: also build the dst-major / src-major lists in the same pass)."""
        key = (etypes.data_ptr(), etypes._version, etypes.device,
               None if norm is None else (norm.data_ptr(), norm._version), int(num_etypes))
        if self._index is not None and self._index[0] == key:
            return self._index[1]
        dev = etypes.device
        if dev.type != "cuda":
            raise RuntimeError("kgvae_b200: RelGraphConv needs CUDA tensors (no CPU fallback)")
        src, dst = self.device_edges(dev)
        if etypes.numel() != src.numel():
            raise RuntimeError(f"etypes has {etypes.numel()} entries for {src.numel()} edges")
        gi = ops.graph_index(src, dst, ops.as_i32(etypes), norm, self._n, int(num_etypes), node_major=node_major)
        # the keyed tensors are kept alive so their data_ptr cannot be recycled under the cache
        self._index = (key, gi, etypes, norm)
        return gi

    def adopt_index(self, gi, etypes, norm, num_etypes):
        """Install an index built elsewhere (ops.graph_build) for the given tensors."""
        key = (etypes.data_ptr(), etypes._version, etypes.device,
               None if norm is None else (norm.data_ptr(), norm._version), int(num_etypes))
        self._index = (key, gi, etypes, norm)


# the reference spells it dgl.DGLGraph
DGLGraph = Graph
