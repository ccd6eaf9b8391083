"""The kernel family kg_bdd_rel_fwd / kg_bdd_rel_bwd (rgcn_bdd_rel.cu) run for a block shape: the block-owner kernels
(rgcn_bdd_warp.cuh) for the benchmarked 5x5 / 5x10 blocks, the register-tile kernels (rgcn_bdd_tile.cuh) for blocks
whose sides divide by 4, 5, 8, 10, 20, 25 or 50, and the generic pair for every other shape.  The results of these block
shapes are checked against the oracle in test_gpu_ops.py.

The kernels are listed by torch.profiler in a child process: profiler sessions in the pytest process before
test_gpu_driver's captured train steps leave the later sessions of test_gpu_flow without kernel records."""
import json
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import kernels_run

from gcn_vae_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# name fragments of each family, found in demangled (bddtile::fwd_kernel<8, 4>) and mangled (_ZN7bddtile...) names
FAMILIES = {"bddwarp": ("bddwarp",), "bddtile": ("bddtile",),
            "generic": ("bdd_rel_scatter_generic", "bdd_rel_backward_generic")}
REMOVED = ("bdd_rel_scatter_kernel", "bdd_rel_backward_kernel")
SHAPES = [(100, 5, 5, "bddwarp"), (100, 5, 10, "bddwarp"),       # FB15k-237 / wikikg2 layers
          (25, 20, 20, "bddtile"), (25, 20, 40, "bddtile"),      # WN18 layers
          (125, 4, 4, "bddtile"), (62, 8, 8, "bddtile"), (50, 10, 10, "bddtile"), (31, 16, 16, "bddtile"),
          (160, 5, 5, "generic"),                                # past the block-owner kernels; no register tile fits
          (3, 7, 2, "generic")]


def layer_kernels(B, si, so):
    """Kernels one BddConvFn forward + backward launches on a small random graph."""
    n, e, r = 200, 3000, 7
    rng = np.random.default_rng(B * si * so)
    src, dst, et = rng.integers(0, n, e), rng.integers(0, n, e), rng.integers(0, r, e)
    norm = rng.random(e).astype(np.float32) + 0.1
    t = lambda a, dt: torch.from_numpy(a).to(dt).to(DEV)
    gi = ops.graph_index(t(src, torch.int32), t(dst, torch.int32), t(et, torch.int32), t(norm, torch.float32), n, r)
    g = torch.Generator(device=DEV).manual_seed(B * si * so)
    x = torch.randn(n, B * si, device=DEV, generator=g, requires_grad=True)
    weight = torch.randn(r, B * si * so, device=DEV, generator=g, requires_grad=True)
    gout = torch.randn(n, B * so, device=DEV, generator=g)
    return kernels_run(lambda: ops.BddConvFn.apply(x, weight, None, None, gi, B, 0, None).backward(gout))


@pytest.fixture(scope="module")
def kernels_by_shape():
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [__file__]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-4000:]
    return json.loads(proc.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("B,si,so,family", SHAPES)
def test_bdd_kernel_family(B, si, so, family, kernels_by_shape):
    names = kernels_by_shape[f"{B},{si},{so}"]
    for fam, fragments in FAMILIES.items():
        ran = [f for f in fragments if f in names]
        want = list(fragments) if fam == family else []
        assert ran == want, f"{B} x {si}x{so}: expected the {family} kernels, ran: {names}"
    assert not any(k in names for k in REMOVED), names


if __name__ == "__main__":
    print(json.dumps({f"{B},{si},{so}": layer_kernels(B, si, so) for B, si, so, _ in SHAPES}))
