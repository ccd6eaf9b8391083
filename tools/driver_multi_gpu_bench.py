"""Measurements of the multi-GPU link-prediction driver (one JSON document on stdout, or --out FILE).

  driver    ``link_predict`` under ``torchrun --nproc-per-node N`` at the FB15k-237 shape, N in --gpus: mean iteration
            time (rank 0's "Mean forward time" line) for ``--capture-step --device-sampler`` and full-graph
            ``--capture-step``
  eval      sharded ``calc_mrr`` (the --test-mode ranking, raw and filtered) and ``generate`` (k = 10, raw and
            filtered) on a random embedding of the FB15k-237 shape, at each N (this script re-run under torchrun)
  topk      unsharded kg_distmult_topk / _filtered of this tree against a second build (--parent-lib, e.g. the parent
            commit's libkgvae_b200.so), alternated on one card, outputs compared bit for bit
  bench     ``bench.py --gpus 1`` of this tree and of --parent-tree, alternated

The card name and power limit are read in the same run and stored with the numbers."""
import argparse
import ctypes
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpus": len(q), "cards": q}


def _torchrun(n, argv, cwd=ROOT, timeout=1800):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={n}", *argv]
    p = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True, timeout=timeout)
    if p.returncode != 0:
        raise RuntimeError(f"{cmd} failed:\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}")
    return p.stdout


def driver(ns, epochs):
    modes = {"capture-sampled": ["--capture-step", "--device-sampler", "--graph-batch-size", "20000"],
             "capture-full": ["--capture-step", "--graph-batch-size", "1000000"]}
    out = {}
    for name, extra in modes.items():
        for n in ns:
            with_tmp = os.path.join("/tmp", f"driver_bench_{os.getpid()}_{name}_{n}.pth")
            log = _torchrun(n, ["-m", "gcn_vae_b200.link_predict", "-d", "FB15k-237", "--n-epochs", str(epochs),
                                "--evaluate-every", str(10 ** 9), "--model-state-file", with_tmp, *extra])
            t = float(re.search(r"Mean forward time: ([0-9.]+)s", log).group(1))
            out[f"{name}/N={n}"] = {"iteration_ms": t * 1e3, "epochs": epochs}
    return out


def eval_worker(reps):
    """Run under torchrun: time sharded calc_mrr / generate on every rank; rank 0 prints one JSON line."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import gcn_vae_b200 as K
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    try:
        data = K.datasets.load_data("FB15k-237")
        g = torch.Generator().manual_seed(0)
        emb = torch.randn(data.num_nodes, 500, generator=g).to(dev)
        w = torch.randn(data.num_rels, 500, generator=g).to(dev)
        test = torch.from_numpy(data.test).to(dev)
        fi = K.utils.FilterIndex(np.concatenate([data.train, data.valid, data.test]), data.num_nodes, data.num_rels,
                                 dev)
        sharded = world > 1
        calls = {
            "test_mode_raw": lambda: K.utils.calc_mrr(emb, w, test, eval_bz=400, verbose=False, sharded=sharded),
            "test_mode_filtered": lambda: K.utils.calc_mrr(emb, w, test, eval_bz=400, verbose=False, filter_index=fi,
                                                           sharded=sharded),
            "generate_k10_raw": lambda: K.utils.generate(emb, w, test, topk=10, sharded=sharded),
            "generate_k10_filtered": lambda: K.utils.generate(emb, w, test, topk=10, filter_index=fi,
                                                              sharded=sharded)}
        res = {}
        for name, fn in calls.items():
            fn()
            ts = []
            for _ in range(reps):
                if sharded:
                    dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            res[name] = {"median_ms": float(np.median(ts)), "min_ms": float(min(ts))}
        if int(os.environ.get("RANK", "0")) == 0:
            print("EVAL " + json.dumps(res), flush=True)
    finally:
        if world > 1:
            dist.destroy_process_group()


def evals(ns, reps):
    out = {}
    for n in ns:
        log = _torchrun(n, [os.path.abspath(__file__), "--eval-worker", "--reps", str(reps)])
        out[f"N={n}"] = json.loads(log.split("EVAL ", 1)[1].splitlines()[0])
    return out


def topk_vs(parent_lib, rounds, reps):
    import numpy as np
    import torch
    import gcn_vae_b200 as K
    L = K._lib
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    old = ctypes.CDLL(parent_lib)
    _P, _I, _Z = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
    old.kg_distmult_topk.argtypes = [_P, _P, _P, _P, _I, _I, _I, _P, _I, _P, _Z, _P, _P, _P]
    old.kg_distmult_topk_filtered.argtypes = [_P, _P, _P, _P, _I, _I, _I, _P, _I, _P, _P, _P, _Z, _P, _P, _P]
    old.kg_distmult_topk_workspace_bytes.restype = _Z
    old.kg_distmult_topk_workspace_bytes.argtypes = [_I, _I, _I, _I]
    data = K.datasets.load_data("FB15k-237")
    g = torch.Generator().manual_seed(1)
    V, h, k = data.num_nodes, 500, 10
    emb = torch.randn(V, h, generator=g).to(dev)
    w = torch.randn(data.num_rels, h, generator=g).to(dev)
    test = torch.from_numpy(data.test).to(dev)
    a, r = test[:, 0].to(torch.int32).contiguous(), test[:, 1].to(torch.int32).contiguous()
    M = a.numel()
    fi = K.utils.FilterIndex(np.concatenate([data.train, data.valid, data.test]), V, data.num_rels, dev)
    fp, fx = fi.lists(a, r, "object")
    ws = torch.empty(old.kg_distmult_topk_workspace_bytes(M, V, h, k), dtype=torch.uint8, device=dev)
    shift = torch.tensor([0.25], device=dev)

    def parent(filtered):
        idx = torch.empty((M, k), dtype=torch.int32, device=dev)
        sc = torch.empty((M, k), dtype=torch.float32, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        if filtered:
            rc = old.kg_distmult_topk_filtered(emb.data_ptr(), w.data_ptr(), a.data_ptr(), r.data_ptr(), M, V, h,
                                               shift.data_ptr(), k, fp.data_ptr(), fx.data_ptr(), ws.data_ptr(),
                                               ws.numel(), idx.data_ptr(), sc.data_ptr(), st)
        else:
            rc = old.kg_distmult_topk(emb.data_ptr(), w.data_ptr(), a.data_ptr(), r.data_ptr(), M, V, h,
                                      shift.data_ptr(), k, ws.data_ptr(), ws.numel(), idx.data_ptr(), sc.data_ptr(), st)
        assert rc == 0
        return idx, sc

    def new(filtered):
        return K.ops.distmult_topk(emb, w, a, r, k=k, shift=shift, filt_ptr=fp if filtered else None,
                                   filt_idx=fx if filtered else None)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    out = {"queries": M, "entities": V, "h": h, "k": k}
    for filtered in (False, True):
        p, q = parent(filtered), new(filtered)
        torch.cuda.synchronize()
        same = bool(torch.equal(p[0], q[0]) and torch.equal(p[1], q[1]))
        ts = {"parent": [], "new": []}
        for _ in range(rounds):
            ts["parent"].append(timed(lambda: parent(filtered)))
            ts["new"].append(timed(lambda: new(filtered)))
        out["filtered" if filtered else "unfiltered"] = {"bitwise_equal": same, "ms": ts}
    return out


def bench_vs(parent_tree, rounds, steps, warmup):
    out = {"parent": [], "new": []}
    for _ in range(rounds):
        for key, tree in (("parent", parent_tree), ("new", ROOT)):
            p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup",
                                str(warmup)], cwd=tree, capture_output=True, text=True, timeout=1800)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
            res = json.loads(line)
            out[key].append({k: v for k, v in res.items() if isinstance(v, (int, float)) and
                             any(s in k for s in ("step", "eval", "e2e"))})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="topk,bench,eval,driver")
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--epochs", type=int, default=60)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--eval-worker", action="store_true")
    args = ap.parse_args()
    if args.eval_worker:
        eval_worker(args.reps)
        return
    res = {"card": card()}
    ns = [n for n in (int(x) for x in args.gpus.split(",")) if n <= res["card"]["gpus"]]
    parts = args.parts.split(",")
    if "topk" in parts and args.parent_lib:
        res["topk_unsharded_vs_parent"] = topk_vs(args.parent_lib, 5, args.reps)
    if "bench" in parts and args.parent_tree:
        res["bench_py_vs_parent"] = bench_vs(args.parent_tree, 2, 10, 3)
    if "eval" in parts:
        res["sharded_eval"] = evals(ns, args.reps)
    if "driver" in parts:
        res["driver_iteration"] = driver(ns, args.epochs)
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
