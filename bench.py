#!/usr/bin/env python
"""Benchmark of the GCN-VAE link-prediction hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W     # the CPU oracle port, host cores

Workload (config.workload = "fb15k237-full", BASELINE.json configs[1]): synthetic FB15k-237-shaped
KG (14 541 entities, 237 relations, 272 115 train triples), h=500, 100 blocks, 10-component MoG
prior, dropout 0.2, negative rate 10.  One STEP = one full-graph training step through the
reference-shaped API: every train triple is sampled (graph_batch_size = 272 115), half become the
message-passing graph (272 114 directed edges), all 2 993 265 scored triplets go through DistMult +
BCE; timed region = graph index build + forward + loss + backward + grad clip + Adam.
`value` = directed message-passing edges processed per second with inputs resident in HBM;
`e2e` = the same step with every input copied from pinned host memory and the loss read back.
`eval` = all-entity rank evaluation (both perturbation directions) of the 20 466 test triples.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line: NCCL's version banner / warnings go to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

METRIC = "train edges/s (fwd+bwd) + eval triples/s, FB15k-237 shape, 1/2/4/8 B200"
H, BASES, MOG_K, DROPOUT, NEG = 500, 100, 10, 0.2, 10
REG, KL = 0.01, 1e-5


# ------------------------------------------------------------------------------------------------
# shared: synthetic inputs produced by the reference's own sampler path (host, numpy)
# ------------------------------------------------------------------------------------------------
def sample_step(utils_mod, data, batch, seed):
    np.random.seed(seed)
    return utils_mod.generate_sampled_graph_and_labels(data.train, batch, 0.5, data.num_rels, None, None,
                                                       NEG, "uniform")


DUMP_MAX_ELEMS = 15 << 20       # float32 elements of one dump: 60 MiB in all, below 64 MB with the .npy headers


def dump_step_outputs(out_dir, loss, model):
    """--dump-outputs: what the timed train step hands its caller after its last step - the loss, and every
    parameter as Adam left it with the gradient it was updated from - as <out_dir>/<name>.npy in float32 (loss:
    float64).  When these arrays hold more than DUMP_MAX_ELEMS elements together, each is written as the same seeded
    sample of the same share of its flattened elements in every run, so that two builds can be compared output for
    output."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = [("param." + name, p) for name, p in model.named_parameters()]
    arrays += [("grad." + name, p.grad) for name, p in model.named_parameters() if p.grad is not None]
    share = min(1.0, DUMP_MAX_ELEMS / sum(t.numel() for _, t in arrays))
    np.save(os.path.join(out_dir, "loss.npy"), np.asarray([float(loss)], dtype=np.float64))
    for name, t in arrays:
        a = t.detach().float().cpu().numpy().reshape(-1)
        keep = int(a.size * share)
        if keep < a.size:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# the workload both arms run: one dict, built by one function, so the two JSON lines name the same config
# ------------------------------------------------------------------------------------------------
def workload_config(args, data, n_nodes, n_edges, n_triplets, world):
    return {"workload": args.workload, "entities": int(data.num_nodes), "relations": int(data.num_rels),
            "train_triples": int(len(data.train)), "graph_edges": int(n_edges), "scored_triplets": int(n_triplets),
            "nodes": int(n_nodes), "h": H, "bases": BASES, "mog_k": MOG_K, "n_flows": args.n_flows, "negative_rate": NEG,
            "parallelism": f"replicas x{world} (grad all-reduce), eval entity-sharded; the CPU arm runs one replica",
            "timed": "one train step = (device edge index on the GPU arm) + fwd + loss + bwd + grad clip + Adam",
            "l2": "GPU arm: flushed between steps (256 MiB write); CPU arm: not applicable"}


def load_datasets_module():
    """gcn-vae_b200/datasets.py without importing the package (the reference arm loads no kernels)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("kg_datasets", os.path.join(ROOT, "gcn-vae_b200", "datasets.py"))
    datasets = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(datasets)
    return datasets


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_oracle_rates(steps, warmup, n_flows, sample_edges, eval_queries=100, log=None, shape="FB15k-237",
                     anomaly_steps=1, warmup_edges=20000):
    """Times oracle/kgvae_oracle.py (the CPU restatement of the reference path, the reference's own op
    sequence) on the host cores, on the SAME workload as the GPU arm: `sample_edges` sampled train edges per
    step (all of them for the *-full workloads: 272 114 graph edges, 2 993 265 scored triplets at the
    FB15k-237 shape), h = 500, 100 blocks, and the same timed region: forward + loss + backward + gradient
    clipping + Adam (kgvae/link_predict.py:223-228).  Warm-up steps run the reference's default 20 000-edge
    sample (they only warm the thread pool and the allocator).  The reference turns autograd anomaly
    detection on at import (kgvae/model.py:10); `value` is measured with it OFF (the faster, fairer
    figure) and `anomaly_steps` extra steps with it ON give the faithful one.  Evaluation: `eval_queries`
    test triples in both directions against all entities."""
    from oracle import kgvae_oracle as O
    datasets = load_datasets_module()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    data = datasets.synthetic_kg(shape, seed=0)
    params = O.init_params(data.num_nodes, H, data.num_rels, BASES, MOG_K, n_flows, seed=0)
    for p in params.values():
        p.requires_grad_(True)
    leaves = [p for p in params.values() if p.requires_grad]
    opt = torch.optim.Adam(leaves, lr=1e-3)

    def one_step(it, n_sample):
        np.random.seed(100 + it)
        graph, node_id, samples, labels = O.generate_sampled_graph_and_labels(
            data.train, n_sample, 0.5, data.num_rels, NEG)
        n = len(node_id)
        eps = torch.randn(n, H)
        masks = tuple((torch.rand(n, w) < 1 - DROPOUT).float() / (1 - DROPOUT) for w in (H, 2 * H))
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        enc = O.kgvae_encode(params, graph, node_id, eps, BASES, n_flows, masks)
        out = O.kgvae_loss(params, enc, samples, labels, REG, KL, n_flows)
        out["loss"].backward()
        torch.nn.utils.clip_grad_norm_([p for p in leaves if p.grad is not None], 1.0)
        opt.step()
        dt = time.perf_counter() - t0
        return dt, len(graph["etype"]), len(labels)

    times, edges = [], sample_edges
    for it in range(warmup + steps):
        warm = it < warmup
        dt, edges_it, trip_it = one_step(it, warmup_edges if warm else sample_edges)
        if not warm:
            times.append(dt)
            edges = edges_it
        if log:
            log(f"[cpu oracle] {'warm-up' if warm else 'step'} {it}: {dt:.2f}s ({edges_it} edges, {trip_it} triplets)")
    anomaly_times = []
    if anomaly_steps > 0:
        with torch.autograd.set_detect_anomaly(True):
            for it in range(anomaly_steps):
                dt, _, _ = one_step(warmup + steps + it, sample_edges)
                anomaly_times.append(dt)
                if log:
                    log(f"[cpu oracle] anomaly-detection ON step: {dt:.2f}s")
    step_s = sum(times) / len(times)
    # evaluation sample
    with torch.no_grad():
        emb = params["encoder.input_layer.embedding.weight"].detach()
        t = torch.from_numpy(data.test[:eval_queries])
        t0 = time.perf_counter()
        O.calc_mrr(emb, params["w_relation"].detach(), t, eval_bz=eval_queries, policy="reference")
        eval_dt = time.perf_counter() - t0
    res = {"train_edges_per_s": edges / step_s, "step_s": step_s, "cores": cores, "edges": edges,
           "eval_triples_per_s": eval_queries / eval_dt,
           "sample": f"same workload as the GPU arm: {edges} graph edges, {trip_it} scored triplets per step, "
                     f"fwd+loss+bwd+clip+Adam, {len(times)} timed steps (autograd anomaly detection off; warm-up "
                     f"steps on a {warmup_edges}-edge sample); eval: {eval_queries} test triples x 2 directions "
                     f"x {data.num_nodes} candidates"}
    if anomaly_times:
        a = sum(anomaly_times) / len(anomaly_times)
        res["anomaly_on"] = {"edges_per_s": edges / a, "step_s": a, "steps": len(anomaly_times),
                             "note": "torch.autograd.set_detect_anomaly(True) as the reference sets at import "
                                     "(kgvae/model.py:10)"}
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload in ("am-entity", "wikikg2-part"):
        # the timed CPU port covers the link-prediction step at the FB15k-237 / WN18 shapes; the reference itself
        # runs neither of these two on one host in bounded time (8.9 GB table / 32 M-edge graph)
        print(json.dumps({"impl": "reference", "unavailable": f"no bounded CPU sample for workload {args.workload}"}))
        return
    shape = "wn18" if args.workload.startswith("wn18") else "FB15k-237"
    log = lambda m: print(m, file=sys.stderr, flush=True)
    datasets = load_datasets_module()
    data = datasets.synthetic_kg(shape, seed=0)
    batch = 20000 if args.workload.endswith("-step") else len(data.train)
    r = cpu_oracle_rates(args.steps, args.warmup, args.n_flows, sample_edges=batch, log=log, shape=shape)
    # the sizes the GPU arm reports for the same sampler call (seed 0): nodes after relabelling, 2 * batch // 2 edges
    from oracle import kgvae_oracle as O
    np.random.seed(0)
    graph, node_id, samples, labels = O.generate_sampled_graph_and_labels(data.train, batch, 0.5, data.num_rels, NEG)
    cfg = workload_config(args, data, len(node_id), len(graph["etype"]), len(labels), args.gpus)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["train_edges_per_s"], "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["step_s"] * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": r["train_edges_per_s"], "unit": "edges/s", "cores": r["cores"],
                         "kind": "port", "sample": r["sample"], "anomaly_on": r.get("anomaly_on"),
                         "eval_triples_per_s": r["eval_triples_per_s"]},
        "e2e": {"value": r["train_edges_per_s"], "unit": "edges/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clock / throttle-reason samples taken while the benchmark runs.  nvidia-smi needs about a
    second to start, so the sampler is created first thing; `mark()` / `stop()` bracket the window whose
    samples are reported (warm-up through the last timed region - all of it GPU load)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=20):
        self.rows, self.proc, self.t0 = [], None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", str(period_ms),
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark(self, wait_s=3.0):
        """Start of the reported window; waits (bounded) until nvidia-smi has produced its first sample."""
        deadline = time.time() + wait_s
        while self.proc is not None and not self.rows and time.time() < deadline:
            time.sleep(0.02)
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time() + 0.03
        time.sleep(0.05)                                      # let the last in-window sample arrive
        self.proc.terminate()
        self.thread.join(timeout=2)
        t0 = self.t0 if self.t0 is not None else 0.0
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 7] or [r for _, r in self.rows if len(r) >= 7]
        num = lambda x: x.replace(".", "").isdigit()
        sm = [float(r[0]) for r in rows if num(r[0])]
        mx = [float(r[1]) for r in rows if num(r[1])]
        pw = [float(r[2]) for r in rows if num(r[2])]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i] == "Active" for r in rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": reasons, "samples": len(sm)}


def algorithmic_bytes(tag, shp):
    """Algorithmic (compulsory) HBM bytes of one launch of the named op; DESIGN.md section 4."""
    N, E, S, R2, h = shp["N"], shp["E"], shp["S"], shp["R2"], H
    if tag.startswith("kg_bdd_rel_fwd"):                # SURVEY 8(d): per edge 4*in + 12, per node 4*out, weights once
        si, so = (int(x) for x in tag[tag.index("[") + 1:-1].split("x"))
        return E * (4 * BASES * si + 16) + 4 * N * BASES * so + 4 * R2 * BASES * si * so
    if tag.startswith("kg_bdd_rel_bwd"):                # per edge 4*(in+out) + 12, per node 4*in (dx), weights r+w
        si, so = (int(x) for x in tag[tag.index("[") + 1:-1].split("x"))
        return E * (4 * BASES * (si + so) + 16) + 4 * N * BASES * si + 2 * 4 * R2 * BASES * si * so
    if tag == "kg_distmult_bce_fwd":                    # SURVEY 8(d): 3 rows + record per triplet for the score, and
        # the backward into z in the same pass: one row of gradient into dz[s] and one into dz[o]; dw, dz once
        return S * (5 * 4 * h + 16 + 4 + 4) + 4 * shp["R"] * h + 4 * N * h
    if tag == "kg_distmult_bwd_dz":                     # each triplet seen from both ends: w row + other row + record
        return 2 * S * (2 * 4 * h + 16 + 4) + 4 * N * h
    return None


def measure_l2_peak(dev, rows, row_floats, n_ops=3_000_000, reps=5):
    """kg_probe_l2 on two L2-resident [rows, row_floats] fp32 matrices: GB/s of whole-row random reads, of
    whole-row random reductions (red.global.add.v4.f32), and of both at once (bytes of both directions
    counted) - best of `reps` launches each, CUDA events on the launching stream."""
    from gcn_vae_b200 import _lib as L
    src = torch.randn(rows, row_floats, device=dev)
    dst = torch.zeros(rows, row_floats, device=dev)
    sink = torch.zeros(4, device=dev)
    out = {"rows": rows, "row_bytes": 4 * row_floats, "ops": n_ops}
    for name, mode in (("read", 1), ("reduce", 2), ("mixed", 3)):
        best = None
        for it in range(reps + 1):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            L.call("kg_probe_l2", L.f32(src), L.f32(dst), rows, row_floats, n_ops, mode, L.f32(sink), L.stream())
            b.record()
            b.synchronize()
            if it > 0:
                ms = a.elapsed_time(b)
                best = ms if best is None else min(best, ms)
        nbytes = n_ops * 4 * row_floats * (2 if mode == 3 else 1)
        out[name + "_gbs"] = nbytes / (best * 1e-3) / 1e9
        out[name + "_ms"] = best
    return out


def gemm_vs_library(dev, log, iters=10):
    """kg_gemm_f32 (tcgen05, fp32-accurate two-term fp16 split, operand conversion included) next to the library
    kernel it replaces on the same box: torch.matmul in fp32 with TF32 off (cuBLAS SGEMM - what DGL / F.linear
    run in the reference, kgvae/model.py:55,58, kgvae/flow_network.py:15), at the benchmarked shapes."""
    from gcn_vae_b200 import ops
    gen = torch.Generator(device=dev).manual_seed(3)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    out = {}
    try:
        for (M, N, Kd, ta, tb) in [(14541, 500, 500, False, False), (14541, 1000, 500, False, False),
                                   (14541, 500, 1000, False, True), (500, 1000, 14541, True, False),
                                   (40914, 500, 500, False, True), (500, 500, 40914, True, False)]:
            a = torch.randn((Kd, M) if ta else (M, Kd), device=dev, generator=gen)
            b = torch.randn((N, Kd) if tb else (Kd, N), device=dev, generator=gen)
            c = torch.empty(M, N, device=dev)
            am, bm = (a.t() if ta else a), (b.t() if tb else b)

            def t_of(fn):
                for _ in range(3):
                    fn()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    fn()
                e1.record()
                e1.synchronize()
                return e0.elapsed_time(e1) / iters
            ours = t_of(lambda: ops.gemm(a, b, c, trans_a=ta, trans_b=tb))
            lib = t_of(lambda: torch.matmul(am, bm, out=c))
            err = float((c - ops.gemm(a, b, torch.empty_like(c), trans_a=ta, trans_b=tb)).abs().max() / c.abs().max())
            tag = f"{M}x{N}x{Kd},{'T' if ta else 'N'}{'T' if tb else 'N'}"
            out[tag] = {"kg_gemm_f32_ms": ours, "torch_matmul_fp32_ms": lib, "speedup": lib / ours,
                        "tflops_algorithmic": 2.0 * M * N * Kd / (ours * 1e-3) / 1e12, "max_rel_diff": err}
            log(f"  [gemm {tag}] kg_gemm_f32 {ours:.3f} ms, torch.matmul fp32 {lib:.3f} ms ({lib / ours:.2f}x), diff {err:.1e}")
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return out


def streaming_layer_bench(dev, pk, log, n_nodes=2_500_000, n_etypes=1070, n_edges=32_000_000, iters=5, l2_peak=None):
    """RGCN(bdd) message passing at the ogbl-wikikg2 shape (BASELINE.json configs[4]: 2.5 M entities,
    2 x 535 relation types, 2 x 16 M directed edges, h = 500, 100 blocks) on ONE GPU: the regime the
    HBM-roofline target of north_star is about - every feature matrix (5 / 10 GB) is far larger than
    L2, so gathered rows really stream from HBM.  Times the four message-passing launches of one
    encoder (layer 1: 500 -> 500, layer 2: 500 -> 1000; forward and fused dX + dW backward) with CUDA
    events; algorithmic bytes per SURVEY.md 8(d) / DESIGN.md section 4."""
    import gcn_vae_b200 as K
    from gcn_vae_b200 import _lib as L
    from gcn_vae_b200 import ops
    out = {"shape": {"nodes": n_nodes, "etypes": n_etypes, "edges": n_edges, "h": H, "bases": BASES},
           "regime": "streaming (x, agg, dagg, dx are 5-10 GB each; L2 is 126 MB)", "kernels": {}}
    gen = torch.Generator(device=dev).manual_seed(0)
    for graph_kind in ("uniform", "skewed"):
        if graph_kind == "uniform":
            src = torch.randint(0, n_nodes, (n_edges,), device=dev, generator=gen, dtype=torch.int32)
            dst = torch.randint(0, n_nodes, (n_edges,), device=dev, generator=gen, dtype=torch.int32)
            et = torch.randint(0, n_etypes, (n_edges,), device=dev, generator=gen, dtype=torch.int32)
        else:       # heavy-tailed degrees and relation frequencies (real KGs): id = floor(n * u^3)
            pw = lambda n: (torch.rand(n_edges, device=dev, generator=gen).pow(3) * n).to(torch.int32).clamp_(max=n - 1)
            src, dst, et = pw(n_nodes), pw(n_nodes), pw(n_etypes)
        deg = torch.bincount(dst.long(), minlength=n_nodes).clamp_(min=1).float()
        norm = (1.0 / deg)[dst.long()].contiguous()
        t0 = time.perf_counter()
        gi = ops.graph_index(src, dst, et, norm, n_nodes, n_etypes)
        torch.cuda.synchronize()
        index_ms = (time.perf_counter() - t0) * 1e3
        x = torch.randn(n_nodes, H, device=dev, generator=gen)
        res = {}
        for si, so in ((H // BASES, H // BASES), (H // BASES, 2 * H // BASES)):
            in_f, out_f = BASES * si, BASES * so
            weight = torch.randn(n_etypes, BASES * si * so, device=dev, generator=gen) * 0.05
            w_fwd = w_bwd = None
            if L.lib().kg_bdd_layouts_needed(BASES, si, so):
                w_fwd = torch.empty((n_etypes, si, out_f), device=dev)
                w_bwd = torch.empty((n_etypes, so, in_f), device=dev)
                L.call("kg_bdd_weight_layouts", L.f32(weight), n_etypes, BASES, si, so, L.f32(w_fwd), L.f32(w_bwd), L.stream())
            agg = torch.empty((n_nodes, out_f), device=dev)
            dx = torch.empty((n_nodes, in_f), device=dev)
            dw = torch.empty_like(weight)
            p_fwd = ops._rel_order(gi, 0, n_nodes, 4 * out_f)
            p_bwd = ops._rel_order(gi, 1, n_nodes, 8 * in_f)

            def fwd():
                L.call("kg_bdd_rel_fwd", L.f32(x), None, 0, L.i32(p_fwd), n_edges, L.f32(weight), L.f32(w_fwd), BASES, si, so, L.f32(agg),
                       ops.HINT_STREAM_X | ops.HINT_TILE_RESIDENT, L.stream())

            def bwd():
                L.call("kg_bdd_rel_bwd", L.f32(x), None, 0, L.f32(agg), L.i32(p_bwd), n_edges, L.f32(weight), L.f32(w_bwd), BASES, si, so,
                       L.f32(dx), L.f32(dw), ops.HINT_STREAM_D | ops.HINT_TILE_RESIDENT, L.stream())

            for name, fn, zero in ((f"kg_bdd_rel_fwd[{si}x{so}]", fwd, (agg,)), (f"kg_bdd_rel_bwd[{si}x{so}]", bwd, (dx, dw))):
                ms = []
                for it in range(iters + 2):
                    for z in zero:
                        z.zero_()                       # outside the timed events; also sweeps L2 (>= 5 GB)
                    if name.startswith("kg_bdd_rel_bwd") and it == 0:
                        agg.normal_(generator=gen)      # a dense upstream gradient
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    fn()
                    b.record()
                    b.synchronize()
                    if it >= 2:
                        ms.append(a.elapsed_time(b))
                t = sum(ms) / len(ms)
                ab = algorithmic_bytes(name, {"N": n_nodes, "E": n_edges, "S": 0, "R2": n_etypes, "R": n_etypes // 2})
                res[name] = {"ms": t, "algorithmic_bytes": ab, "achieved_gbs": ab / t / 1e6,
                             "frac_of_hbm_peak": ab / t / 1e6 / pk["hbm_gbs"], "edges_per_s": n_edges / t * 1e3}
                # the second bound of these launches: every edge's message (forward: `out` floats) or source gradient
                # (backward: `in` floats) is REDUCED into an L2-resident tile; the probe gives what L2 sustains for
                # whole-row reductions.  The 5x10 forward reduces 4 KB per edge for 2 KB gathered: reduce-bound.
                red_bytes = n_edges * 4 * (out_f if name.startswith("kg_bdd_rel_fwd") else in_f)
                res[name]["reduce_bytes"] = red_bytes
                if l2_peak:
                    floor_ms = max(ab / pk["hbm_gbs"] / 1e6, red_bytes / l2_peak["reduce_gbs"] / 1e6)
                    res[name]["l2_reduce_gbs"] = red_bytes / t / 1e6
                    res[name]["frac_of_l2_reduce_probe"] = red_bytes / t / 1e6 / l2_peak["reduce_gbs"]
                    res[name]["floor_ms"] = floor_ms
                    res[name]["frac_of_floor"] = floor_ms / t
                    res[name]["bound"] = "l2 reductions" if red_bytes / l2_peak["reduce_gbs"] > ab / pk["hbm_gbs"] else "hbm"
                log(f"  [streaming/{graph_kind}] {name:26s} {t:8.2f} ms  {ab / t / 1e6:8.0f} GB/s  "
                    f"{100 * ab / t / 1e6 / pk['hbm_gbs']:5.1f}% of measured HBM peak")
            del agg, dx, dw, weight, w_fwd, w_bwd
        out["kernels"][graph_kind] = res
        out.setdefault("graph_index_ms", {})[graph_kind] = index_ms
        del gi, x, src, dst, et, norm
        torch.cuda.empty_cache()
    return out


def partitioned_leg(args, dev, world, rank, log, allgather, steps, warmup, scale):
    """One measurement of the destination-partitioned wikikg2-shaped training step (see run_partitioned) on the
    already initialised process group; returns a dict (every rank; timing = max over ranks)."""
    import torch.distributed as dist
    import gcn_vae_b200 as K
    from gcn_vae_b200 import _lib as L
    from gcn_vae_b200 import parallel

    n_nodes, n_rels, n_trip = int(2_500_000 * scale), 535, int(16_000_000 * scale)
    n_scored = n_trip * (NEG + 1)          # every train triple + NEG corruptions each, as the reference scores them
    # the same global graph on every rank (same device generator seed), then this rank's share
    gen = torch.Generator(device=dev).manual_seed(1234)
    s = torch.randint(0, n_nodes, (n_trip,), device=dev, generator=gen, dtype=torch.int32)
    o = torch.randint(0, n_nodes, (n_trip,), device=dev, generator=gen, dtype=torch.int32)
    r = torch.randint(0, n_rels, (n_trip,), device=dev, generator=gen, dtype=torch.int32)
    src, dst, et = torch.cat([s, o]), torch.cat([o, s]), torch.cat([r, r + n_rels])     # + reverse edges
    deg = torch.bincount(dst.long(), minlength=n_nodes).clamp_(min=1).float()
    n_edges_global = int(src.numel())
    # this rank's share of the scored triplets: positives + corruptions (subject or object replaced at random)
    t0, t1 = parallel.block_range(n_trip, rank, world)
    gen_t = torch.Generator(device=dev).manual_seed(99 + rank)
    pos = torch.stack([s[t0:t1], r[t0:t1], o[t0:t1]], 1)
    neg = pos.repeat(NEG, 1)
    vals = torch.randint(0, n_nodes, (neg.shape[0],), device=dev, generator=gen_t, dtype=torch.int32)
    head = torch.rand(neg.shape[0], device=dev, generator=gen_t) > 0.5
    neg[:, 0] = torch.where(head, vals, neg[:, 0])
    neg[:, 2] = torch.where(head, neg[:, 2], vals)
    trip = torch.cat([pos, neg]).contiguous()
    labels = torch.zeros(trip.shape[0], device=dev)
    labels[:pos.shape[0]] = 1
    del pos, neg, vals, head
    if world > 1:
        lo, hi = parallel.uniform_block_range(n_nodes, rank, world)
        keep = (dst >= lo) & (dst < hi)
        src, dst, et = src[keep].contiguous(), (dst[keep] - lo).contiguous(), et[keep].contiguous()
        norm = (1.0 / deg)[lo:hi][dst.long()].contiguous()
        del keep
    else:
        lo, hi = 0, n_nodes
        norm = (1.0 / deg)[dst.long()].contiguous()
    del deg, s, o, r
    n_local = hi - lo
    g = K.Graph()
    g._n = n_nodes if world > 1 else n_local
    g._dev_edges[dev] = (src, dst)
    if world > 1:
        g.partition = parallel.Partition(lo, hi, n_nodes, peer_gather=not allgather, col_chunks=args.col_chunks)
    torch.manual_seed(0)
    # the embedding table is sharded by owner: each rank holds (and updates) only its rows
    model = K.LinkPredict(K.KGVAE, max(n_local, 1), H, n_rels, num_bases=BASES, dropout=DROPOUT, use_cuda=True,
                          reg_param=REG, kl_param=KL, k=MOG_K, n_flows=0).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, fused=True)
    emb_w = model.encoder.input_layer.embedding.weight
    buckets = model.grad_buckets(average=False, sharded=[emb_w])       # replicated parameters: SUM over the ranks
    ids = torch.arange(n_local, dtype=torch.int32, device=dev).view(-1, 1)
    norm2 = norm.view(-1, 1)

    def step():
        buckets.zero()
        emb_w.grad = None
        embed = model(g, ids, et, norm2)
        loss, _, _, _ = model.get_loss(g, embed, trip, labels)
        loss.backward()
        buckets.finish()
        opt.step()
        return loss

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    model.train()
    for _ in range(max(warmup, 3)):
        step()
    sync_all()
    L.launches = 0
    L.profile = {}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        loss = step()
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b)
    launches = L.launches
    prof, L.profile = L.profile, None
    sync_all()
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    op_ms = {tag: sum(x.elapsed_time(y) for x, y in evs) / steps for tag, evs in prof.items()}
    comm_ms = sum(v for tag, v in op_ms.items() if tag.startswith("nccl_exposed"))
    for tag, v in sorted(op_ms.items(), key=lambda kv: -kv[1])[:12]:
        log(f"  [wikikg2-part x{world}] {tag:44s} {v:8.3f} ms/step")
    loss_v = float(loss)
    if world > 1:
        for cache in g.partition._peer_rows.values():
            cache.close()
    res = {"ms_per_step": ms / steps, "edges_per_s": n_edges_global * steps / (ms * 1e-3), "n_gpus": world,
           "steps": steps, "warmup": max(warmup, 3), "loss": loss_v, "gpu_launches": launches,
           "comm_ms": comm_ms, "comm_what": "NCCL time NOT hidden behind compute (CUDA events on the compute stream "
                                            "around every collective / wait), rank 0, ms per step",
           "entities": n_nodes, "relations": n_rels, "graph_edges": n_edges_global,
           "scored_triplets": n_scored, "scale": scale,
           "mode": ("single GPU, unpartitioned" if world == 1 else
                    f"NCCL all-gather of layer inputs in {g.partition.col_chunks} column chunk(s), pipelined with message passing "
                    f"and the self-loop GEMM" if allgather else
                    "layer inputs gathered from peer HBM by the message-passing kernels (NVLink, CUDA IPC)"),
           "top_ops_ms": dict(sorted(op_ms.items(), key=lambda kv: -kv[1])[:8]),
           "all_ops_ms": {k_: round(v, 3) for k_, v in sorted(op_ms.items(), key=lambda kv: -kv[1])},
           "ops_total_ms": sum(op_ms.values())}
    del model, opt, buckets, g, trip, labels, src, dst, et, norm, norm2, ids
    torch.cuda.empty_cache()
    return res


def run_partitioned(args):
    """--workload wikikg2-part (BASELINE.json configs[4]): full-graph GCN-VAE training step on a synthetic
    ogbl-wikikg2-shaped KG (2.5 M entities, 535 relations, 16 M triples = 32 M directed edges, 176 M scored
    triplets = every triple + 10 corruptions, h = 500, 100 blocks), destination-partitioned over the N GPUs of
    one box: rank p owns a block of nodes, every edge into it, and its rows of the embedding table / h1 / h2 /
    z.  Layer inputs reach the edges either by an NCCL all-gather (asynchronous, overlapped with the self-loop
    GEMM; default) or, with --peer, straight from the owners' HBM inside the message-passing kernels; gradients
    wrt the sources are reduce-scattered (overlapped with the weight-gradient GEMM); the decoder scores each
    rank's share of the triplets against the all-gathered z.  STRONG scaling: the graph is fixed, value =
    32 M edges / step time (max over ranks).  N = 1 runs the same step unpartitioned."""
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    log = (lambda m: print(m, file=sys.stderr, flush=True)) if rank == 0 else (lambda m: None)
    clocks = ClockSampler(local)
    clocks.mark()
    r = partitioned_leg(args, dev, world, rank, log, allgather=not args.peer, steps=args.steps, warmup=args.warmup,
                        scale=args.scale)
    clock_info = clocks.stop()
    if rank == 0:
        line = {
            "metric": METRIC, "value": r["edges_per_s"], "unit": "edges/s", "n_gpus": world,
            "steps": args.steps, "warmup": r["warmup"], "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "wikikg2-part", "entities": r["entities"], "relations": r["relations"],
                       "graph_edges": r["graph_edges"], "scored_triplets": r["scored_triplets"], "h": H, "bases": BASES,
                       "scale": args.scale, "parallelism": f"destination-partitioned x{world}: " + r["mode"],
                       "timed": "fwd + loss + bwd + grad all-reduce + Adam; one CUDA-event pair over all steps",
                       "l2": "inputs (5 GB feature matrices) far larger than L2"},
            "loss": r["loss"], "gpu_launches": r["gpu_launches"], "clocks": clock_info, "top_ops_ms": r["top_ops_ms"],
        }
        print(json.dumps(line), flush=True)
    leave_process_group(world)


def run_entity(args):
    """--workload am-entity (BASELINE.json configs[3]): baselines/rgcn entity classification on a synthetic
    AM-shaped typed graph (1 666 764 nodes, 133 relation types, 5 988 321 directed edges, 11 classes), the
    reference's AM flags (kgvae/entity_classify.py:138-170 with baselines/rgcn/README.md:35-38: --n-bases 40
    --n-hidden 10 --l2norm 5e-4, two layers, featureless nodes = integer ids).  One STEP = one full-graph
    training epoch as in entity_classify.py:106-113: forward over every edge (input layer = basis lookup
    sum_b coef[r,b] V[b, src, :] without materialising the [R, N, h] table, output layer = dense basis
    conv + softmax), cross-entropy on the training nodes, backward, Adam(weight_decay).  value = directed
    edges per second.  N > 1: ONE graph over the N GPUs (strong scaling) - the 2.67 GB basis table and its Adam
    state are sharded by source-node owner, the partial hidden states (67 MB) are all-reduced, the output layer
    is destination-partitioned (entity_classify.PartitionedEntityClassify); --replicas runs the old weak-scaling
    form (one full graph per rank, gradients all-reduced)."""
    import torch.distributed as dist
    import torch.nn.functional as F
    import gcn_vae_b200 as K
    from gcn_vae_b200 import _lib as L
    from gcn_vae_b200 import entity_classify as EC

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    log = (lambda m: print(m, file=sys.stderr, flush=True)) if rank == 0 else (lambda m: None)
    clocks = ClockSampler(local)
    n_hidden, n_bases, l2norm = 10, 40, 5e-4
    t0 = time.perf_counter()
    partitioned = world > 1 and not args.replicas
    data = EC.synthetic_graph("am", seed=0 if partitioned else rank, scale=args.scale)
    log(f"synthetic AM-shaped graph: {time.perf_counter() - t0:.1f}s; nodes={data.num_nodes} edges={len(data.edge_src)}")
    E, N = len(data.edge_src), data.num_nodes
    pin = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).pin_memory()
    host = {"src": pin(data.edge_src, torch.int32), "dst": pin(data.edge_dst, torch.int32),
            "etype": pin(data.edge_type, torch.int32), "norm": pin(data.edge_norm.reshape(-1, 1), torch.float32),
            "labels": pin(data.labels, torch.int64), "train_idx": pin(data.train_idx, torch.int64)}
    h2d_bytes = sum(t.numel() * t.element_size() for t in host.values())
    resident = {k: v.to(dev) for k, v in host.items()}
    torch.manual_seed(0)
    n_table = N
    if partitioned:
        lo_p, hi_p = K.parallel.block_range(N, rank, world)
        n_table = hi_p - lo_p
    model = EC.EntityClassify(n_table, n_hidden, data.num_classes, data.num_rels, num_bases=n_bases, num_hidden_layers=0,
                              dropout=0.0, use_self_loop=False, use_cuda=True).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-2, weight_decay=l2norm, fused=True)
    params = [p for p in model.parameters() if p.requires_grad]
    feats = model.create_features()
    pe = EC.PartitionedEntityClassify(model, data, rank, world, dev) if partitioned else None

    graphs = {}

    def graph_of(t):
        """The graph object is built ONCE, before the epoch loop, as in the reference
        (kgvae/entity_classify.py:80-82); its device edge index is built on first use and reused by every
        epoch.  (The e2e leg hands over freshly copied tensors each step, so there the index is rebuilt.)"""
        key = t["src"].data_ptr()
        if key not in graphs:
            gr = K.Graph()
            gr._n = N
            gr._dev_edges[dev] = (t["src"], t["dst"])
            graphs.clear()
            graphs[key] = gr
        return graphs[key]

    def step_partitioned():
        opt.zero_grad(set_to_none=True)
        loss = pe.loss(pe.logits())
        loss.backward()
        pe.reduce_grads()
        opt.step()
        return loss

    def step(t):
        if partitioned:
            return step_partitioned()
        gr = graph_of(t)
        opt.zero_grad(set_to_none=True)
        logits = model(gr, feats, t["etype"], t["norm"])
        loss = F.cross_entropy(logits[t["train_idx"]], t["labels"][t["train_idx"]])
        loss.backward()
        if world > 1:
            K.parallel.allreduce_mean_grads(params)
        opt.step()
        return loss

    def e2e_step():
        if partitioned:                      # the graph shards stay resident (built once, as in the reference)
            return float(step_partitioned())
        return float(step({k: v.to(dev, non_blocking=True) for k, v in host.items()}))

    def timed(fn, n_steps):
        total = 0.0
        for _ in range(n_steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            total += a.elapsed_time(b)
        return total

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    model.train()
    clocks.mark()
    for _ in range(max(args.warmup, 3)):
        step(resident)
    sync_all()
    L.launches = 0
    L.profile = {}
    ms_dev = max_over_ranks(timed(lambda: step(resident), args.steps))
    launches = L.launches
    prof, L.profile = L.profile, None
    sync_all()
    for _ in range(2):
        e2e_step()
    sync_all()
    ms_e2e = max_over_ranks(timed(e2e_step, args.steps))
    sync_all()
    clock_info = clocks.stop()
    if rank != 0:
        leave_process_group(world)
        return
    op_ms = {tag: sum(a.elapsed_time(b) for a, b in evs) for tag, evs in prof.items()}
    op_n = {tag: len(evs) for tag, evs in prof.items()}
    total_ops = sum(op_ms.values())
    top = sorted(op_ms.items(), key=lambda kv: -kv[1])
    for tag, ms in top[:12]:
        log(f"  {tag:44s} {ms / args.steps:8.3f} ms/step  {100 * ms / total_ops:5.1f}%  x{op_n[tag] // args.steps}")
    pk = peaks()
    # algorithmic bytes of the input-layer lookup (SURVEY 8(d), row a4): per edge the n_bases rows
    # V[b, src, :] (4*h bytes each) + the 16-byte record + the coefficient row; per node the h-wide output
    table = 4 * n_bases * n_table * n_hidden          # this rank's rows of the basis table V [n_bases, N, h] (2.67 GB in all)
    e_rank = E // world if partitioned else E         # edges one launch walks
    ab = {"kg_basis_id_src_fwd": table + e_rank * (16 + 4 * n_hidden) + 4 * N * n_hidden,   # V once, record + out row per edge
          # backward: V read once, dV written once, record + upstream gradient row per edge
          "kg_basis_id_src_bwd": 2 * table + e_rank * (16 + 4 * n_hidden)}
    roof = None
    for tag, ms in top:
        if tag in ab:
            per = ms / op_n[tag]
            ach = ab[tag] / (per * 1e-3) / 1e9
            tfile = os.path.join(ROOT, "profiles", "traffic.json")
            measured = json.load(open(tfile)).get(tag) if (os.path.exists(tfile) and not partitioned) else None
            roof = {"kernel": tag, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / pk["hbm_gbs"], "traffic": measured, "peak_source": pk["source"], "ms_per_launch": per,
                    "algorithmic_bytes": ab[tag], "share_of_step": ms / total_ops,
                    "regime": "streaming: the basis table V is 2.67 GB, its gradient another 2.67 GB; ncu: DRAM traffic "
                              "1.10x algorithmic, sm__throughput 54 % - the launch is bound by instruction issue, "
                              "not by DRAM (profiles/r02o_am_kernels_ncu_full.txt)"}
            break
    total_edges = E * (1 if partitioned else world) * args.steps
    line = {
        "metric": METRIC, "value": total_edges / (ms_dev * 1e-3), "unit": "edges/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": "strong" if partitioned else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "am-entity", "nodes": N, "relations": data.num_rels, "graph_edges": E,
                   "classes": data.num_classes, "n_hidden": n_hidden, "n_bases": n_bases, "l2norm": l2norm,
                   "train_nodes": len(data.train_idx), "scale": args.scale,
                   "parallelism": (f"one graph over {world} GPUs: basis table sharded by source owner, hidden state "
                                   f"all-reduced, output layer destination-partitioned") if partitioned else
                                  f"replicas x{world} (grad all-reduce)",
                   "timed": "fwd + cross-entropy + bwd + Adam (graph built once before the epochs, as in the reference); "
                            "per-step CUDA events",
                   "l2": "inputs (2.67 GB basis table) far larger than L2"},
        "e2e": {"value": total_edges / (ms_e2e * 1e-3), "unit": "edges/s",
                "h2d_bytes_per_step": 0 if partitioned else h2d_bytes,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "clocks": clock_info, "roofline": roof, "cpu_baseline": None,
    }
    print(json.dumps(line), flush=True)
    leave_process_group(world)


def leave_process_group(world):
    """dist.destroy_process_group() that cannot hold the launcher: the result line is already printed when this is
    called, so if the communicator teardown is still stuck after 60 s a watchdog ends the process (exit code 0)."""
    if world <= 1:
        return
    import torch.distributed as dist
    sys.stdout.flush()
    sys.stderr.flush()
    dog = threading.Timer(60.0, lambda: os._exit(0))
    dog.daemon = True
    dog.start()
    torch.cuda.synchronize()
    dist.destroy_process_group()
    dog.cancel()


def run_gpu(args):
    import torch.distributed as dist
    import gcn_vae_b200 as K
    from gcn_vae_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    log = (lambda m: print(m, file=sys.stderr, flush=True)) if rank == 0 else (lambda m: None)
    clocks = ClockSampler(local)

    shape = "wn18" if args.workload.startswith("wn18") else "FB15k-237"
    data = K.datasets.synthetic_kg(shape, seed=0)
    batch = 20000 if args.workload.endswith("-step") else len(data.train)
    torch.manual_seed(0)
    model = K.LinkPredict(K.KGVAE, data.num_nodes, H, data.num_rels, num_bases=BASES, dropout=DROPOUT,
                          use_cuda=True, reg_param=REG, kl_param=KL, k=MOG_K, n_flows=args.n_flows).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, fused=True, capturable=True)
    # gradients are views of one flat buffer cut into buckets; with N > 1 a bucket is all-reduced (averaged) as soon
    # as backward has produced it, overlapping the rest of backward; clipping runs on the flat buffer
    buckets = model.grad_buckets()

    # ---- the step's inputs: the reference's own host sampler (weak scaling: one sample per rank) --
    t0 = time.perf_counter()
    g, node_id, etype, node_norm, samples, labels = sample_step(K.utils, data, batch, seed=rank)
    log(f"host sampling: {time.perf_counter() - t0:.2f}s; nodes={len(node_id)} edges={len(etype)} triplets={len(labels)}")
    E, S, N = len(etype), len(labels), len(node_id)
    pin = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).pin_memory()
    host = {"node_id": pin(node_id, torch.int32), "src": pin(g._src, torch.int32), "dst": pin(g._dst, torch.int32),
            "etype": pin(etype, torch.int32), "norm": pin(node_norm[g._dst].reshape(-1, 1), torch.float32),
            "samples": pin(samples, torch.int32), "labels": pin(labels, torch.float32)}
    h2d_bytes = sum(t.numel() * t.element_size() for t in host.values())
    resident = {k: v.to(dev) for k, v in host.items()}
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def make_graph(t):
        gr = K.Graph()
        gr._n, gr._src, gr._dst = N, g._src, g._dst
        gr._dev_edges[dev] = (t["src"], t["dst"])
        return gr

    def train_step(gr, node_id_t, etype_t, norm_t, samples_t, labels_t):
        buckets.zero()
        embed = model(gr, node_id_t, etype_t, norm_t)
        loss, _, _, _ = model.get_loss(gr, embed, samples_t, labels_t)
        loss.backward()
        buckets.finish()                                    # replicas: bucket all-reduces launched during backward
        buckets.clip_(1.0)
        opt.step()
        return loss

    def step(t):
        gr = make_graph(t)                                  # fresh graph: the index is rebuilt
        return train_step(gr, t["node_id"].view(-1, 1), t["etype"], t["norm"], t["samples"], t["labels"])

    def pinned_sample(seed):
        """One fresh sample from the reference's host sampler as pinned int32 / fp32 tensors."""
        g2, nid, et2, nn2, sm2, lb2 = sample_step(K.utils, data, batch, seed=seed)
        return {"node_id": pin(nid, torch.int32), "src": pin(g2._src, torch.int32), "dst": pin(g2._dst, torch.int32),
                "etype": pin(et2, torch.int32), "norm": pin(nn2[g2._dst].reshape(-1, 1), torch.float32),
                "samples": pin(sm2, torch.int32), "labels": pin(lb2, torch.float32)}, len(nid)

    def timed_with_host_sampler(n_steps, threaded):
        """The loop of kgvae/link_predict.py:200-236 with a FRESH sample every step: host sampler (numpy, the
        reference's random stream) + H2D copies + edge index + step + loss read-back.  `threaded`: the sampler
        runs one step ahead in a worker thread (the bit-exact stream is kept: one thread owns np.random)."""
        import queue
        q = queue.Queue(maxsize=2)
        if threaded:
            def producer():
                for i in range(n_steps):
                    q.put(pinned_sample(5000 + i))
            th = threading.Thread(target=producer, daemon=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if threaded:
            th.start()
        for i in range(n_steps):
            hs, n_i = q.get() if threaded else pinned_sample(5000 + i)
            t = {k: v.to(dev, non_blocking=True) for k, v in hs.items()}
            gr = K.Graph()
            gr._n = n_i
            gr._dev_edges[dev] = (t["src"], t["dst"])
            float(train_step(gr, t["node_id"].view(-1, 1), t["etype"], t["norm"], t["samples"], t["labels"]).detach())
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    train_dev = torch.from_numpy(np.asarray(data.train)).to(dev)
    samp_gen = torch.Generator(device=dev).manual_seed(77 + rank)

    def timed_with_device_sampler(n_steps):
        """Same loop with utils.generate_sampled_graph_and_labels_device (--device-sampler): the uniform edge
        sample, relabelling, negatives, graph split and edge index all on the GPU; nothing crosses PCIe but the
        loss read-back."""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n_steps):
            gr, nid, et2, en2, sm2, lb2 = K.utils.generate_sampled_graph_and_labels_device(
                train_dev, batch, 0.5, data.num_rels, NEG, generator=samp_gen)
            float(train_step(gr, nid, et2, en2, sm2, lb2).detach())
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    def e2e_step():
        t = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        return float(step(t).detach())                      # D2H read of the loss

    prefetch = K.utils.DevicePrefetcher(dev)
    loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_done = [torch.cuda.Event() for _ in range(2)]
    e2e_losses = []

    def timed_e2e(n_steps):
        """K steps through the public API with HOST inputs: every step's 52 MB of pinned inputs are copied
        inside the timed region (step i+1's copy is submitted before step i runs, so it overlaps the
        kernels; step 0's does not overlap anything), the loss is read back every step, and the L2 flush
        is inside the region too.  One event pair around the whole loop."""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        prefetch.submit(host)
        losses = []
        for i in range(n_steps):
            t = prefetch.take()
            if i + 1 < n_steps:
                prefetch.submit(host)
            flush_buf.fill_(1)
            loss_host[i & 1].copy_(step(t).detach().reshape(1), non_blocking=True)   # D2H read of the loss ...
            loss_done[i & 1].record()
            if i > 0:                                       # ... consumed on the host one step later, so that the
                loss_done[(i - 1) & 1].synchronize()        # device never waits for the host between steps
                losses.append(float(loss_host[(i - 1) & 1]))
        loss_done[(n_steps - 1) & 1].synchronize()
        losses.append(float(loss_host[(n_steps - 1) & 1]))
        b.record()
        b.synchronize()
        assert len(losses) == n_steps
        e2e_losses[:] = losses
        return a.elapsed_time(b)

    def timed(fn, n_steps):
        total = 0.0
        for _ in range(n_steps):
            flush_buf.fill_(1)                              # L2 flush, outside the timed events
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            total += a.elapsed_time(b)
        return total

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # Every timed section starts from the SAME model / optimizer state (in-place restore: the captured step keeps its
    # addresses).  With IAF flows the reference's loss is unbounded below (the flows' mean log-determinant is added
    # to every score, kgvae/link_predict.py:75-76) and a few dozen consecutive steps on one batch overflow.
    def snapshot():
        return ([p.detach().clone() for p in model.parameters()],
                [{k: v.clone() for k, v in opt.state[p].items() if torch.is_tensor(v)} for p in model.parameters() if p in opt.state])

    def restore(snap):
        with torch.no_grad():
            for p, v in zip(model.parameters(), snap[0]):
                p.copy_(v)
            for p, st in zip([p for p in model.parameters() if p in opt.state], snap[1]):
                for k, v in st.items():
                    opt.state[p][k].copy_(v)

    model.train()
    clocks.mark()
    for _ in range(max(args.warmup, 3)):
        step(resident)
    sync_all()
    snap = snapshot()
    # per-op CUDA-event times of the EAGER step (the op list under `roofline`, and the eager step time itself)
    L.launches = 0
    L.profile = {}
    ms_eager_prof = max_over_ranks(timed(lambda: step(resident), args.steps))
    launches = L.launches
    prof, L.profile = L.profile, None
    restore(snap)
    last_eager_loss = []

    def eager_step():
        # detached: an autograd graph that outlives its step would make the capture below fail
        last_eager_loss[:] = [step(resident).detach()]

    ms_eager = max_over_ranks(timed(eager_step, args.steps))
    if args.dump_outputs and args.eager and rank == 0:
        dump_step_outputs(args.dump_outputs, last_eager_loss[0], model)
    sync_all()
    restore(snap)
    captured = None
    if not args.eager:
        # the step's shapes are fixed (one sampled batch / the full graph): capture it once, replay it
        captured = K.link_predict.CapturedTrainStep(
            model, opt, {"node_id": resident["node_id"].view(-1, 1), "src": resident["src"], "dst": resident["dst"],
                         "etype": resident["etype"], "norm": resident["norm"], "samples": resident["samples"],
                         "labels": resident["labels"]}, N, buckets=buckets, grad_norm=1.0, warmup=max(args.warmup, 3))
        sync_all()
        restore(snap)
        launches = captured.launches_per_step * args.steps
        ms_dev = max_over_ranks(timed(lambda: captured.step(), args.steps))
        if args.dump_outputs and rank == 0:
            dump_step_outputs(args.dump_outputs, captured.loss, model)

        def step(t):                                            # e2e: new inputs copied into place, then the replay
            return captured.step(node_id=t["node_id"], src=t["src"], dst=t["dst"], etype=t["etype"], norm=t["norm"],
                                 samples=t["samples"], labels=t["labels"])
    else:
        ms_dev = ms_eager
    sync_all()
    restore(snap)
    for _ in range(2):
        e2e_step()
    timed_e2e(2)
    sync_all()
    restore(snap)
    ms_e2e = max_over_ranks(timed_e2e(args.steps))
    sync_all()
    log("  e2e losses read back: " + " ".join(f"{v:.4f}" for v in e2e_losses))
    if captured is not None:
        captured.close()        # a CUDA graph that holds NCCL kernels must be gone before its communicator is
        sync_all()
    # end to end INCLUDING the sampler (fresh sample every step), three ways
    restore(snap)
    timed_with_device_sampler(2)
    sync_all()
    ms_dev_sampler = max_over_ranks(timed_with_device_sampler(args.steps)) / args.steps
    # the same loop as ONE replay per step: the full-batch device sampler captured together with the train step
    ms_dev_sampler_captured = None
    if not args.eager and batch == len(data.train):
        restore(snap)
        torch.manual_seed(1000 + rank)
        sampler = K.utils.FullBatchDeviceSampler(train_dev, data.num_rels, NEG, split_size=0.5)
        cap2 = K.link_predict.CapturedTrainStep(model, opt, None, sampler.n, buckets=buckets, grad_norm=1.0, warmup=3,
                                                sampler=sampler)
        sync_all()

        def timed_captured_sampler(n_steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            got = []
            for i in range(n_steps):
                loss_host[i & 1].copy_(cap2.step().reshape(1), non_blocking=True)
                loss_done[i & 1].record()
                if i > 0:
                    loss_done[(i - 1) & 1].synchronize()
                    got.append(float(loss_host[(i - 1) & 1]))
            loss_done[(n_steps - 1) & 1].synchronize()
            got.append(float(loss_host[(n_steps - 1) & 1]))
            b.record()
            b.synchronize()
            return a.elapsed_time(b), got

        timed_captured_sampler(2)
        sync_all()
        ms_c, sampler_losses = timed_captured_sampler(args.steps)
        ms_dev_sampler_captured = max_over_ranks(ms_c) / args.steps
        log(f"  sampler + step as one replay: {ms_dev_sampler_captured:.3f} ms/step; losses " +
            " ".join(f"{v:.4f}" for v in sampler_losses))
        cap2.close()
        sync_all()
    ms_host_sampler = max_over_ranks(timed_with_host_sampler(args.steps, threaded=False)) / args.steps
    ms_host_threaded = max_over_ranks(timed_with_host_sampler(args.steps, threaded=True)) / args.steps
    sync_all()

    # ---- L2 throughput of this GPU for whole-row gathers / reductions (roofline denominator) --------
    l2_peak = None
    if rank == 0:
        l2_peak = measure_l2_peak(dev, N, H)
        log(f"  [l2 probe] read {l2_peak['read_gbs']:.0f} GB/s, reduce {l2_peak['reduce_gbs']:.0f} GB/s, "
            f"read+reduce {l2_peak['mixed_gbs']:.0f} GB/s")
    gemm_cmp = gemm_vs_library(dev, log) if (rank == 0 and world == 1) else None

    # ---- evaluation: encoder on the test graph + all-entity ranks -----------------------------
    model.eval()
    test = torch.from_numpy(data.test)
    tg, trel, tnorm = K.utils.build_test_graph(data.num_nodes, data.num_rels, test)
    t_ids = torch.arange(data.num_nodes, dtype=torch.int32, device=dev).view(-1, 1)
    t_rel = torch.from_numpy(trel).to(torch.int32).to(dev)
    t_norm = torch.from_numpy(tnorm[tg._dst].reshape(-1, 1).astype(np.float32)).to(dev)
    test_host = test.to(torch.int32).pin_memory()
    test_dev = test_host.to(dev)
    lo, hi = K.parallel.entity_shard(data.num_nodes, rank, world)

    # filtered setting (BASELINE.json configs[1]; an extension - the reference reports raw ranks only,
    # kgvae/link_predict.py:7): every other known-true candidate of a query (train + valid + test) is
    # taken out of the count inside the rank launch.  The filter lists are built once, outside the timing.
    known = np.concatenate([data.train, data.valid, data.test])
    filt_s = K.utils.build_filter(known, data.test[:, 2], data.test[:, 1], data.num_rels, "subject", dev)
    filt_o = K.utils.build_filter(known, data.test[:, 0], data.test[:, 1], data.num_rels, "object", dev)

    def eval_ranks(tt, filtered=False, emb=None):
        with torch.no_grad():
            if emb is None:                                 # the encoder runs (and samples z) on every evaluation
                emb = model(tg, t_ids, t_rel, t_norm)
            s, r, o = tt[:, 0].contiguous(), tt[:, 1].contiguous(), tt[:, 2].contiguous()
            shift = model._flow_shift()
            fs, fo = (filt_s, filt_o) if filtered else ((None, None), (None, None))
            rk = torch.cat([K.ops.distmult_rank(emb, model.w_relation, o, r, s, shift=shift, cand_range=(lo, hi),
                                                filt_ptr=fs[0], filt_idx=fs[1]),
                            K.ops.distmult_rank(emb, model.w_relation, s, r, o, shift=shift, cand_range=(lo, hi),
                                                filt_ptr=fo[0], filt_idx=fo[1])])
            if world > 1:                                   # entity-sharded counts add up
                dist.all_reduce(rk)
            return rk

    for _ in range(3):
        eval_ranks(test_dev)
    sync_all()
    L.profile = {}
    ms_eval = max_over_ranks(timed(lambda: eval_ranks(test_dev), args.steps))
    eval_prof, L.profile = L.profile, None
    ms_eval_e2e = max_over_ranks(timed(lambda: eval_ranks(test_host.to(dev, non_blocking=True)).cpu(), args.steps))
    sync_all()
    eval_ranks(test_dev, filtered=True)
    ms_eval_filt = max_over_ranks(timed(lambda: eval_ranks(test_dev, filtered=True), args.steps))
    with torch.no_grad():
        emb_once = model(tg, t_ids, t_rel, t_norm)          # one sample of z for the raw / filtered comparison
    rk_raw = eval_ranks(test_dev, emb=emb_once).float() + 1
    rk_filt = eval_ranks(test_dev, filtered=True, emb=emb_once).float() + 1
    # single-product tensor-core mode (north_star: reduced-precision GEMM variant, reported separately): one fp16
    # product per k-step instead of the fp32-accurate three-term split; ranks then carry the 11-bit operand rounding
    with K.ops.tensor_core_terms(1):
        eval_ranks(test_dev)
        L.profile = {}
        ms_eval_1p = max_over_ranks(timed(lambda: eval_ranks(test_dev), args.steps))
        prof_1p, L.profile = L.profile, None
        rk_1p = eval_ranks(test_dev, emb=emb_once).float() + 1
    d1p = (rk_1p - rk_raw).abs()
    single_product = {"value": len(data.test) * args.steps / (ms_eval_1p * 1e-3), "unit": "triples/s",
                      "ms": ms_eval_1p / args.steps,
                      "rank_launch_ms": (lambda e: sum(a.elapsed_time(b) for a, b in e) / len(e))(prof_1p["kg_distmult_rank"]),
                      "ranks_identical_frac": float((d1p == 0).float().mean()), "max_rank_diff": float(d1p.max()),
                      "mrr_exact": float((1.0 / rk_raw).mean()), "mrr_single_product": float((1.0 / rk_1p).mean()),
                      "what": "kg_set_tc_terms(1): operands rounded to 11 significant bits (per-row scaled fp16), no "
                              "fp32 re-scoring band; NOT the default - every parity claim is on the three-term mode"}
    mrr_raw, mrr_filt = float((1.0 / rk_raw).mean()), float((1.0 / rk_filt).mean())
    filt_ok = bool((rk_filt <= rk_raw).all())              # filtering can only improve a rank
    sync_all()
    clock_info = clocks.stop()

    # ---- BASELINE.json configs[4] inside the default job: the destination-partitioned wikikg2-shaped step at
    # this N (strong scaling; N = 1 is the unpartitioned denominator), and at N > 1 the partition parity checks
    partitioned = None
    if not args.no_partitioned and args.workload == "fb15k237-full":
        model = opt = buckets = None
        del resident
        torch.cuda.empty_cache()
        partitioned = {"what": "full-graph GCN-VAE train step, ogbl-wikikg2 shape (2.5 M entities, 32 M directed "
                               "edges, 176 M scored triplets), destination-partitioned over the N GPUs; strong "
                               "scaling: edges_per_s = 32 M / step time (max over ranks)", "modes": {}}
        if world > 1:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import partition_selfcheck
            partitioned["parity"] = partition_selfcheck.run_all(K, dev, rank, world)      # asserts
            log(f"  partition parity checks passed: {partitioned['parity']}")
        # the peer-memory gather measured 2.4x slower at N = 8 (profiles/r02f): only on request (--peer)
        legs = (("single", True),) if world == 1 else ((("allgather", True), ("peer", False)) if args.peer else (("allgather", True),))
        for name, ag in legs:
            partitioned["modes"][name] = partitioned_leg(args, dev, world, rank, log, allgather=ag, steps=args.steps, warmup=3,
                                                         scale=args.scale)
            log(f"  [wikikg2-part x{world}, {name}] {partitioned['modes'][name]['ms_per_step']:.1f} ms/step")
        best = min(partitioned["modes"].values(), key=lambda m: m["ms_per_step"])
        partitioned.update(ms_per_step=best["ms_per_step"], edges_per_s=best["edges_per_s"], n_gpus=world)
        sync_all()

    if rank != 0:
        leave_process_group(world)
        return

    # ---- roofline of the dominant kernel ------------------------------------------------------
    shp = {"N": N, "E": E, "S": S, "R2": 2 * data.num_rels, "R": data.num_rels}
    op_ms = {tag: sum(a.elapsed_time(b) for a, b in evs) for tag, evs in prof.items()}
    op_n = {tag: len(evs) for tag, evs in prof.items()}
    total_ops = sum(op_ms.values())
    top = sorted(op_ms.items(), key=lambda kv: -kv[1])
    for tag, ms in top[:14]:
        log(f"  {tag:44s} {ms / args.steps:8.3f} ms/step  {100 * ms / total_ops:5.1f}%  x{op_n[tag] // args.steps}")
    pk = peaks()
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    traffic = json.load(open(traffic_file)) if os.path.exists(traffic_file) else {}
    roof = None
    for tag, ms in top:
        ab = algorithmic_bytes(tag, shp)
        if ab is None:
            continue
        per_launch_ms = ms / op_n[tag]
        if l2_peak and (N * H * 4 <= 96 << 20):
            # Every matrix this launch gathers from / reduces into (z, dz, h: N x 500 fp32 = 29 MB) stays in the
            # 126 MB L2 - ncu: 2 % DRAM throughput - so the bound is L2, not HBM.  achieved = the launch's
            # algorithmic L2 bytes per second (per scored triplet one whole row of z read and one whole row reduced
            # into dz; per message-passing edge one row gathered and one row of `out` floats reduced); peak = what
            # kg_probe_l2 sustains for the same mix of whole-row reads and reductions on this GPU, measured in
            # this process a moment ago.
            if tag == "kg_distmult_bce_fwd":
                l2_bytes, mix = S * 2 * 4 * H, "mixed"
            elif tag.startswith("kg_bdd_rel"):
                si, so = (int(x) for x in tag[tag.index("[") + 1:-1].split("x"))
                l2_bytes = E * 4 * BASES * (si + so) * (2 if "bwd" in tag else 1)
                mix = "mixed"
            else:
                l2_bytes, mix = ab, "read"
            ach = l2_bytes / (per_launch_ms * 1e-3) / 1e9
            roof = {"kernel": tag, "bound": "l2", "achieved": ach, "peak": l2_peak[mix + "_gbs"], "unit": "GB/s",
                    "frac": ach / l2_peak[mix + "_gbs"], "traffic": traffic.get(tag + ":lts_bytes"),
                    "peak_source": "kg_probe_l2, measured in this run (random whole-row reads + reductions on two "
                                   "L2-resident 29 MB matrices)",
                    "ms_per_launch": per_launch_ms, "algorithmic_bytes": l2_bytes, "share_of_step": ms / total_ops,
                    "dram_traffic": traffic.get(tag), "hbm_algorithmic_bytes": ab,
                    "regime": "L2-resident (z, dz, h are 29 MB each; L2 is 126 MB): bounded by L2, not HBM",
                    "l2_probe": l2_peak}
        else:
            ach = ab / (per_launch_ms * 1e-3) / 1e9
            roof = {"kernel": tag, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / pk["hbm_gbs"], "traffic": traffic.get(tag), "peak_source": pk["source"],
                    "ms_per_launch": per_launch_ms, "algorithmic_bytes": ab, "share_of_step": ms / total_ops}
        break
    eval_top = sorted(((t, sum(a.elapsed_time(b) for a, b in e) / len(e)) for t, e in eval_prof.items()),
                      key=lambda kv: -kv[1])
    T = len(data.test)
    rank_ms = dict(eval_top).get("kg_distmult_rank")
    eval_roof = None
    if rank_ms:
        # algorithmic work of one launch (one perturbation direction): 2*T*V*h flops.  The kernel
        # executes 3x that on the tensor cores (two-term fp16 split: lo*hi + hi*lo + hi*hi, K padded
        # to a multiple of 64) so that the fp32 decision is kept; both figures are reported.
        flops = 2.0 * T * (hi - lo) * H
        kp = (H + 63) // 64 * 64
        executed = 3.0 * 2.0 * T * (hi - lo) * kp
        eval_roof = {"kernel": "kg_distmult_rank (rank_tc_kernel, tcgen05 kind::f16)", "bound": "tensor",
                     "achieved": flops / (rank_ms * 1e-3) / 1e12, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": flops / (rank_ms * 1e-3) / 1e12 / pk["bf16_tflops"],
                     "executed_tflops": executed / (rank_ms * 1e-3) / 1e12,
                     "executed_frac": executed / (rank_ms * 1e-3) / 1e12 / pk["bf16_tflops"],
                     "ms_per_launch": rank_ms,
                     "note": "achieved = algorithmic fp32 flops (2*T*V*h); executed = tensor-core flops "
                             "of the fp32-exact two-term fp16 split (3 products, K padded to 512); the "
                             "launch time includes the operand split kernels; peak = measured bf16 sustained"}

    streaming = None
    if world == 1 and not args.no_streaming:
        model = opt = buckets = None
        torch.cuda.empty_cache()
        streaming = streaming_layer_bench(dev, pk, log, l2_peak=l2_peak)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_oracle_rates(2, 1, args.n_flows, sample_edges=batch, log=log, shape=shape)
        cpu = {"value": r["train_edges_per_s"], "unit": "edges/s", "cores": r["cores"], "kind": "port",
               "sample": r["sample"], "eval_triples_per_s": r["eval_triples_per_s"], "anomaly_on": r.get("anomaly_on")}

    # the driver's record keeps `roofline` and `config` but not free-form keys: the HBM-bound and tensor-bound
    # launches and the evaluation figures are folded into `roofline` so that they are part of the record
    eval_summary = {"value": T * args.steps / (ms_eval * 1e-3), "unit": "triples/s", "ms": ms_eval / args.steps,
                    "filtered_value": T * args.steps / (ms_eval_filt * 1e-3),
                    "setting": f"{T} test triples x 2 directions x {data.num_nodes} candidates, encoder included"}
    if roof is not None:
        roof["tensor"] = eval_roof
        if eval_roof is not None:
            flops_1p = 2.0 * len(data.test) * (hi - lo) * H
            single_product["algorithmic_tflops"] = flops_1p / (single_product["rank_launch_ms"] * 1e-3) / 1e12
            single_product["frac_of_bf16_sustained"] = single_product["algorithmic_tflops"] / pk["bf16_tflops"]
            eval_roof["single_product"] = single_product
        roof["eval"] = eval_summary
        roof["partitioned"] = partitioned
        roof["gemm_vs_library"] = gemm_cmp
        if streaming:
            # each streaming launch against the resource that binds it: HBM for the launches whose HBM floor is the larger
            # one, the L2 reduction rate (probe) for the 5x10 forward, which reduces 4 KB per edge for 2 KB gathered
            ks = streaming["kernels"]["uniform"]
            hbm_bound = {k_: v for k_, v in ks.items() if v.get("bound", "hbm") == "hbm"} or ks
            worst = min(hbm_bound.items(), key=lambda kv: kv[1]["frac_of_hbm_peak"])
            roof["hbm"] = {"kernel": worst[0] + " @ wikikg2 shape (2.5 M nodes, 32 M edges)", "bound": "hbm",
                           "achieved": worst[1]["achieved_gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s",
                           "frac": worst[1]["frac_of_hbm_peak"], "traffic": traffic.get(worst[0] + ":streaming"),
                           "peak_source": pk["source"], "ms_per_launch": worst[1]["ms"],
                           "algorithmic_bytes": worst[1]["algorithmic_bytes"],
                           "note": "the HBM-bound message-passing launch furthest below the HBM roofline in the "
                                   "streaming regime; all four launches under rgcn_streaming"}
            red_bound = {k_: v for k_, v in ks.items() if v.get("bound") == "l2 reductions"}
            if red_bound:
                w2 = min(red_bound.items(), key=lambda kv: kv[1]["frac_of_l2_reduce_probe"])
                roof["l2_reduction"] = {
                    "kernel": w2[0] + " @ wikikg2 shape (2.5 M nodes, 32 M edges)", "bound": "l2",
                    "achieved": w2[1]["l2_reduce_gbs"], "peak": l2_peak["reduce_gbs"], "unit": "GB/s",
                    "frac": w2[1]["frac_of_l2_reduce_probe"], "ms_per_launch": w2[1]["ms"],
                    "algorithmic_bytes": w2[1]["reduce_bytes"], "frac_of_hbm_peak": w2[1]["frac_of_hbm_peak"],
                    "traffic": traffic.get(w2[0] + ":streaming"),
                    "peak_source": "kg_probe_l2 (whole-row reductions into an L2-resident matrix), measured in this run",
                    "note": "every edge's message is reduced into an L2-resident tile: 4 KB reduced per edge for 2 KB "
                            "gathered, so the L2 reduction rate binds this launch, not HBM (frac_of_hbm_peak for reference)"}

    total_edges = E * world * args.steps
    line = {
        "metric": METRIC, "value": total_edges / (ms_dev * 1e-3), "unit": "edges/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args, data, N, E, S, world),
        "e2e": {"value": total_edges / (ms_e2e * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                "losses_read_back": [float(v) for v in e2e_losses],
                "how": "pinned host inputs copied every step inside the timed region (double-buffered on a side "
                       "stream: step i+1's copy overlaps step i), every step's loss copied to pinned host memory and "
                       "read by the host one step later (all K losses are read inside the region), L2 flush inside",
                "with_sampler": {
                    "what": "kgvae/link_predict.py:200-236 with a FRESH sample every step: sampler + copies + edge "
                            "index + step + loss read-back; ms per step, max over ranks",
                    "device_sampler_ms": ms_dev_sampler, "device_sampler_edges_per_s": E * world / (ms_dev_sampler * 1e-3),
                    "device_sampler_captured_ms": ms_dev_sampler_captured,
                    "device_sampler_captured_edges_per_s": (E * world / (ms_dev_sampler_captured * 1e-3)
                                                            if ms_dev_sampler_captured else None),
                    "device_sampler_captured_what": "utils.FullBatchDeviceSampler drawn INSIDE the captured step "
                                                    "(link_predict.CapturedTrainStep(sampler=...)): one CUDA-graph "
                                                    "replay per training iteration, loss read back every step",
                    "host_sampler_ms": ms_host_sampler, "host_sampler_edges_per_s": E * world / (ms_host_sampler * 1e-3),
                    "host_sampler_threaded_ms": ms_host_threaded,
                    "note": "the host sampler is the reference's numpy code (bit-exact sampled indices), single "
                            "threaded by construction; --device-sampler is the fast path"}},
        "eval": {"value": T * args.steps / (ms_eval * 1e-3), "unit": "triples/s", "test_triples": T,
                 "candidates": data.num_nodes, "ms": ms_eval / args.steps, "setting": "raw, both directions",
                 "e2e_value": T * args.steps / (ms_eval_e2e * 1e-3), "mrr_raw_random_init": mrr_raw,
                 "filtered": {"value": T * args.steps / (ms_eval_filt * 1e-3), "unit": "triples/s",
                              "ms": ms_eval_filt / args.steps, "mrr_random_init": mrr_filt,
                              "known_triples": int(len(known)), "never_worse_than_raw": filt_ok,
                              "setting": "filtered (train + valid + test), both directions, same launch + correction"},
                 "roofline": eval_roof},
        "scored_triplets_per_s": S * world * args.steps / (ms_dev * 1e-3),
        "step_mode": {"mode": "eager" if captured is None else "CUDA graph replay (link_predict.CapturedTrainStep)",
                      "eager_ms_per_step": ms_eager / args.steps,
                      "eager_ms_per_step_with_op_events": ms_eager_prof / args.steps,
                      "note": "the eager step issues ~150 launches through autograd + ctypes and is host-bound; the "
                              "captured step replays the same kernels on the same buffers in one launch"},
        "gpu_launches": launches, "clocks": clock_info, "roofline": roof, "cpu_baseline": cpu,
        "rgcn_streaming": streaming, "partitioned": partitioned,
    }
    print(json.dumps(line), flush=True)
    leave_process_group(world)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of every train-step and evaluation loop on the GPU; the CPU baseline (2 steps) "
                         "and the GEMM, L2 and streaming probes keep their fixed repetition counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="fb15k237-full",
                    choices=["fb15k237-full", "fb15k237-step", "wn18-full", "wn18-step", "wikikg2-part", "am-entity"],
                    help="fb15k237-full is the headline (BASELINE.json configs[1]); wn18-* with --n-flows 3 is configs[2]; "
                         "am-entity is configs[3] (entity classification, basis RGCN); wikikg2-part is configs[4]")
    ap.add_argument("--n-flows", type=int, default=0)
    ap.add_argument("--bases", type=int, default=None,
                    help="bdd blocks per relation (default 100; 25 at wn18 shape: DGL clamps num_bases to the "
                         "36 directed relation types, which does not divide 500)")
    ap.add_argument("--scale", type=float, default=1.0, help="wikikg2-part / am-entity: shrink the graph (tests)")
    ap.add_argument("--peer", action="store_true",
                    help="wikikg2-part: the message-passing kernels gather layer inputs from peer HBM (CUDA IPC over "
                         "NVLink) instead of the NCCL all-gather")
    ap.add_argument("--replicas", action="store_true",
                    help="am-entity with N > 1: independent replicas (weak scaling) instead of one graph over the N GPUs")
    ap.add_argument("--col-chunks", type=int, default=0,
                    help="partitioned step: column chunks the layer-input all-gather / source-gradient reduce-scatter are "
                         "pipelined in (1 = one collective per layer; 0 = by world size: 2 from 4 GPUs up)")
    ap.add_argument("--no-partitioned", action="store_true",
                    help="skip the wikikg2-shaped destination-partitioned leg of the default workload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true",
                    help="time the eager train step instead of the CUDA-graph replay of it")
    ap.add_argument("--streaming-only", action="store_true",
                    help="run only the wikikg2-shaped message-passing leg (profiling aid; prints its JSON object)")
    ap.add_argument("--no-streaming", action="store_true",
                    help="skip the wikikg2-shaped message-passing leg (HBM-streaming regime, N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss, parameters and gradients to DIR/<name>.npy "
                         "(link-prediction workloads of this repo's CUDA path)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.streaming_only or args.workload in ("wikikg2-part", "am-entity")):
        ap.error("--dump-outputs writes the outputs of the link-prediction train step: use it with --impl b200 and a "
                 "fb15k237-* / wn18-* workload")
    global BASES
    BASES = args.bases if args.bases else (25 if args.workload.startswith("wn18") else 100)
    if args.streaming_only:
        dev = torch.device("cuda", 0)
        torch.cuda.set_device(dev)
        print(json.dumps(streaming_layer_bench(dev, peaks(), lambda m: print(m, file=sys.stderr, flush=True),
                                               iters=max(1, args.steps))))
    elif args.impl == "reference":
        run_reference(args)
    elif args.workload == "wikikg2-part":
        run_partitioned(args)
    elif args.workload == "am-entity":
        run_entity(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
