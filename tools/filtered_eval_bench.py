"""Cost of filtered evaluation and filtered generation on the GPU.

Per shape - FB15k-237 (uniform and Zipf skew 1.0) and wikikg2 (h = 500), triples from datasets.synthetic_kg, the
known set is train + valid + test:

  build     the filter lists of the whole test set in both directions: utils.FilterIndex (the two device tables, from
            known triples already on the device) plus FilterIndex.lists for the (s, r, ?) and (o, r, ?) queries,
            against utils.build_filter on the host (numpy, both directions, host clock, --host-reps runs); the GPU
            lists are checked to equal the host ones
  rank      kg_distmult_rank raw against filtered (both directions, lists built beforehand)
  topk      kg_distmult_topk against kg_distmult_topk_filtered, k = 10, the (s, r, ?) queries; also per kernel
            (torch.profiler, device time, in a pass of its own), with the real lists and with empty ones - the
            filtered kernels on lists that exclude nothing, whose output equals the unfiltered one

GPU times are CUDA events after warm-up, median of --reps runs, raw and filtered alternated run by run.  Entity
embeddings and relation vectors are Gaussian; at FB15k-237 they are L2-resident (29 MB), as in bench.py's
evaluation.  At the wikikg2 shape rank and top-k run on the first --wiki-queries test triples (the top-k candidate
lists of all 599 k queries would need 0.5 TB of workspace).  The card's name, power limit and maximum SM clock are
read with nvidia-smi in the same run.

    python tools/filtered_eval_bench.py --out-dir OUT [--reps 10 --host-reps 1 --wiki-queries 4096]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import gcn_vae_b200 as K  # noqa: E402

H, TOPK = 500, 10
# (label, shape, skew, query limit for rank / top-k: None = the whole test set)
SHAPES = [("FB15k-237", "FB15k-237", 0.0, None), ("FB15k-237 skew 1.0", "FB15k-237", 1.0, None),
          ("wikikg2", "wikikg2", 0.0, "wiki")]


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True)
    name, power, clock = (x.strip() for x in q.stdout.strip().splitlines()[0].split(","))
    return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def alternate(fns, reps, warmup=2):
    """median ms of each callable, run in turn rep by rep after ``warmup`` rounds"""
    for _ in range(warmup):
        for fn in fns:
            fn()
    torch.cuda.synchronize()
    times = [[] for _ in fns]
    for _ in range(reps):
        for t, fn in zip(times, fns):
            t.append(event_ms(fn))
    return [float(np.median(t)) for t in times]


def kernel_ms(fn, reps=3):
    """device ms per call of each kernel fn launches (torch.profiler), after one warm-up call"""
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            name = e.name.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
            out[name] = out.get(name, 0.0) + e.device_time / reps / 1e3
    return {k: round(v, 4) for k, v in sorted(out.items(), key=lambda kv: -kv[1]) if v >= 0.005}


def run_shape(label, shape, skew, limit, args, dev):
    d = K.datasets.synthetic_kg(shape, seed=0, skew=skew)
    N, R = d.num_nodes, d.num_rels
    known = np.concatenate([d.train, d.valid, d.test])
    test = d.test
    out = {"label": label, "entities": N, "relations": R, "known_triples": len(known), "test_queries": len(test),
           "key_bits": 2 * int(np.ceil(np.log2(N))) + int(np.ceil(np.log2(R)))}

    # ---- filter build: host reference against the device index -------------------------------
    host_s = []
    for _ in range(args.host_reps):
        t0 = time.perf_counter()
        want_o = K.utils.build_filter(known, test[:, 0], test[:, 1], R, "object", "cpu")
        want_s = K.utils.build_filter(known, test[:, 2], test[:, 1], R, "subject", "cpu")
        host_s.append(time.perf_counter() - t0)
    known_dev = torch.from_numpy(known).to(dev)
    s, r, o = (torch.from_numpy(test[:, i]).to(torch.int32).to(dev) for i in range(3))

    def build():
        fi = K.utils.FilterIndex(known_dev, N, R, dev)
        return fi, fi.lists(s, r, "object"), fi.lists(o, r, "subject")

    fi, lists_o, lists_s = build()
    for got, want in ((lists_o, want_o), (lists_s, want_s)):
        assert torch.equal(got[0].cpu(), want[0]) and torch.equal(got[1].cpu(), want[1]), label
    tables_ms, lists_ms = alternate([lambda: K.utils.FilterIndex(known_dev, N, R, dev),
                                     lambda: (fi.lists(s, r, "object"), fi.lists(o, r, "subject"))], args.reps)
    total_ms = alternate([build], args.reps)[0]
    lens = (lists_o[0][1:] - lists_o[0][:-1]).float()
    out["build"] = {"host_build_filter_s": float(np.median(host_s)), "gpu_total_ms": total_ms,
                    "gpu_tables_ms": tables_ms, "gpu_lists_ms": lists_ms,
                    "speedup": float(np.median(host_s)) * 1e3 / total_ms,
                    "listed_object": int(lists_o[1].numel()), "listed_subject": int(lists_s[1].numel()),
                    "object_list_len_mean": float(lens.mean()), "object_list_len_max": int(lens.max())}
    del known_dev

    # ---- rank raw / filtered, top-k raw / filtered ----------------------------------------------
    M = len(test) if limit is None else min(len(test), args.wiki_queries)
    gen = torch.Generator(device=dev).manual_seed(0)
    emb = torch.randn(N, H, device=dev, generator=gen) / H ** 0.25
    w = torch.randn(R, H, device=dev, generator=gen) / H ** 0.25
    sq, rq, oq = s[:M].contiguous(), r[:M].contiguous(), o[:M].contiguous()
    fo = fi.lists(sq, rq, "object")
    fs = fi.lists(oq, rq, "subject")
    rank = lambda f_s, f_o: (K.ops.distmult_rank(emb, w, oq, rq, sq, filt_ptr=f_s[0], filt_idx=f_s[1]),
                             K.ops.distmult_rank(emb, w, sq, rq, oq, filt_ptr=f_o[0], filt_idx=f_o[1]))
    none = (None, None)
    raw_ms, filt_ms = alternate([lambda: rank(none, none), lambda: rank(fs, fo)], args.reps)
    rk_raw, rk_filt = (torch.cat(x).float() + 1 for x in (rank(none, none), rank(fs, fo)))
    out["rank"] = {"queries": 2 * M, "raw_ms": raw_ms, "filtered_ms": filt_ms, "filtered_over_raw": filt_ms / raw_ms,
                   "mrr_raw": float((1 / rk_raw).mean()), "mrr_filtered": float((1 / rk_filt).mean())}
    topk = lambda f: K.ops.distmult_topk(emb, w, sq, rq, k=TOPK, filt_ptr=f[0], filt_idx=f[1])
    un_ms, fk_ms = alternate([lambda: topk(none), lambda: topk(fo)], args.reps)
    idx_f = topk(fo)[0]
    empty = (torch.zeros(M + 1, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev))
    assert torch.equal(topk(empty)[0], topk(none)[0]), label
    out["topk"] = {"queries": M, "k": TOPK, "unfiltered_ms": un_ms, "filtered_ms": fk_ms,
                   "filtered_over_unfiltered": fk_ms / un_ms,
                   "rows_with_trailing_minus1": int((idx_f[:, -1] < 0).sum()),
                   "kernel_ms": {"unfiltered": kernel_ms(lambda: topk(none)), "filtered": kernel_ms(lambda: topk(fo)),
                                 "filtered_empty_lists": kernel_ms(lambda: topk(empty))}}
    del emb, w
    torch.cuda.empty_cache()
    return out


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--out-dir", required=True, help="directory that receives filtered_eval_bench.json")
    p.add_argument("--reps", type=int, default=10)
    p.add_argument("--host-reps", type=int, default=1)
    p.add_argument("--wiki-queries", type=int, default=4096)
    p.add_argument("--only", default=None, help="run the shapes whose label contains this string")
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("filtered_eval_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    result = {"tool": "tools/filtered_eval_bench.py", "gpu": gpu_info(0), "h": H, "reps": args.reps,
              "wiki_queries": args.wiki_queries, "shapes": []}
    for label, shape, skew, limit in SHAPES:
        if args.only and args.only not in label:
            continue
        res = run_shape(label, shape, skew, limit, args, dev)
        print(json.dumps(res), flush=True)
        result["shapes"].append(res)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "filtered_eval_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
