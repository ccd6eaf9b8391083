"""The device neighbourhood-expansion edge sampler (kg_neighbor_sample, --edge-sampler neighbor) against the host one.

Per shape (FB15k-237, FB15k-237 at Zipf skew 1.0, wn18, and the wikikg2 entity count, whose per-sample state does
not fit shared memory):

  host      one draw of utils.sample_edge_neighborhood (the reference's loop, numpy, one thread), host clock; at the
            wikikg2 shape the first --host-picks picks are timed and scaled to B (the loop is O(B N));
  refill    NeighborEdgeBank.refill(): the K x B x 8 words from torch's generator plus one kernel launch drawing the
            K samples of the bank; CUDA events, median of --refills refills after one warm-up; also per sample;
  kernel    the launch alone, CUDA events, median of --refills launches;
  fallback  the share of picks that needed the unpicked-entry scan (all R rejection tries hit picked edges).

At the FB15k-237 shape it also times the training iteration of --capture-step --device-sampler (one CUDA-graph
replay per iteration, the model of bench.py) with the neighbour sampler against the uniform sampler, alternating the
two round by round; the neighbour loop refills its bank between replays, and the rounds together cover at least two
refills.  The card's name, power limit and maximum SM clock are read with nvidia-smi in the same run.

    python tools/neighbor_sampler_bench.py --out-dir OUT [--refills 5 --rounds 3 --steps 250]
"""
import argparse
import copy
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import gcn_vae_b200 as K  # noqa: E402

B = 20000
H, BASES, MOG_K, DROPOUT, NEG, REG, KL, SPLIT = 500, 100, 10, 0.2, 10, 0.01, 1e-5, 0.5
# (label, shape, skew, triple scale, sample size)
SHAPES = [("FB15k-237", "FB15k-237", 0.0, 1.0, B), ("FB15k-237 skew 1.0", "FB15k-237", 1.0, 1.0, B),
          ("wn18", "wn18", 0.0, 1.0, B), ("wikikg2 entities, 0.001 of its triples", "wikikg2", 0.0, 0.001, 8000)]


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True)
    name, power, clock = (x.strip() for x in q.stdout.strip().splitlines()[0].split(","))
    return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}


def events_ms(fn, n):
    out = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


def bench_shape(label, shape, skew, scale, b, args, dev):
    data = K.datasets.synthetic_kg(shape, seed=0, skew=skew, scale=scale)
    T, n = len(data.train), data.num_nodes
    adj, deg = K.utils.get_adj_and_degrees(n, data.train)
    np.random.seed(0)
    picks = b if shape != "wikikg2" else min(b, args.host_picks)
    t0 = time.perf_counter()
    K.utils.sample_edge_neighborhood(adj, deg, T, picks)
    host_s = (time.perf_counter() - t0) * b / picks

    bank = K.utils.NeighborEdgeBank(torch.from_numpy(data.train).to(dev), n, b)
    bank.refill()
    torch.cuda.synchronize()
    refill = events_ms(bank.refill, args.refills)
    fb = torch.zeros(bank.K, dtype=torch.int32, device=dev)
    launch = lambda: K.ops.neighbor_sample(bank.adj_ptr, bank.adj, n, b, bank.words, out=bank.bank, fallbacks=fb,
                                           workspace=bank.workspace)
    kernel = events_ms(launch, args.refills)
    distinct = [len(np.unique(data.train[r][:, [0, 2]])) for r in bank.bank[:8].cpu().numpy()]
    med = float(np.median(refill))
    return {"label": label, "shape": shape, "skew": skew, "triple_scale": scale, "entities": n, "triples": T,
            "sample_size": b, "max_degree": int(deg.max()), "samples_per_launch": bank.K,
            "state_in_shared_memory": bank.workspace.numel() <= 16,
            "host_draw_s": host_s, "host_draw_timed_picks": picks,
            "refill_ms": med, "refill_ms_all": refill, "refill_ms_per_sample": med / bank.K,
            "kernel_ms": float(np.median(kernel)), "kernel_ms_all": kernel,
            "fallback_share": float(fb.sum().item()) / (bank.K * b),
            "distinct_entities_mean_of_8": float(np.mean(distinct)),
            "host_over_amortised_device": host_s * 1e3 / (med / bank.K)}


def bench_capture(args, dev):
    data = K.datasets.synthetic_kg("FB15k-237", seed=0)
    train_dev = torch.from_numpy(np.asarray(data.train)).to(dev)
    torch.manual_seed(0)
    base = K.LinkPredict(K.KGVAE, data.num_nodes, H, data.num_rels, num_bases=BASES, dropout=DROPOUT, use_cuda=True,
                         reg_param=REG, kl_param=KL, k=MOG_K).to(dev)
    loops = {}
    for kind in ("uniform", "neighbor"):
        m = copy.deepcopy(base).train()
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, fused=True, capturable=True)
        sm = K.utils.SampledDeviceSampler(train_dev, B, SPLIT, data.num_rels, NEG, edge_sampler=kind)
        loops[kind] = (sm, K.link_predict.CapturedTrainStep(m, opt, None, sm.n, grad_norm=1.0, warmup=3, sampler=sm))
    bank = loops["neighbor"][0].bank
    steps = max(args.steps, math.ceil((2 * bank.K + 1) / args.rounds))
    for _, cap in loops.values():
        for _ in range(5):
            cap.step()
    torch.cuda.synchronize()
    refills0 = bank.refills
    ms = {k: [] for k in loops}
    last = {}
    for _ in range(args.rounds):
        for kind, (_, cap) in loops.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                loss = cap.step()
            b.record()
            b.synchronize()
            ms[kind].append(a.elapsed_time(b) / steps)
            last[kind] = float(loss)
    out = {"shape": "FB15k-237", "sample_size": B, "h": H, "bases": BASES, "mog_k": MOG_K, "steps_per_round": steps,
           "rounds": args.rounds, "bank_rows": bank.K, "refills_in_timed_rounds": bank.refills - refills0}
    for kind in loops:
        out[kind] = {"ms_per_iter": float(np.median(ms[kind])), "ms_per_iter_rounds": ms[kind],
                     "last_loss": last[kind], "node_budget": loops[kind][0].n}
    out["neighbor_over_uniform"] = out["neighbor"]["ms_per_iter"] / out["uniform"]["ms_per_iter"]
    for _, cap in loops.values():
        cap.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--refills", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=250, help="captured iterations per loop and round (at least 50)")
    ap.add_argument("--host-picks", type=int, default=200, help="picks timed on the host at the wikikg2 shape")
    ap.add_argument("--gpu", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("neighbor_sampler_bench needs a CUDA device")
    if args.steps < 50 or args.rounds < 2:
        raise ValueError("--steps must be at least 50 and --rounds at least 2")
    torch.cuda.set_device(args.gpu)
    dev = torch.device("cuda", args.gpu)
    result = {"gpu": gpu_info(args.gpu), "words_per_pick": K.ops.NEIGHBOR_WORDS,
              "rejection_tries": K.ops.NEIGHBOR_TRIES, "shapes": []}
    for label, shape, skew, scale, b in SHAPES:
        r = bench_shape(label, shape, skew, scale, b, args, dev)
        print(f"{label}: host {r['host_draw_s']:.2f} s, refill of {r['samples_per_launch']} samples "
              f"{r['refill_ms']:.2f} ms ({r['refill_ms_per_sample']:.4f} ms per sample, kernel {r['kernel_ms']:.2f} "
              f"ms), fallback share {r['fallback_share']:.4f}", flush=True)
        result["shapes"].append(r)
    c = bench_capture(args, dev)
    print(f"FB15k-237 captured iteration: uniform {c['uniform']['ms_per_iter']:.3f} ms, neighbour "
          f"{c['neighbor']['ms_per_iter']:.3f} ms ({c['refills_in_timed_rounds']} refills)", flush=True)
    result["capture"] = c
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "neighbor_sampler_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"gpu": result["gpu"], "refill_ms": {s["label"]: s["refill_ms"] for s in result["shapes"]},
                      "capture_ms": [c["uniform"]["ms_per_iter"], c["neighbor"]["ms_per_iter"]]}))


if __name__ == "__main__":
    main()
