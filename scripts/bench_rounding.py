#!/usr/bin/env python
"""Hyperplane rounding on C5 (MaxCut, 10M-vertex power-law graph, rank 10: the graph and seed of bench.py), with R after a
few sdplrp_iterate steps.  Prints one JSON line:
  - CUDA-event time on the handle's stream of sdplrp_round_hyperplane for K = 64 and K = 1024 (ms per call, per 64
    candidates), and the sign / evaluation pass kernel times from a separate torch.profiler run;
  - the algorithmic bytes and flops of each pass, the achieved rates and the share of the bound that applies;
  - the card name and power limit, read in the same run;
  - the NumPy / SciPy host time for K = 8 on the downloaded R, and an exact cross-check of those 8 candidates.
Writes nothing into the tree (--out FILE copies the JSON line to FILE)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 7700.0       # HGX B200 data sheet, one GPU
FP64_TFLOPS = 37.0     # HGX B200 data sheet, one GPU, FP64


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vertices", dest="n", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=80_000_000)
    ap.add_argument("--rank", type=int, default=10)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--iters", type=int, default=5, help="sdplrp_iterate steps before rounding")
    ap.add_argument("--reps", type=int, default=5, help="timed calls per K")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import scipy.sparse as sps
    import sdplrplus.jl_b200 as sp
    from bench import SimpleData, generate, pinned_uniform
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}), flush=True)
        return 2
    n, r = args.n, args.rank
    handle = sp.Handle(device=0)
    asm, b, _, E, _ = generate(sp, n, args.edges, args.seed, keep_on_device=False)
    eng = sp.B200Engine(SimpleData(n, n, b), handle=handle, asm=asm)
    nnzT, nnzF, _ = handle.pattern_sizes()
    _, R0 = pinned_uniform((n, r), 0)
    eng.init_vars(r, R0, np.zeros(n), 2.0, 4)
    eng.fg()
    eng.iterate(args.iters)
    stream = torch.cuda.ExternalStream(handle.stream)

    eng.round_hyperplane(64, seed=1)      # warm-up: first launches, first-use buffers
    eng.round_hyperplane(1024, seed=1)
    timing = {}
    for K in (64, 1024):
        ms = []
        for rep in range(args.reps):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            eng.round_hyperplane(K, seed=100 + rep)
            ev1.record(stream)
            torch.cuda.synchronize()
            ms.append(ev0.elapsed_time(ev1))
        timing[K] = {"ms_per_call_median": float(np.median(ms)), "ms_per_call_all": ms,
                     "ms_per_64_candidates": float(np.median(ms)) / (K / 64)}

    # kernel split (separate run: the profiler slows the host)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.round_hyperplane(1024, seed=7)
        torch.cuda.synchronize()
    kern = {"sign": [0.0, 0], "eval": [0.0, 0], "other": [0.0, 0]}
    for evt in prof.key_averages():
        dev_us = getattr(evt, "device_time_total", None)
        if dev_us is None:
            dev_us = getattr(evt, "cuda_time_total", 0.0)
        key = "sign" if "k_round_sign" in evt.key else ("eval" if "k_round_eval" in evt.key else "other")
        if dev_us > 0:
            kern[key][0] += dev_us / 1e3
            kern[key][1] += evt.count
    batches = 1024 // 64
    sign_ms = kern["sign"][0] / max(1, kern["sign"][1])
    eval_ms = kern["eval"][0] / max(1, kern["eval"][1])
    lo, hi = handle.row_range()
    # algorithmic work of one batch of 64 candidates
    sign_bytes = 8.0 * r * n + 8.0 * n                                    # R read once, one word written per vertex
    sign_flops = 2.0 * 64 * r * n
    eval_bytes = 12.0 * nnzF + 4.0 * (n + 1) + 8.0 * nnzF + 8.0 * n       # index + value per entry, row pointers, one word per entry and per row
    eval_updates = 64.0 * nnzF                                             # candidate accumulations (predicated FP64 adds)
    passes = {
        "sign": {"ms_per_batch": sign_ms, "launches": kern["sign"][1], "bytes": sign_bytes, "flops": sign_flops,
                 "GBs": sign_bytes / (sign_ms * 1e-3) / 1e9, "GFLOPs": sign_flops / (sign_ms * 1e-3) / 1e9,
                 "bound": "FP64 FMA (data sheet 37 TFLOP/s)" if sign_flops / FP64_TFLOPS / 1e12 > sign_bytes / HBM_GBS / 1e9 else "HBM",
                 "share_of_bound": max(sign_flops / (FP64_TFLOPS * 1e12), sign_bytes / (HBM_GBS * 1e9)) / (sign_ms * 1e-3)},
        "eval": {"ms_per_batch": eval_ms, "launches": kern["eval"][1], "bytes": eval_bytes, "candidate_adds": eval_updates,
                 "GBs": eval_bytes / (eval_ms * 1e-3) / 1e9, "Gadds": eval_updates / (eval_ms * 1e-3) / 1e9,
                 "bound": "FP64 add issue (data sheet 37 TFLOP/s = 18.5e12 FP64 instructions/s)"
                          if eval_updates / 18.5e12 > eval_bytes / HBM_GBS / 1e9 else "HBM",
                 "share_of_bound": max(eval_updates / 18.5e12, eval_bytes / (HBM_GBS * 1e9)) / (eval_ms * 1e-3)},
        "other_kernels_ms_per_call": kern["other"][0],
        "batches_profiled": batches,
    }

    # host reference for K = 8 on the downloaded R, and an exact cross-check of those candidates
    R = eng.get_R()
    res = eng.round_hyperplane(8, seed=3)
    G = res["G_used"]
    I_, J_, V_ = asm.I, asm.J, asm.V
    c0, c1 = int(asm.mat_off[n]), int(asm.mat_off[n + 1])
    C = sps.csr_matrix((V_[c0:c1], (I_[c0:c1] - 1, J_[c0:c1] - 1)), shape=(n, n))
    del I_, J_, V_
    t0 = time.perf_counter()
    D = R @ G.T
    X = np.where(D >= 0, 1.0, -1.0)
    obj = np.einsum("ik,ik->k", X, C @ X)
    tot = X.sum(axis=0)
    host_s = time.perf_counter() - t0
    scale = np.linalg.norm(R, axis=1)[:, None] * np.linalg.norm(G, axis=1)[None, :]
    amb = np.any(np.abs(D) <= 1e-12 * scale, axis=0)
    ok = ~amb
    try:
        from threadpoolctl import threadpool_info
        threads = {i.get("internal_api", "?"): i.get("num_threads") for i in threadpool_info()}
    except Exception:
        threads = {"os.cpu_count": os.cpu_count(), "note": "threadpoolctl unavailable; SciPy sparse products are single-threaded"}
    check = {"candidates": 8, "ambiguous": int(amb.sum()), "obj_exact": bool(np.array_equal(res["obj"][ok], obj[ok])),
             "sum_exact": bool(np.array_equal(res["sum"][ok], tot[ok])), "best": int(res["best"]),
             "best_x_exact": bool(np.array_equal(res["best_x"], X[:, res["best"]])) if ok[res["best"]] else None}
    out = {"workload": f"C5: MaxCut, power-law graph n={n}, {E} edges, nnz of the full pattern {nnzF}, rank {r}, seed {args.seed}, "
                       f"R after {args.iters} sdplrp_iterate steps",
           "card": card(), "timing_cuda_events": timing, "passes_per_batch_of_64": passes,
           "host_numpy_scipy_K8_s": host_s, "host_threads": threads, "exact_check": check,
           "note": "share_of_bound = (larger of flops / data-sheet peak and bytes / 7.7 TB/s) / kernel time; "
                   "per-call times include the hyperplane upload, the D2H of the results and the 80 MB best_x download"}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if check["obj_exact"] and check["sum_exact"] else 1


if __name__ == "__main__":
    sys.exit(main())
