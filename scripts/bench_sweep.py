#!/usr/bin/env python
"""Sweep rounding on C5 (MaxCut, 10M-vertex power-law graph, rank 10: the graph and seed of bench.py), with R after a few
sdplrp_iterate steps.  Prints one JSON line:
  - CUDA-event time on the handle's stream of sdplrp_round_sweep for K = 16 and K = 64 (median ms per call), with and
    without the best candidate's outputs (best_x, profile, order);
  - the kernel time of each pass per batch of 16 candidates from a separate torch.profiler run: projection, sort (key
    gather + CUB radix sort), delta, scan (tile sums, tile offsets, rescan, selection), words + evaluation;
  - the card name and power limit, read in the same run;
  - one candidate checked exactly against the NumPy / SciPy restatement on the downloaded R.
Writes nothing into the tree (--out FILE copies the JSON line to FILE, e.g. profiles/sweep_c5.json)."""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

PASSES = {   # kernel name fragment -> pass
    "k_round_sign": "projection", "k_sw_keys": "sort", "DeviceRadixSort": "sort", "k_sw_delta": "delta",
    "k_sw_tile": "scan", "k_sw_scan": "scan", "k_sw_select": "scan", "k_sw_words": "words_eval", "k_round_eval": "words_eval",
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vertices", dest="n", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=80_000_000)
    ap.add_argument("--rank", type=int, default=10)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--iters", type=int, default=5, help="sdplrp_iterate steps before rounding")
    ap.add_argument("--reps", type=int, default=3, help="timed calls per K")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import scipy.sparse as sps
    import sdplrplus.jl_b200 as sp
    from bench import SimpleData, generate, pinned_uniform
    from bench_rounding import card
    from test_gpu_sweep import numpy_sweep
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
    mem0 = torch.cuda.mem_get_info()[0]
    eng.round_sweep(16, seed=1)                 # warm-up: first launches, first-use buffers, CUB scratch
    mem1 = torch.cuda.mem_get_info()[0]

    def timed(K, full):
        ms = []
        for rep in range(args.reps):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            if full:
                eng.round_sweep(K, seed=100 + rep)
            else:   # obj / best only: no recomputation of the best candidate, no n-sized downloads
                _sweep_min(handle, K, 100 + rep)
            ev1.record(stream)
            torch.cuda.synchronize()
            ms.append(ev0.elapsed_time(ev1))
        return {"ms_per_call_median": float(np.median(ms)), "ms_per_call_all": ms, "ms_per_16_candidates": float(np.median(ms)) / (K / 16)}

    timing = {f"K{K}_{'full' if full else 'obj_only'}": timed(K, full) for K in (16, 64) for full in (False, True)}
    hp_ms = []
    for rep in range(args.reps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        eng.round_hyperplane(64, seed=100 + rep)
        ev1.record(stream)
        torch.cuda.synchronize()
        hp_ms.append(ev0.elapsed_time(ev1))
    timing["round_hyperplane_K64"] = {"ms_per_call_median": float(np.median(hp_ms)), "ms_per_call_all": hp_ms}

    # kernel split (separate run: the profiler slows the host); obj / best only, so every launch belongs to a batch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _sweep_min(handle, 64, 7)
        torch.cuda.synchronize()
    kern = {p: 0.0 for p in set(PASSES.values()) | {"other"}}
    for evt in prof.key_averages():
        dev_us = getattr(evt, "device_time_total", None)
        if dev_us is None:
            dev_us = getattr(evt, "cuda_time_total", 0.0)
        key = next((p for frag, p in PASSES.items() if frag in evt.key), "other")
        kern[key] += dev_us / 1e3
    batches = 64 // 16
    per_batch = {k: v / batches for k, v in kern.items()}

    # one candidate exactly against the host restatement
    R = eng.get_R()
    res = eng.round_sweep(1, seed=3)
    G = res["G_used"]
    c0, c1 = int(asm.mat_off[n]), int(asm.mat_off[n + 1])
    C = sps.csr_matrix((asm.V[c0:c1], (asm.I[c0:c1] - 1, asm.J[c0:c1] - 1)), shape=(n, n))
    t0 = time.perf_counter()
    p = exact_projection(R, G[0])
    ref = numpy_sweep(C, p[:, None])[0]
    host_s = time.perf_counter() - t0
    check = {"candidates": 1, "min_adjacent_gap": float(np.min(np.diff(np.sort(p)))),
             "thresh": int(res["thresh"][0]), "thresh_exact": bool(res["thresh"][0] == ref["t"]),
             "obj": float(res["obj"][0]), "obj_exact": bool(res["obj"][0] == ref["obj"]),
             "best_x_exact": bool(np.array_equal(res["best_x"], ref["x"])),
             "order_exact": bool(np.array_equal(res["best_order"], ref["order"])),
             "profile_exact": bool(np.array_equal(res["best_profile"], ref["profile"]))}
    hp = eng.round_hyperplane(64, seed=100)
    sw = eng.round_sweep(64, seed=100)
    quality = {"hyperplane_best_obj_K64": float(hp["obj"].min()), "sweep_best_obj_K64": float(sw["obj"].min()),
               "sweep_le_hyperplane_every_k": bool(np.all(sw["obj"] <= hp["obj"]))}
    out = {"workload": f"C5: MaxCut, power-law graph n={n}, {E} edges, nnz of the full pattern {nnzF}, rank {r}, seed {args.seed}, "
                       f"R after {args.iters} sdplrp_iterate steps",
           "card": card(), "timing_cuda_events": timing, "kernel_ms_per_batch_of_16": per_batch,
           "sweep_buffers_GB": (mem0 - mem1) / 1e9, "host_numpy_scipy_K1_s": host_s, "exact_check": check, "quality": quality,
           "note": "obj_only calls pass only obj and best (no recomputation of the best candidate, no n-sized downloads); "
                   "full calls also return best_x, best_profile and best_order"}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if all(check[k] for k in ("thresh_exact", "obj_exact", "best_x_exact", "order_exact", "profile_exact")) else 1


def exact_projection(R, g, margin=1e-10):
    """R g as the device forms it (per row: fma over the columns in order, -0.0 -> +0.0).  BLAS gives it up to rounding;
    the rows whose value lies within `margin` (relative) of a neighbour in sorted order are recomputed with that exact fma
    chain (Fraction arithmetic, correctly rounded), so the order of the host restatement is the device's."""
    from fractions import Fraction
    p = R @ g
    scale = np.linalg.norm(R, axis=1) * np.linalg.norm(g)
    o = np.argsort(p, kind="stable")
    close = np.abs(np.diff(p[o])) <= margin * np.maximum(scale[o][1:], scale[o][:-1])
    rows = np.unique(np.concatenate([o[:-1][close], o[1:][close]]))
    for i in rows:
        acc = Fraction(0)
        for c in range(R.shape[1]):
            acc = Fraction(float(Fraction(float(R[i, c])) * Fraction(float(g[c])) + acc))
        p[i] = float(acc) + 0.0
    return p


def _sweep_min(handle, K, seed):
    """sdplrp_round_sweep with only the obj / best outputs"""
    import ctypes as C
    obj, best = np.empty(K), C.c_int64()
    handle._check(handle.lib.sdplrp_round_sweep(handle._h, K, None, seed, None, -math.inf, math.inf, None,
                                                obj.ctypes.data_as(C.POINTER(C.c_double)), None, None, None, C.byref(best),
                                                None, None, None))
    return obj, best.value - 1


if __name__ == "__main__":
    sys.exit(main())
