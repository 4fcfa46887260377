#!/usr/bin/env python
"""One-flip local search after hyperplane rounding on C5 (MaxCut, 10M-vertex power-law graph, rank 10: the graph and seed
of bench.py), with R after a few sdplrp_iterate steps.  Prints one JSON line:
  - the card name and power limit, read in the same run;
  - CUDA-event time on the handle's stream of sdplrp_round_local_search for K = 64 (ms per call), next to
    sdplrp_round_hyperplane for the same K;
  - rounds, flips per round and the best objective after every round of the timed batch, from max_rounds-truncated calls;
  - the want / flip / apply kernel times from a separate torch.profiler run;
  - the best objective before and after the descent;
  - an exact check of one candidate (K = 1) against a NumPy / SciPy run of the same algorithm on the downloaded R.
Writes nothing into the tree (--out FILE copies the JSON line to FILE)."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vertices", dest="n", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=80_000_000)
    ap.add_argument("--rank", type=int, default=10)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--iters", type=int, default=5, help="sdplrp_iterate steps before rounding")
    ap.add_argument("--reps", type=int, default=3, help="timed calls")
    ap.add_argument("--no-check", action="store_true", help="skip the host reference run")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import scipy.sparse as sps
    import sdplrplus.jl_b200 as sp
    from bench import SimpleData, generate, pinned_uniform
    from bench_rounding import card
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}), flush=True)
        return 2
    n, r, K = args.n, args.rank, 64
    handle = sp.Handle(device=0)
    asm, b, _, E, _ = generate(sp, n, args.edges, args.seed, keep_on_device=False)
    eng = sp.B200Engine(SimpleData(n, n, b), handle=handle, asm=asm)
    _, nnzF, _ = handle.pattern_sizes()
    _, R0 = pinned_uniform((n, r), 0)
    eng.init_vars(r, R0, np.zeros(n), 2.0, 4)
    eng.fg()
    eng.iterate(args.iters)
    stream = torch.cuda.ExternalStream(handle.stream)

    def timed(fn):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        out = fn()
        ev1.record(stream)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1), out

    eng.round_local_search(K, seed=1)   # warm-up: first launches, first-use buffers
    eng.round_hyperplane(K, seed=1)
    ls_ms, hp_ms, res = [], [], None
    for rep in range(args.reps):
        ms, res = timed(lambda: eng.round_local_search(K, seed=100))
        ls_ms.append(ms)
        hp_ms.append(timed(lambda: eng.round_hyperplane(K, seed=100))[0])
    rounds = int(res["rounds"].max())

    # per-round trajectory of the timed batch: flips and the objective after t rounds (truncated calls)
    flips_after, best_after = [0], [float(res["obj_round"].min())]
    for t in range(1, rounds + 1):
        rt = eng.round_local_search(K, seed=100, max_rounds=t)
        flips_after.append(int(rt["flips"].sum()))
        best_after.append(float(rt["obj"].min()))
    flips_per_round = list(np.diff(flips_after).astype(int).tolist())

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.round_local_search(K, seed=100)
        torch.cuda.synchronize()
    kern = {}
    for evt in prof.key_averages():
        dev_us = getattr(evt, "device_time_total", None)
        if dev_us is None:
            dev_us = getattr(evt, "cuda_time_total", 0.0)
        for name in ("k_ls_want_seg", "k_ls_want_combine", "k_ls_want", "k_ls_flip_seg", "k_ls_flip", "k_ls_apply_seg", "k_ls_apply",
                     "k_ls_count", "k_round_sign", "k_round_eval"):
            if name + "(" in evt.key or evt.key.endswith(name) or (name in evt.key and name + "_" not in evt.key):
                k = kern.setdefault(name, [0.0, 0])
                k[0] += dev_us / 1e3
                k[1] += evt.count
                break
    kernels = {k: {"ms_total": v[0], "launches": v[1], "ms_per_launch": v[0] / max(1, v[1])} for k, v in kern.items()}
    per_round = {p: sum(kernels.get(k, {}).get("ms_total", 0.0) for k in kernels if k.startswith("k_ls_" + p)) / max(1, rounds)
                 for p in ("want", "flip", "apply")}

    check = None
    if not args.no_check:
        from test_gpu_local_search import numpy_local_search
        R = eng.get_R()
        r1 = eng.round_local_search(1, seed=100)
        X0 = np.where(R @ r1["G_used"].T >= 0, 1.0, -1.0)
        c0, c1 = int(asm.mat_off[n]), int(asm.mat_off[n + 1])
        C = sps.csr_matrix((asm.V[c0:c1], (asm.I[c0:c1] - 1, asm.J[c0:c1] - 1)), shape=(n, n))
        t0 = time.perf_counter()
        X, obj, tot, flips, rnds = numpy_local_search(C, X0, 1000)
        host_s = time.perf_counter() - t0
        check = {"host_numpy_scipy_K1_s": host_s, "obj": float(obj[0]), "obj_exact": bool(r1["obj"][0] == obj[0]),
                 "sum_exact": bool(r1["sum"][0] == tot[0]), "flips_exact": bool(r1["flips"][0] == flips[0]),
                 "rounds_exact": bool(r1["rounds"][0] == rnds[0]), "x_exact": bool(np.array_equal(r1["best_x"], X[:, 0])),
                 "same_as_candidate_0_of_K64": bool(r1["obj"][0] == res["obj"][0])}
    out = {"workload": f"C5: MaxCut, power-law graph n={n}, {E} edges, nnz of the full pattern {nnzF}, rank {r}, seed {args.seed}, "
                       f"R after {args.iters} sdplrp_iterate steps, K = {K}",
           "card": card(),
           "timing_cuda_events": {"round_local_search_ms_median": float(np.median(ls_ms)), "round_local_search_ms_all": ls_ms,
                                  "round_hyperplane_ms_median": float(np.median(hp_ms)), "round_hyperplane_ms_all": hp_ms},
           "rounds": rounds, "rounds_per_candidate_min_max": [int(res["rounds"].min()), int(res["rounds"].max())],
           "flips_per_round_all_candidates": flips_per_round, "best_obj_after_round": best_after,
           "best_obj_rounded": float(res["obj_round"].min()), "best_obj_refined": float(res["obj"].min()),
           "kernels_profiled": kernels, "kernel_ms_per_round": per_round, "exact_check_K1": check,
           "note": "per-call times include the hyperplane upload, one count download per round and the 80 MB best_x download"}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ok = check is None or all(v for k, v in check.items() if k.endswith("exact"))
    return 0 if ok and out["best_obj_refined"] < out["best_obj_rounded"] else 1


if __name__ == "__main__":
    sys.exit(main())
