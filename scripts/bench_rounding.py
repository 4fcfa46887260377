#!/usr/bin/env python
"""Rounding on C5 (MaxCut, 10M-vertex power-law graph, rank 10: the graph and seed of bench.py), with R after a few
sdplrp_iterate steps.  --method picks the entry point; each prints one JSON line (the keys of profiles/rounding_c5.json,
local_search_c5.json and sweep_c5.json respectively) with the card name and power limit read in the same run:
  hyperplane    CUDA-event time on the handle's stream of sdplrp_round_hyperplane for K = 64 and K = 1024 (ms per call,
                per 64 candidates); the sign / evaluation pass kernel times, algorithmic bytes and flops, achieved rates
                and share of the bound; the NumPy / SciPy host time for K = 8 and an exact check of those 8 candidates.
  local_search  CUDA-event time of sdplrp_round_local_search for K = 64 next to sdplrp_round_hyperplane; rounds, flips per
                round and the best objective after every round (max_rounds-truncated calls); the kernel times per round;
                an exact check of one candidate (K = 1) against the NumPy restatement of the algorithm (--no-check skips it).
  sweep         CUDA-event time of sdplrp_round_sweep for K = 16 and K = 64, with and without the best candidate's outputs
                (best_x, profile, order); the kernel time of each pass per batch of 16 candidates: projection, sort (key
                gather + CUB radix sort), delta, scan (tile sums, tile offsets, rescan, selection), words + evaluation; one
                candidate checked exactly against the NumPy restatement.
Kernel times come from a separate torch.profiler run (the profiler slows the host); the profiler's kernel names and the
pass each one is counted in go to stderr.  Writes nothing into the tree (--out FILE copies the JSON line to FILE)."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_GBS = 7700.0       # HGX B200 data sheet, one GPU
FP64_TFLOPS = 37.0     # HGX B200 data sheet, one GPU, FP64

# per method: (profile key, name fragments of the kernel); a kernel goes to the first entry whose fragments it all contains,
# or to "other".  The want and delta passes are the LsWant / SwDelta instantiations of the neighbour-sum kernels.
KERNELS = {
    "hyperplane": [("sign", ("k_round_sign",)), ("eval", ("k_round_eval(",))],
    "local_search": [("k_ls_want_seg", ("k_nbr_seg<", "LsWant")), ("k_ls_want_combine", ("k_nbr_combine<", "LsWant")),
                     ("k_ls_want", ("k_nbr_short<", "LsWant")), ("k_ls_flip_seg", ("k_ls_flip_seg(",)),
                     ("k_ls_flip", ("k_ls_flip(",)), ("k_ls_apply_seg", ("k_ls_apply_seg(",)), ("k_ls_apply", ("k_ls_apply(",)),
                     ("k_ls_count", ("k_ls_count(",)), ("k_round_sign", ("k_round_sign",)), ("k_round_eval", ("k_round_eval(",))],
    "sweep": [("projection", ("k_round_sign",)), ("sort", ("k_sw_keys",)), ("sort", ("DeviceRadixSort",)), ("delta", ("SwDelta",)),
              ("scan", ("k_sw_tile",)), ("scan", ("k_sw_scan",)), ("scan", ("k_sw_select",)), ("words_eval", ("k_sw_words",)),
              ("words_eval", ("k_round_eval(",))],
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:
        return {"error": str(e)}


class Bench:
    """C5 with R after `iters` sdplrp_iterate steps, and the timing / profiling helpers every method uses"""

    def __init__(self, args):
        import torch
        import sdplrplus.jl_b200 as sp
        from bench import SimpleData, generate, pinned_uniform
        self.torch, self.args = torch, args
        self.n, self.r = n, r = args.n, args.rank
        self.handle = sp.Handle(device=0)
        self.asm, b, _, self.E, _ = generate(sp, n, args.edges, args.seed, keep_on_device=False)
        self.eng = sp.B200Engine(SimpleData(n, n, b), handle=self.handle, asm=self.asm)
        _, self.nnzF, _ = self.handle.pattern_sizes()
        _, R0 = pinned_uniform((n, r), 0)
        self.eng.init_vars(r, R0, np.zeros(n), 2.0, 4)
        self.eng.fg()
        self.eng.iterate(args.iters)
        self.stream = torch.cuda.ExternalStream(self.handle.stream)

    def workload(self):
        return (f"C5: MaxCut, power-law graph n={self.n}, {self.E} edges, nnz of the full pattern {self.nnzF}, rank {self.r}, "
                f"seed {self.args.seed}, R after {self.args.iters} sdplrp_iterate steps")

    def timed(self, fn):
        """(ms, fn()) with CUDA events on the handle's stream"""
        ev0, ev1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        ev0.record(self.stream)
        out = fn()
        ev1.record(self.stream)
        self.torch.cuda.synchronize()
        return ev0.elapsed_time(ev1), out

    def kernel_times(self, fn, method):
        """{profile key or "other": [device ms, launches]} of the kernels fn launches, by the method's KERNELS table"""
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            self.torch.cuda.synchronize()
        kern = {}
        for evt in prof.key_averages():
            dev_us = getattr(evt, "device_time_total", None)
            if dev_us is None:
                dev_us = getattr(evt, "cuda_time_total", 0.0)
            if dev_us <= 0:
                continue
            key = next((k for k, frags in KERNELS[method] if all(f in evt.key for f in frags)), "other")
            print(f"kernel {key:18s} {dev_us / 1e3:10.3f} ms {evt.count:5d}x  {evt.key}", file=sys.stderr, flush=True)
            k = kern.setdefault(key, [0.0, 0])
            k[0] += dev_us / 1e3
            k[1] += evt.count
        return kern

    def host_C(self):
        asm, n = self.asm, self.n
        import scipy.sparse as sps
        c0, c1 = int(asm.mat_off[n]), int(asm.mat_off[n + 1])
        return sps.csr_matrix((asm.V[c0:c1], (asm.I[c0:c1] - 1, asm.J[c0:c1] - 1)), shape=(n, n))


def hyperplane(bn):
    eng, n, r, args = bn.eng, bn.n, bn.r, bn.args
    eng.round_hyperplane(64, seed=1)      # warm-up: first launches, first-use buffers
    eng.round_hyperplane(1024, seed=1)
    timing = {}
    for K in (64, 1024):
        ms = [bn.timed(lambda: eng.round_hyperplane(K, seed=100 + rep))[0] for rep in range(args.reps)]
        timing[K] = {"ms_per_call_median": float(np.median(ms)), "ms_per_call_all": ms,
                     "ms_per_64_candidates": float(np.median(ms)) / (K / 64)}

    kern = bn.kernel_times(lambda: eng.round_hyperplane(1024, seed=7), "hyperplane")
    sign, ev, other = kern.get("sign", [0.0, 0]), kern.get("eval", [0.0, 0]), kern.get("other", [0.0, 0])
    sign_ms, eval_ms = sign[0] / max(1, sign[1]), ev[0] / max(1, ev[1])
    # algorithmic work of one batch of 64 candidates
    sign_bytes = 8.0 * r * n + 8.0 * n                                    # R read once, one word written per vertex
    sign_flops = 2.0 * 64 * r * n
    eval_bytes = 12.0 * bn.nnzF + 4.0 * (n + 1) + 8.0 * bn.nnzF + 8.0 * n   # index + value per entry, row pointers, one word per entry and per row
    eval_updates = 64.0 * bn.nnzF                                           # candidate accumulations (predicated FP64 adds)
    passes = {
        "sign": {"ms_per_batch": sign_ms, "launches": sign[1], "bytes": sign_bytes, "flops": sign_flops,
                 "GBs": sign_bytes / (sign_ms * 1e-3) / 1e9, "GFLOPs": sign_flops / (sign_ms * 1e-3) / 1e9,
                 "bound": "FP64 FMA (data sheet 37 TFLOP/s)" if sign_flops / FP64_TFLOPS / 1e12 > sign_bytes / HBM_GBS / 1e9 else "HBM",
                 "share_of_bound": max(sign_flops / (FP64_TFLOPS * 1e12), sign_bytes / (HBM_GBS * 1e9)) / (sign_ms * 1e-3)},
        "eval": {"ms_per_batch": eval_ms, "launches": ev[1], "bytes": eval_bytes, "candidate_adds": eval_updates,
                 "GBs": eval_bytes / (eval_ms * 1e-3) / 1e9, "Gadds": eval_updates / (eval_ms * 1e-3) / 1e9,
                 "bound": "FP64 add issue (data sheet 37 TFLOP/s = 18.5e12 FP64 instructions/s)"
                          if eval_updates / 18.5e12 > eval_bytes / HBM_GBS / 1e9 else "HBM",
                 "share_of_bound": max(eval_updates / 18.5e12, eval_bytes / (HBM_GBS * 1e9)) / (eval_ms * 1e-3)},
        "other_kernels_ms_per_call": other[0],
        "batches_profiled": 1024 // 64,
    }

    # host reference for K = 8 on the downloaded R, and an exact cross-check of those candidates
    R = eng.get_R()
    res = eng.round_hyperplane(8, seed=3)
    G = res["G_used"]
    C = bn.host_C()
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
    out = {"workload": bn.workload(), "card": card(), "timing_cuda_events": timing, "passes_per_batch_of_64": passes,
           "host_numpy_scipy_K8_s": host_s, "host_threads": threads, "exact_check": check,
           "note": "share_of_bound = (larger of flops / data-sheet peak and bytes / 7.7 TB/s) / kernel time; "
                   "per-call times include the hyperplane upload, the D2H of the results and the 80 MB best_x download"}
    return out, check["obj_exact"] and check["sum_exact"]


def local_search(bn):
    eng, args, K = bn.eng, bn.args, 64
    eng.round_local_search(K, seed=1)   # warm-up: first launches, first-use buffers
    eng.round_hyperplane(K, seed=1)
    ls_ms, hp_ms, res = [], [], None
    for rep in range(args.reps):
        ms, res = bn.timed(lambda: eng.round_local_search(K, seed=100))
        ls_ms.append(ms)
        hp_ms.append(bn.timed(lambda: eng.round_hyperplane(K, seed=100))[0])
    rounds = int(res["rounds"].max())

    # per-round trajectory of the timed batch: flips and the objective after t rounds (truncated calls)
    flips_after, best_after = [0], [float(res["obj_round"].min())]
    for t in range(1, rounds + 1):
        rt = eng.round_local_search(K, seed=100, max_rounds=t)
        flips_after.append(int(rt["flips"].sum()))
        best_after.append(float(rt["obj"].min()))
    flips_per_round = list(np.diff(flips_after).astype(int).tolist())

    kern = bn.kernel_times(lambda: eng.round_local_search(K, seed=100), "local_search")
    kernels = {k: {"ms_total": v[0], "launches": v[1], "ms_per_launch": v[0] / max(1, v[1])} for k, v in kern.items() if k != "other"}
    per_round = {p: sum(kernels.get(k, {}).get("ms_total", 0.0) for k in kernels if k.startswith("k_ls_" + p)) / max(1, rounds)
                 for p in ("want", "flip", "apply")}

    check = None
    if not args.no_check:
        from rounding_reference import numpy_local_search
        R = eng.get_R()
        r1 = eng.round_local_search(1, seed=100)
        X0 = np.where(R @ r1["G_used"].T >= 0, 1.0, -1.0)
        C = bn.host_C()
        t0 = time.perf_counter()
        X, obj, tot, flips, rnds = numpy_local_search(C, X0, 1000)
        host_s = time.perf_counter() - t0
        check = {"host_numpy_scipy_K1_s": host_s, "obj": float(obj[0]), "obj_exact": bool(r1["obj"][0] == obj[0]),
                 "sum_exact": bool(r1["sum"][0] == tot[0]), "flips_exact": bool(r1["flips"][0] == flips[0]),
                 "rounds_exact": bool(r1["rounds"][0] == rnds[0]), "x_exact": bool(np.array_equal(r1["best_x"], X[:, 0])),
                 "same_as_candidate_0_of_K64": bool(r1["obj"][0] == res["obj"][0])}
    out = {"workload": bn.workload() + f", K = {K}", "card": card(),
           "timing_cuda_events": {"round_local_search_ms_median": float(np.median(ls_ms)), "round_local_search_ms_all": ls_ms,
                                  "round_hyperplane_ms_median": float(np.median(hp_ms)), "round_hyperplane_ms_all": hp_ms},
           "rounds": rounds, "rounds_per_candidate_min_max": [int(res["rounds"].min()), int(res["rounds"].max())],
           "flips_per_round_all_candidates": flips_per_round, "best_obj_after_round": best_after,
           "best_obj_rounded": float(res["obj_round"].min()), "best_obj_refined": float(res["obj"].min()),
           "kernels_profiled": kernels, "kernel_ms_per_round": per_round, "exact_check_K1": check,
           "note": "per-call times include the hyperplane upload, one count download per round and the 80 MB best_x download"}
    ok = check is None or all(v for k, v in check.items() if k.endswith("exact"))
    return out, ok and out["best_obj_refined"] < out["best_obj_rounded"]


def sweep(bn):
    from rounding_reference import exact_projection, numpy_sweep
    eng, handle, args, torch = bn.eng, bn.handle, bn.args, bn.torch
    mem0 = torch.cuda.mem_get_info()[0]
    eng.round_sweep(16, seed=1)                 # warm-up: first launches, first-use buffers, CUB scratch
    mem1 = torch.cuda.mem_get_info()[0]

    def timed(K, full):
        # obj / best only: no recomputation of the best candidate, no n-sized downloads
        ms = [bn.timed(lambda: eng.round_sweep(K, seed=100 + rep) if full else _sweep_min(handle, K, 100 + rep))[0]
              for rep in range(args.reps)]
        return {"ms_per_call_median": float(np.median(ms)), "ms_per_call_all": ms, "ms_per_16_candidates": float(np.median(ms)) / (K / 16)}

    timing = {f"K{K}_{'full' if full else 'obj_only'}": timed(K, full) for K in (16, 64) for full in (False, True)}
    hp_ms = [bn.timed(lambda: eng.round_hyperplane(64, seed=100 + rep))[0] for rep in range(args.reps)]
    timing["round_hyperplane_K64"] = {"ms_per_call_median": float(np.median(hp_ms)), "ms_per_call_all": hp_ms}

    # obj / best only, so every launch belongs to a batch
    kern = bn.kernel_times(lambda: _sweep_min(handle, 64, 7), "sweep")
    batches = 64 // 16
    per_batch = {p: kern.get(p, [0.0])[0] / batches for p in {k for k, _ in KERNELS["sweep"]} | {"other"}}

    # one candidate exactly against the host restatement
    R = eng.get_R()
    res = eng.round_sweep(1, seed=3)
    G = res["G_used"]
    C = bn.host_C()
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
    out = {"workload": bn.workload(), "card": card(), "timing_cuda_events": timing, "kernel_ms_per_batch_of_16": per_batch,
           "sweep_buffers_GB": (mem0 - mem1) / 1e9, "host_numpy_scipy_K1_s": host_s, "exact_check": check, "quality": quality,
           "note": "obj_only calls pass only obj and best (no recomputation of the best candidate, no n-sized downloads); "
                   "full calls also return best_x, best_profile and best_order"}
    return out, all(check[k] for k in ("thresh_exact", "obj_exact", "best_x_exact", "order_exact", "profile_exact"))


def _sweep_min(handle, K, seed):
    """sdplrp_round_sweep with only the obj / best outputs"""
    import ctypes as C
    obj, best = np.empty(K), C.c_int64()
    handle._check(handle.lib.sdplrp_round_sweep(handle._h, K, None, seed, None, -math.inf, math.inf, None,
                                                obj.ctypes.data_as(C.POINTER(C.c_double)), None, None, None, C.byref(best),
                                                None, None, None))
    return obj, best.value - 1


METHODS = {"hyperplane": hyperplane, "local_search": local_search, "sweep": sweep}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--method", choices=list(METHODS), default="hyperplane")
    ap.add_argument("--vertices", dest="n", type=int, default=10_000_000)
    ap.add_argument("--edges", type=int, default=80_000_000)
    ap.add_argument("--rank", type=int, default=10)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--iters", type=int, default=5, help="sdplrp_iterate steps before rounding")
    ap.add_argument("--reps", type=int, help="timed calls per configuration (default: 5 for hyperplane, else 3)")
    ap.add_argument("--no-check", action="store_true", help="local_search: skip the host reference run")
    ap.add_argument("--out")
    args = ap.parse_args()
    if args.reps is None:
        args.reps = 5 if args.method == "hyperplane" else 3
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}), flush=True)
        return 2
    out, ok = METHODS[args.method](Bench(args))
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
