"""Sweep rounding on several GPUs: run under torchrun with N ranks (one GPU each).  Every rank holds the same R and calls
sdplrp_round_sweep with the same K, hyperplanes, weights and window (SPMD); every rank's thresh, obj, sum, wS, best, best_x,
best_order and best_profile must equal the NumPy restatement on the full R exactly (unit-weight MaxCut and integer degree
weights: every value is exact)."""
import math
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import sdplrplus.jl_b200 as sp
from sdplrplus.jl_b200 import dist as spdist
import torch
from test_gpu_sweep import numpy_sweep, projections

rank, world, local = spdist.init_process_group()
torch.cuda.set_device(local)
P_ = sp.problems
cases = {"powerlaw": P_.powerlaw_graph(20000, 160000, 5), "g1shape": P_.gnm_graph(800, 19176, 1)}
fail = 0
for name, A in cases.items():
    C, As, bs = P_.maxcut(A)
    n, r, K = A.shape[0], 8, 20
    deg = np.asarray(A.sum(axis=1)).reshape(-1)
    vol = float(deg.sum())
    rng = np.random.default_rng(0)
    R = 2.0 * rng.random((n, r)) - 1.0
    G = rng.standard_normal((K, r))
    P = projections(R, G)
    windows = {"none": (None, (-math.inf, math.inf)), "bisection": (None, (n // 2, (n + 1) // 2)),
               "mu0.1": (deg, (0.1 * vol, 0.9 * vol))}
    refs = {key: numpy_sweep(C, P, w, win) for key, (w, win) in windows.items()}
    for relabel in (1, 0):
        h = spdist.make_handle(sp.Handle)
        h.set_option("relabel", relabel)
        eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=h)
        eng.init_vars(r, R, np.zeros(n), 2.0, 4)
        for key, (w, win) in windows.items():
            res = eng.round_sweep(K, G, w=w, window=win)
            ref = refs[key]
            thresh = np.array([c["t"] for c in ref])
            obj = np.array([c["obj"] for c in ref])
            b = int(np.argmin(obj))
            ok = (np.array_equal(res["thresh"], thresh) and np.array_equal(res["obj"], obj)
                  and np.array_equal(res["sum"], n - 2.0 * thresh)
                  and np.array_equal(res["wS"], [c["W"][c["t"]] for c in ref]) and res["best"] == b
                  and np.array_equal(res["best_x"], ref[b]["x"]) and np.array_equal(res["best_order"], ref[b]["order"])
                  and np.array_equal(res["best_profile"], ref[b]["profile"]))
            if not ok:
                fail += 1
                print(f"  MISMATCH rank {rank} {name} relabel={relabel} window={key}: thresh {res['thresh'][:4]} vs {thresh[:4]}, "
                      f"best {res['best']} vs {b}", flush=True)
        if rank == 0:
            print(f"{name:10s} relabel={relabel} world={world} rows={h.row_range()} ok so far (fail={fail})", flush=True)
        h.close()
fail = int(spdist.max_over_ranks(float(fail)))
spdist.barrier()
if rank == 0:
    print("MULTIGPU SWEEP", "FAILED" if fail else "OK", flush=True)
sys.exit(1 if fail else 0)
