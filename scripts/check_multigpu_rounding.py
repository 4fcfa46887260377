"""Hyperplane rounding, one-flip local search and sweep rounding on several GPUs: run under torchrun with N ranks (one GPU
each).  Every rank holds the same R and calls each entry point with the same K, hyperplanes, max_rounds, weights and window
(SPMD); every rank's outputs must equal the NumPy restatements on the full R exactly (unit-weight MaxCut and integer degree
weights: every objective, gain and weight is exact).  Prints one OK / FAILED marker per method."""
import math
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import scipy.sparse as sps
import sdplrplus.jl_b200 as sp
from sdplrplus.jl_b200 import dist as spdist
import torch
from rounding_reference import numpy_local_search, numpy_sweep, projections

rank, world, local = spdist.init_process_group()
torch.cuda.set_device(local)
P_ = sp.problems
cases = {"powerlaw": P_.powerlaw_graph(20000, 160000, 5), "g1shape": P_.gnm_graph(800, 19176, 1)}
fail = {"ROUNDING": 0, "LOCAL SEARCH": 0, "SWEEP": 0}


def mismatch(method, msg):
    fail[method] += 1
    print(f"  MISMATCH rank {rank} {method.lower()} {msg}", flush=True)


def hyperplane(eng, C, R, G, K, name, relabel):
    Cs = sps.csr_matrix(C)
    for G_arg, seed in ((G, 0), (None, 3)):
        res = eng.round_hyperplane(K, G_arg, seed)
        X = np.where(R @ res["G_used"].T >= 0, 1.0, -1.0)   # seeded: the reference from the hyperplanes reported
        obj = np.einsum("ik,ik->k", X, Cs @ X)
        b = int(np.argmin(obj))
        ok = (np.array_equal(res["G_used"], G if G_arg is not None else res["G_used"]) and np.array_equal(res["obj"], obj)
              and np.array_equal(res["sum"], X.sum(axis=0)) and res["best"] == b and np.array_equal(res["best_x"], X[:, b]))
        if not ok:
            mismatch("ROUNDING", f"{name} relabel={relabel} G={'given' if G_arg is not None else 'seeded'}: max obj err "
                     f"{np.max(np.abs(res['obj'] - obj)):.3e} best {res['best']} vs {b}")


def local_search(eng, C, K, G, X0, obj0, want, name, relabel):
    for mr, (X, obj, tot, flips, rounds) in want.items():
        res = eng.round_local_search(K, G, 0, mr)
        b = int(np.argmin(obj))
        ok = (np.array_equal(res["obj_round"], obj0) and np.array_equal(res["obj"], obj) and np.array_equal(res["sum"], tot)
              and np.array_equal(res["flips"], flips) and np.array_equal(res["rounds"], rounds) and res["best"] == b
              and np.array_equal(res["best_x"], X[:, b]))
        if not ok:
            mismatch("LOCAL SEARCH", f"{name} relabel={relabel} max_rounds={mr}: max obj err "
                     f"{np.max(np.abs(res['obj'] - obj)):.3e} best {res['best']} vs {b}")


def sweep(eng, n, K, G, windows, refs, name, relabel):
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
            mismatch("SWEEP", f"{name} relabel={relabel} window={key}: thresh {res['thresh'][:4]} vs {thresh[:4]}, "
                     f"best {res['best']} vs {b}")


for name, A in cases.items():
    C, As, bs = P_.maxcut(A)
    n, r, K, K_sweep = A.shape[0], 8, 100, 20
    rng = np.random.default_rng(0)
    R = 2.0 * rng.random((n, r)) - 1.0
    G = rng.standard_normal((K, r))
    X0 = np.where(R @ G.T >= 0, 1.0, -1.0)
    obj0 = np.einsum("ik,ik->k", X0, sps.csr_matrix(C) @ X0)
    want = {mr: numpy_local_search(C, X0, mr) for mr in (1000, 2)}
    deg = np.asarray(A.sum(axis=1)).reshape(-1)
    vol = float(deg.sum())
    G_sweep = G[:K_sweep]
    P = projections(R, G_sweep)
    windows = {"none": (None, (-math.inf, math.inf)), "bisection": (None, (n // 2, (n + 1) // 2)),
               "mu0.1": (deg, (0.1 * vol, 0.9 * vol))}
    refs = {key: numpy_sweep(C, P, w, win) for key, (w, win) in windows.items()}
    for relabel in (1, 0):
        h = spdist.make_handle(sp.Handle)
        h.set_option("relabel", relabel)
        eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=h)
        eng.init_vars(r, R, np.zeros(n), 2.0, 4)
        hyperplane(eng, C, R, G, K, name, relabel)
        local_search(eng, C, K, G, X0, obj0, want, name, relabel)
        sweep(eng, n, K_sweep, G_sweep, windows, refs, name, relabel)
        if rank == 0:
            print(f"{name:10s} relabel={relabel} world={world} rows={h.row_range()} ok so far (fail={fail})", flush=True)
        h.close()
failed = {m: int(spdist.max_over_ranks(float(f))) for m, f in fail.items()}
spdist.barrier()
if rank == 0:
    for m, f in failed.items():
        print(f"MULTIGPU {m}", "FAILED" if f else "OK", flush=True)
sys.exit(1 if any(failed.values()) else 0)
