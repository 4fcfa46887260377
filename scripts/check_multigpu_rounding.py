"""Hyperplane rounding on several GPUs: run under torchrun with N ranks (one GPU each).  Every rank holds the same R and
calls sdplrp_round_hyperplane with the same K and hyperplanes (SPMD); every rank's obj, sum, best and best_x must equal the
NumPy result on the full R exactly (unit-weight MaxCut: every objective is a multiple of 1/4)."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.sparse as sps
import sdplrplus.jl_b200 as sp
from sdplrplus.jl_b200 import dist as spdist
import torch

rank, world, local = spdist.init_process_group()
torch.cuda.set_device(local)
P = sp.problems
cases = {"powerlaw": P.powerlaw_graph(20000, 160000, 5), "g1shape": P.gnm_graph(800, 19176, 1)}
fail = 0
for name, A in cases.items():
    C, As, bs = P.maxcut(A)
    n, r, K = A.shape[0], 8, 100
    rng = np.random.default_rng(0)
    R = 2.0 * rng.random((n, r)) - 1.0
    G = rng.standard_normal((K, r))
    D = R @ G.T
    X = np.where(D >= 0, 1.0, -1.0)
    obj = np.einsum("ik,ik->k", X, sps.csr_matrix(C) @ X)
    tot = X.sum(axis=0)
    for relabel in (1, 0):
        h = spdist.make_handle(sp.Handle)
        h.set_option("relabel", relabel)
        eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=h)
        eng.init_vars(r, R, np.zeros(n), 2.0, 4)
        for G_arg, seed in ((G, 0), (None, 3)):
            res = eng.round_hyperplane(K, G_arg, seed)
            if G_arg is None:   # device-generated hyperplanes: recompute the reference from the ones reported
                Xs = np.where(R @ res["G_used"].T >= 0, 1.0, -1.0)
                want_obj, want_sum, want_X = np.einsum("ik,ik->k", Xs, sps.csr_matrix(C) @ Xs), Xs.sum(axis=0), Xs
            else:
                want_obj, want_sum, want_X = obj, tot, X
            b = int(np.argmin(want_obj))
            ok = (np.array_equal(res["obj"], want_obj) and np.array_equal(res["sum"], want_sum) and res["best"] == b
                  and np.array_equal(res["best_x"], want_X[:, b]))
            if not ok:
                fail += 1
                print(f"  MISMATCH rank {rank} {name} relabel={relabel} G={'given' if G_arg is not None else 'seeded'}: "
                      f"max obj err {np.max(np.abs(res['obj'] - want_obj)):.3e} best {res['best']} vs {b}", flush=True)
        if rank == 0:
            print(f"{name:10s} relabel={relabel} world={world} rows={h.row_range()} ok so far (fail={fail})", flush=True)
        h.close()
fail = int(spdist.max_over_ranks(float(fail)))
spdist.barrier()
if rank == 0:
    print("MULTIGPU ROUNDING", "FAILED" if fail else "OK", flush=True)
sys.exit(1 if fail else 0)
