"""One-flip local search after hyperplane rounding on several GPUs: run under torchrun with N ranks (one GPU each).  Every
rank holds the same R and calls sdplrp_round_local_search with the same K, hyperplanes and max_rounds (SPMD); every rank's
obj_round, obj, sum, flips, rounds, best and best_x must equal the NumPy restatement of the algorithm exactly (unit-weight
MaxCut: every gain is a multiple of 1/2)."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
import scipy.sparse as sps
import sdplrplus.jl_b200 as sp
from sdplrplus.jl_b200 import dist as spdist
from test_gpu_local_search import numpy_local_search
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
    X0 = np.where(R @ G.T >= 0, 1.0, -1.0)
    obj0 = np.einsum("ik,ik->k", X0, sps.csr_matrix(C) @ X0)
    want = {mr: numpy_local_search(C, X0, mr) for mr in (1000, 2)}
    for relabel in (1, 0):
        h = spdist.make_handle(sp.Handle)
        h.set_option("relabel", relabel)
        eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=h)
        eng.init_vars(r, R, np.zeros(n), 2.0, 4)
        for mr, (X, obj, tot, flips, rounds) in want.items():
            res = eng.round_local_search(K, G, 0, mr)
            b = int(np.argmin(obj))
            ok = (np.array_equal(res["obj_round"], obj0) and np.array_equal(res["obj"], obj) and np.array_equal(res["sum"], tot)
                  and np.array_equal(res["flips"], flips) and np.array_equal(res["rounds"], rounds) and res["best"] == b
                  and np.array_equal(res["best_x"], X[:, b]))
            if not ok:
                fail += 1
                print(f"  MISMATCH rank {rank} {name} relabel={relabel} max_rounds={mr}: max obj err "
                      f"{np.max(np.abs(res['obj'] - obj)):.3e} best {res['best']} vs {b}", flush=True)
        if rank == 0:
            print(f"{name:10s} relabel={relabel} world={world} rows={h.row_range()} ok so far (fail={fail})", flush=True)
        h.close()
fail = int(spdist.max_over_ranks(float(fail)))
spdist.barrier()
if rank == 0:
    print("MULTIGPU LOCAL SEARCH", "FAILED" if fail else "OK", flush=True)
sys.exit(1 if fail else 0)
