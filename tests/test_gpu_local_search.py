"""One-flip local search after hyperplane rounding on the GPU (sdplrp_round_local_search, csrc/rounding.cu) against a NumPy
restatement of the same algorithm: start vectors, every round's priorities and flips, the objectives, sums, flip and round
counts, the best candidate and its vector (exact where the gains are exactly representable), and the one-flip local
optimality of the results for real weights."""
import itertools

import numpy as np
import pytest
import scipy.sparse as sps

from helpers import COMBOS, families, g1_graph, make_case

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1


def mix64(x):
    """splitmix64 finalizer on a uint64 array (wrap-around arithmetic)"""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def priorities(n, t):
    """key(i, t) = mix64(i ^ mix64(0xD1B54A32D192ED03 * (t + 1))) for i = 0..n-1"""
    salt = mix64(np.array([(0xD1B54A32D192ED03 * (t + 1)) & M64], dtype=np.uint64))[0]
    return mix64(np.arange(n, dtype=np.uint64) ^ salt)


def offdiag(C):
    A = sps.csr_matrix(C, dtype=np.float64).copy()
    A.setdiag(0.0)
    A.eliminate_zeros()
    return A


def numpy_local_search(C, X0, max_rounds):
    """Parallel one-flip descent of every column of X0: per round, h = (C - diag C) x, i wants to flip iff x_i h_i > 0, and
    flips iff no neighbour with a higher priority also wants to.  Returns X, obj, sum, flips, rounds (the last round that
    flipped the candidate, 0 if none, -1 if it still wanted to flip after max_rounds rounds)."""
    A = offdiag(C)
    n, K = X0.shape
    coo = A.tocoo()
    rows, cols = coo.row.astype(np.int64), coo.col.astype(np.int64)
    X = X0.copy()
    flips, rounds = np.zeros(K, np.int64), np.zeros(K, np.int64)
    for t in itertools.count():
        W = X * (A @ X) > 0
        cnt = W.sum(axis=0)
        if not cnt.any():
            break
        if t == max_rounds:
            rounds[cnt > 0] = -1
            break
        key = priorities(n, t)
        F = W.copy()
        for k in np.flatnonzero(cnt):
            w = W[:, k]
            sel = w[rows] & w[cols]   # both ends want to flip
            ri, cj = rows[sel], cols[sel]
            beats = (key[cj] > key[ri]) | ((key[cj] == key[ri]) & (cj < ri))   # neighbour j beats i
            F[ri[beats], k] = False
        X[F] *= -1.0
        flips += F.sum(axis=0)
        rounds[cnt > 0] = t + 1
    obj = np.einsum("ik,ik->k", X, sps.csr_matrix(C) @ X)
    return X, obj, X.sum(axis=0), flips, rounds


def start_vectors(R, G):
    return np.where(R @ G.T >= 0, 1.0, -1.0)


def check_against_reference(res, C, X0, max_rounds):
    X, obj, tot, flips, rounds = numpy_local_search(C, X0, max_rounds)
    obj0 = np.einsum("ik,ik->k", X0, sps.csr_matrix(C) @ X0)
    np.testing.assert_array_equal(res["obj_round"], obj0)
    np.testing.assert_array_equal(res["obj"], obj)
    np.testing.assert_array_equal(res["sum"], tot)
    np.testing.assert_array_equal(res["flips"], flips)
    np.testing.assert_array_equal(res["rounds"], rounds)
    b = res["best"]
    assert b == int(np.argmin(obj))
    np.testing.assert_array_equal(res["best_x"], X[:, b])
    return X


def check_local_optimum(res, C, rtol=0.0):
    """obj <= obj_round, obj of best_x, and x_i h_i <= 0 on best_x (every candidate with rounds >= 0 is checked through
    the reference elsewhere; here the returned vector itself)"""
    Cs = sps.csr_matrix(C)
    scale = max(1.0, float(np.max(np.abs(res["obj_round"]))))
    assert np.all(res["obj"] <= res["obj_round"] + rtol * scale)
    x = res["best_x"]
    assert set(np.unique(x)) <= {-1.0, 1.0}
    assert abs(float(x @ (Cs @ x)) - res["obj"][res["best"]]) <= rtol * scale
    if res["rounds"][res["best"]] >= 0:
        h = offdiag(C) @ x
        assert np.all(x * h <= rtol * (abs(offdiag(C)) @ np.ones_like(x) + 1.0))


def engine_with_R(sp, gpu_handle_factory, config, C, As, bs, R):
    eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=gpu_handle_factory(config))
    eng.init_vars(R.shape[1], R, np.zeros(C.shape[0]), 2.0, 4)
    return eng


def graphs(sp):
    return {"g1": g1_graph(), "powerlaw": sp.problems.powerlaw_graph(20000, 160000, 5)}


@pytest.mark.parametrize("graph", ["g1", "powerlaw"])
def test_maxcut_exact_random_R(sp, gpu_handle_factory, graph):
    A = graphs(sp)[graph]
    C, As, bs = sp.problems.maxcut(A)
    n, r, K = A.shape[0], 10, 100   # one full batch of 64 and a partial one
    rng = np.random.default_rng(17)
    R = 2.0 * rng.random((n, r)) - 1.0
    G = rng.standard_normal((K, r))
    X0 = start_vectors(R, G)
    outs = []
    for config in ("default", "relabel"):
        eng = engine_with_R(sp, gpu_handle_factory, config, C, As, bs, R)
        res = eng.round_local_search(K, G)
        eng.close()
        check_against_reference(res, C, X0, 1000)
        check_local_optimum(res, C)
        assert np.all(res["rounds"] >= 1) and np.all(res["flips"] > 0)
        outs.append(res)
    for key in ("obj_round", "obj", "sum", "flips", "rounds", "best_x", "G_used"):
        np.testing.assert_array_equal(outs[0][key], outs[1][key])


def test_maxcut_exact_after_solve(sp, gpu_handle_factory):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    ans = sp.sdplr(C, As, bs, 10, engine_factory=lambda d: sp.B200Engine(d, handle=gpu_handle_factory("relabel")), printlevel=0,
                   prior_trace_bound=800.0, seed=0, objtol=float("inf"), maxtime=120.0)
    R = ans["Rt"]
    G = np.random.default_rng(3).standard_normal((100, R.shape[1]))
    res = ans["engine"].round_local_search(100, G)
    ans["engine"].close()
    check_against_reference(res, C, start_vectors(R, G), 1000)
    check_local_optimum(res, C)


def test_powerlaw_after_iterations(sp, gpu_handle_factory):
    """hubs (rows longer than the per-thread limit, several segments) on an R that the solver moved"""
    A = graphs(sp)["powerlaw"]
    assert np.diff(sps.csr_matrix(A).indptr).max() > 4096
    C, As, bs = sp.problems.maxcut(A)
    n, r, K = A.shape[0], 8, 100
    R0 = 2.0 * np.random.default_rng(2).random((n, r)) - 1.0
    got = []
    for config in ("default", "relabel"):
        eng = engine_with_R(sp, gpu_handle_factory, config, C, As, bs, R0)
        eng.fg()
        eng.iterate(20)
        R = eng.get_R()
        res = eng.round_local_search(K, seed=5)
        eng.close()
        check_against_reference(res, C, start_vectors(R, res["G_used"]), 1000)
        got.append(res)
    np.testing.assert_array_equal(got[0]["obj"], got[1]["obj"])


def test_matches_round_hyperplane_and_independent_of_K(sp, gpu_handle_factory):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    R = 2.0 * np.random.default_rng(5).random((A.shape[0], 6)) - 1.0
    eng = engine_with_R(sp, gpu_handle_factory, "default", C, As, bs, R)
    hp = eng.round_hyperplane(100, seed=9)
    a100 = eng.round_local_search(100, seed=9)
    a64 = eng.round_local_search(64, seed=9)
    a1 = eng.round_local_search(1, seed=9)
    G = np.random.default_rng(8).standard_normal((70, 6))
    hp_g, ls_g = eng.round_hyperplane(70, G), eng.round_local_search(70, G)
    eng.close()
    np.testing.assert_array_equal(a100["obj_round"], hp["obj"])
    np.testing.assert_array_equal(a100["G_used"], hp["G_used"])
    np.testing.assert_array_equal(ls_g["obj_round"], hp_g["obj"])
    np.testing.assert_array_equal(ls_g["G_used"], G)
    for key in ("obj_round", "obj", "sum", "flips", "rounds", "G_used"):
        np.testing.assert_array_equal(a100[key][:64], a64[key])
        np.testing.assert_array_equal(a100[key][:1], a1[key])
    np.testing.assert_array_equal(a1["best_x"], numpy_local_search(C, start_vectors(R, a1["G_used"]), 1000)[0][:, 0])


def test_real_weights_and_families(sp, gpu_handle_factory):
    rng = np.random.default_rng(21)
    A = g1_graph()
    W = sps.triu(A, k=1).tocoo()
    Wr = sps.coo_matrix((rng.uniform(-1.0, 1.0, W.nnz), (W.row, W.col)), shape=A.shape)
    Wr = (Wr + Wr.T).tocsc()
    cases = [("maxcut_real", sp.SDPData(*sp.problems.maxcut(Wr)), None)]
    for name, fam in families(sp):
        if name == "lovasz_theta":
            continue
        for seed, n, p, r in COMBOS:
            data, Rt0, _ = make_case(sp, fam, seed, n, p, r)
            cases.append((f"{name}/{seed}", data, Rt0))
    for name, data, R in cases:
        if R is None:
            R = 2.0 * rng.random((data.n, 8)) - 1.0
        eng = sp.B200Engine(data, handle=gpu_handle_factory("relabel"))
        eng.init_vars(R.shape[1], R, np.zeros(data.m), 2.0, 4)
        res = eng.round_local_search(70, seed=4)
        eng.close()
        X0 = start_vectors(R, res["G_used"])
        C = sps.csr_matrix(data.C)
        scale = max(1.0, float(np.max(np.abs(res["obj_round"]))))
        obj0 = np.einsum("ik,ik->k", X0, C @ X0)
        amb = np.any(np.abs(R @ res["G_used"].T) <= 1e-12 * np.linalg.norm(R, axis=1)[:, None]
                     * np.linalg.norm(res["G_used"], axis=1)[None, :], axis=0)
        assert np.all(np.abs(res["obj_round"][~amb] - obj0[~amb]) <= 1e-12 * scale), name
        assert np.all(res["obj"] <= res["obj_round"] + 1e-12 * scale), name
        assert np.all(res["rounds"] >= 0), name
        check_local_optimum(res, C, rtol=1e-12)
        assert res["best"] == int(np.argmin(res["obj"]))


def test_max_rounds_truncation(sp, gpu_handle_factory):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    R = 2.0 * np.random.default_rng(9).random((A.shape[0], 10)) - 1.0
    eng = engine_with_R(sp, gpu_handle_factory, "relabel", C, As, bs, R)
    for mr in (0, 1, 2):
        res = eng.round_local_search(100, seed=2, max_rounds=mr)
        X0 = start_vectors(R, res["G_used"])
        check_against_reference(res, C, X0, mr)
        if mr == 0:
            np.testing.assert_array_equal(res["obj"], res["obj_round"])
            assert np.all(res["flips"] == 0) and set(np.unique(res["rounds"])) <= {0, -1}
        assert np.any(res["rounds"] == -1)
    eng.close()


def test_argument_and_state_errors(sp, gpu_handle_factory):
    C, As, bs = sp.problems.maxcut(g1_graph())
    eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=gpu_handle_factory())
    with pytest.raises(sp.SdplrpError) as e:   # no rank yet
        eng.round_local_search(4)
    assert e.value.code == -3
    eng.init_vars(3, np.ones((C.shape[0], 3)), np.zeros(C.shape[0]), 2.0, 4)
    for K, mr in ((0, 10), (4, -1)):
        with pytest.raises(sp.SdplrpError) as e:
            eng.round_local_search(K, max_rounds=mr)
        assert e.value.code == -2
    eng.close()
    data, Rt0, _ = make_case(sp, sp.problems.lovasz_theta, 1, 8, 0.4, 2)
    eng = sp.B200Engine(data, handle=gpu_handle_factory())
    eng.init_vars(2, Rt0, np.zeros(data.m), 2.0, 4)
    with pytest.raises(sp.SdplrpError) as e:
        eng.round_local_search(8)
    assert e.value.code == -2
    eng.close()


@pytest.mark.parametrize("config", ["default", "relabel"])
def test_local_search_changes_no_solver_state(sp, gpu_handle_factory, config):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    n, r = A.shape[0], 8
    R0 = 2.0 * np.random.default_rng(2).random((n, r)) - 1.0
    got = []
    for do_search in (False, True):
        eng = engine_with_R(sp, gpu_handle_factory, config, C, As, bs, R0)
        eng.fg()
        eng.iterate(5)
        if do_search:
            eng.round_local_search(100, seed=1)
        last = eng.iterate(5)
        got.append((last, eng.get_R(), eng.get_G(), eng.get_lambda()))
        eng.close()
    assert got[0][0] == got[1][0]
    for a, b in zip(got[0][1:], got[1][1:]):
        np.testing.assert_array_equal(a, b)


def test_quality_after_solve(sp, gpu_handle_factory):
    C, As, bs = sp.problems.maxcut(g1_graph())
    ans = sp.sdplr(C, As, bs, 10, engine_factory=lambda d: sp.B200Engine(d, handle=gpu_handle_factory()), printlevel=0,
                   prior_trace_bound=800.0, seed=0, maxtime=120.0)
    plain = sp.hyperplane_rounding(ans, trials=64, seed=0)
    out = sp.hyperplane_rounding(ans, trials=64, seed=0, local_search_rounds=1000)
    ans["engine"].close()
    np.testing.assert_array_equal(out["objs_rounded"], plain["objs"])
    assert out["obj"] == out["objs"].min() <= plain["obj"] <= 0.0
    assert out["obj"] >= ans["max_dual_value"]
    assert float(out["x"] @ (sps.csr_matrix(C) @ out["x"])) == out["obj"]
    assert np.all(out["rounds"] >= 0) and np.all(out["flips"] >= 0)


def test_powerlaw_million_vertices(sp, gpu_handle_factory):
    n, r, K = 1_000_000, 10, 2
    asm, b, _, _ = sp.problems.powerlaw_maxcut_assembled(n, 8_000_000, 3)
    lo, hi = int(asm.mat_off[n]), int(asm.mat_off[n + 1])
    C = sps.csr_matrix((asm.V[lo:hi], (asm.I[lo:hi] - 1, asm.J[lo:hi] - 1)), shape=(n, n))

    class Data:   # what B200Engine needs when the triplets are pre-assembled
        pass
    data = Data()
    data.n, data.m, data.b = n, n, b
    data.constraint_types = np.zeros(n, dtype=bool)
    data.has_inequalities = False
    eng = sp.B200Engine(data, handle=gpu_handle_factory(), asm=asm)
    rng = np.random.default_rng(4)
    R = 2.0 * rng.random((n, r)) - 1.0
    eng.init_vars(r, R, np.zeros(n), 2.0, 4)
    G = rng.standard_normal((K, r))
    res = eng.round_local_search(K, G)
    eng.close()
    D = R @ G.T
    assert not np.any(np.abs(D) <= 1e-12 * np.linalg.norm(R, axis=1)[:, None] * np.linalg.norm(G, axis=1)[None, :])
    check_against_reference(res, C, start_vectors(R, G), 1000)


def _gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.mark.parametrize("world", [2, 4, 8])
def test_local_search_on_several_gpus(world):
    if _gpus() < world:
        pytest.skip(f"needs {world} GPUs on one node (have {_gpus()})")
    from test_gpu_multi import _torchrun
    out = _torchrun(world, "check_multigpu_local_search.py", 29680 + world)
    tail = out.stdout[-3000:] + "\n" + out.stderr[-3000:]
    assert out.returncode == 0 and "MULTIGPU LOCAL SEARCH OK" in out.stdout, tail
