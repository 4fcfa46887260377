"""Sweep rounding on the GPU (sdplrp_round_sweep, csrc/rounding.cu) against a NumPy / SciPy restatement: project R g_k,
order the vertices by (projection, input index), evaluate every prefix cut x_t (-1 on the first t vertices) and keep the
best one inside the weight window.  Unit-weight objectives and integer weights make every value exact, so thresholds,
objectives, sums, the best vector, its order and its whole profile are compared bit for bit."""
import math

import numpy as np
import pytest
import scipy.sparse as sps

from conftest import GPU_CONFIG_PARAMS
from helpers import g1_graph, make_case
from rounding_reference import INF, assert_order_determined, cut_value, engine_with_R, numpy_sweep, projections

pytestmark = pytest.mark.gpu

def check_exact(res, ref, n):
    thresh = np.array([c["t"] for c in ref])
    obj = np.array([c["obj"] for c in ref])
    np.testing.assert_array_equal(res["thresh"], thresh)
    np.testing.assert_array_equal(res["obj"], obj)
    ok = thresh >= 0
    np.testing.assert_array_equal(res["sum"][ok], n - 2.0 * thresh[ok])
    np.testing.assert_array_equal(res["wS"][ok], [c["W"][c["t"]] for c in np.array(ref)[ok]])
    b = res["best"]
    assert b == int(np.argmin(obj))
    np.testing.assert_array_equal(res["best_x"], ref[b]["x"])
    np.testing.assert_array_equal(res["best_order"], ref[b]["order"])
    np.testing.assert_array_equal(res["best_profile"], ref[b]["profile"])


def check_maxcut(eng, R, C, K=40, seed=None, G=None):
    if G is None:
        G = np.random.default_rng(seed).standard_normal((K, R.shape[1]))
    P = projections(R, G)
    assert_order_determined(R, G, P)
    res = eng.round_sweep(K, G)
    hp = eng.round_hyperplane(K, G)
    ref = numpy_sweep(C, P)
    check_exact(res, ref, R.shape[0])
    np.testing.assert_array_equal(res["G_used"], G)
    assert np.all(res["obj"] <= hp["obj"])                     # the hyperplane cut is one of the thresholds
    b = res["best"]
    t0 = int(np.sum(P[:, b] < 0))
    assert res["best_profile"][t0] == hp["obj"][b]
    return res


@pytest.mark.parametrize("config", GPU_CONFIG_PARAMS)
def test_maxcut_g1_exact(sp, gpu_handle_factory, config):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    data = sp.SDPData(C, As, bs)
    R = 2.0 * np.random.default_rng(7).random((A.shape[0], 10)) - 1.0
    eng = engine_with_R(sp, gpu_handle_factory, config, data, R)
    check_maxcut(eng, R, C, K=40, seed=1)                        # batches of 16, 16 and 8
    eng.close()
    ans = sp.sdplr(C, As, bs, 10, engine_factory=lambda d: sp.B200Engine(d, handle=gpu_handle_factory(config)), printlevel=0,
                   prior_trace_bound=800.0, seed=0, objtol=INF, maxtime=120.0)
    check_maxcut(ans["engine"], ans["Rt"], C, K=40, seed=3)
    out = sp.sweep_rounding(ans, trials=40, seed=0)
    hp = sp.hyperplane_rounding(ans, trials=40, seed=0)
    assert out["obj"] <= hp["obj"]
    assert float(out["x"] @ (sps.csr_matrix(C) @ out["x"])) == out["obj"]
    ans["engine"].close()


@pytest.mark.parametrize("drop", [False, True])
def test_exact_bisection(sp, gpu_handle_factory, drop):
    A = sps.csr_matrix(g1_graph())
    if drop:   # odd n: the window is [(n - 1) / 2, (n + 1) / 2]
        A = A[1:, 1:].tocsc()
    n = A.shape[0]
    assert (n % 2 == 1) == drop
    C, As, bs = sp.problems.minimum_bisection(A)
    ans = sp.sdplr(C, As, bs, 10, engine_factory=lambda d: sp.B200Engine(d, handle=gpu_handle_factory("relabel")), printlevel=0,
                   prior_trace_bound=800.0, seed=0, objtol=INF, maxtime=120.0)
    R = ans["Rt"]
    out = sp.sweep_rounding(ans, trials=40, seed=2, bisection=True)
    G = ans["engine"].round_hyperplane(40, seed=2)["G_used"]      # the directions sweep_rounding used
    res = ans["engine"].round_sweep(40, G, window=(n // 2, (n + 1) // 2))
    ans["engine"].close()
    P = projections(R, G)
    assert_order_determined(R, G, P)
    ref = numpy_sweep(C, P, window=(n // 2, (n + 1) // 2))
    check_exact(res, ref, n)
    assert np.all(np.abs(res["sum"]) == n % 2)
    assert np.all(np.isin(res["thresh"], [n // 2, (n + 1) // 2]))
    for k in range(40):
        assert res["obj"][k] == cut_value(A, ref[k]["x"])
    np.testing.assert_array_equal(out["objs"], res["obj"])
    assert out["x"].sum() == res["sum"][res["best"]] and abs(out["x"].sum()) == n % 2
    assert out["obj"] == cut_value(A, out["x"])


def powerlaw_case(sp):
    A = sp.problems.powerlaw_graph(20000, 160000, 5)
    assert np.diff(sps.csr_matrix(A).indptr).max() > 4096   # hub rows take the segment path of the delta pass
    return A


@pytest.mark.parametrize("config", ["default", "relabel"])
def test_mu_balanced_window(sp, gpu_handle_factory, config):
    A = powerlaw_case(sp)
    C, As, bs = sp.problems.maxcut(A)
    n, r, K = A.shape[0], 8, 20
    deg = np.asarray(A.sum(axis=1)).reshape(-1)
    vol = float(deg.sum())
    rng = np.random.default_rng(31)
    R = 2.0 * rng.random((n, r)) - 1.0
    G = rng.standard_normal((K, r))
    P = projections(R, G)
    assert_order_determined(R, G, P)
    eng = engine_with_R(sp, gpu_handle_factory, config, sp.SDPData(C, As, bs), R)
    mu = 0.1
    win = (mu * vol, (1 - mu) * vol)
    res = eng.round_sweep(K, G, w=deg, window=win)
    ref = numpy_sweep(C, P, deg, win)
    check_exact(res, ref, n)
    assert np.all((win[0] <= res["wS"]) & (res["wS"] <= win[1]))
    # a window only the last thresholds satisfy: every vertex of positive degree in S_t
    late = (vol - 0.5, INF)
    res = eng.round_sweep(K, G, w=deg, window=late)
    ref = numpy_sweep(C, P, deg, late)
    check_exact(res, ref, n)
    assert np.all(res["wS"] == vol) and np.all(res["thresh"] >= n - np.sum(deg == 0))
    with pytest.raises(sp.SdplrpError) as e:                   # no prefix weighs more than vol
        eng.round_sweep(K, G, w=deg, window=(vol + 1.0, INF))
    assert e.value.code == -2
    eng.close()


def test_ties_follow_input_index(sp, gpu_handle_factory):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    n, r, K = A.shape[0], 4, 24
    rng = np.random.default_rng(12)
    base = 2.0 * rng.random((n // 8, r)) - 1.0
    R = base[rng.integers(0, n // 8, n)]                       # every row repeated about 8 times: exact ties
    G = rng.standard_normal((K, r))
    P = projections(R, G)
    assert_order_determined(R, G, P)
    ref = numpy_sweep(C, P)
    outs = []
    for config in ("default", "relabel"):
        eng = engine_with_R(sp, gpu_handle_factory, config, sp.SDPData(C, As, bs), R)
        res = eng.round_sweep(K, G)
        eng.close()
        check_exact(res, ref, n)
        outs.append(res)
    order = outs[0]["best_order"]
    p = P[order, outs[0]["best"]]
    same = p[1:] == p[:-1]
    assert same.sum() > n // 2 and np.all(order[1:][same] > order[:-1][same])
    for key in ("obj", "sum", "wS", "thresh", "best_x", "best_order", "best_profile"):
        np.testing.assert_array_equal(outs[0][key], outs[1][key])


@pytest.mark.parametrize("r", [1, 3, 33, 64, 256])
def test_ranks(sp, gpu_handle_factory, r):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    R = 2.0 * np.random.default_rng(40 + r).random((A.shape[0], r)) - 1.0
    eng = engine_with_R(sp, gpu_handle_factory, "relabel", sp.SDPData(C, As, bs), R)
    check_maxcut(eng, R, C, K=20, seed=50 + r)
    eng.close()


def test_determinism_and_independence_of_K(sp, gpu_handle_factory):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    R = 2.0 * np.random.default_rng(5).random((A.shape[0], 6)) - 1.0
    eng = engine_with_R(sp, gpu_handle_factory, "default", sp.SDPData(C, As, bs), R)
    a = eng.round_sweep(40, seed=9)
    b = eng.round_sweep(40, seed=9)
    c = eng.round_sweep(17, seed=9)
    hp = eng.round_hyperplane(40, seed=9)
    eng.close()
    for key in a:
        np.testing.assert_array_equal(a[key], b[key])
    np.testing.assert_array_equal(a["G_used"], hp["G_used"])
    for key in ("obj", "sum", "wS", "thresh", "G_used"):
        np.testing.assert_array_equal(a[key][:17], c[key])
    P = projections(R, a["G_used"])
    assert_order_determined(R, a["G_used"], P)
    check_exact(a, numpy_sweep(C, P), A.shape[0])


@pytest.mark.parametrize("config", ["default", "relabel"])
def test_sweep_changes_no_solver_state(sp, gpu_handle_factory, config):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    n, r = A.shape[0], 8
    R0 = 2.0 * np.random.default_rng(2).random((n, r)) - 1.0
    got = []
    for do_sweep in (False, True):
        eng = engine_with_R(sp, gpu_handle_factory, config, sp.SDPData(C, As, bs), R0)
        eng.fg()
        eng.iterate(5)
        if do_sweep:
            eng.round_sweep(40, seed=1, w=np.arange(n, dtype=np.float64), window=(1000.0, 2e5))
        last = eng.iterate(5)
        got.append((last, eng.get_R(), eng.get_G(), eng.get_lambda()))
        eng.close()
    assert got[0][0] == got[1][0]
    for a, b in zip(got[0][1:], got[1][1:]):
        np.testing.assert_array_equal(a, b)


def test_argument_errors(sp, gpu_handle_factory):
    import ctypes as C_
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    n = A.shape[0]
    eng = engine_with_R(sp, gpu_handle_factory, "default", sp.SDPData(C, As, bs), np.ones((n, 3)))
    bad = [dict(K=0), dict(K=4, window=(2.0, 1.0)), dict(K=4, window=(math.nan, 1.0)), dict(K=4, window=(0.0, math.nan)),
           dict(K=4, w=np.where(np.arange(n) == 5, -1.0, 1.0)), dict(K=4, w=np.where(np.arange(n) == 5, INF, 1.0))]
    for kw in bad:
        K = kw.pop("K")
        with pytest.raises(sp.SdplrpError) as e:
            eng.round_sweep(K, **kw)
        assert e.value.code == -2, kw
    h = eng.h
    best = C_.c_int64()
    obj = np.empty(4)
    p = C_.POINTER(C_.c_double)
    assert h.lib.sdplrp_round_sweep(h._h, 4, None, 0, None, -INF, INF, None, None, None, None, None, C_.byref(best), None, None,
                                    None) == -2
    assert h.lib.sdplrp_round_sweep(h._h, 4, None, 0, None, -INF, INF, None, obj.ctypes.data_as(p), None, None, None, None, None,
                                    None, None) == -2
    # only obj and best: every other output may be NULL
    assert h.lib.sdplrp_round_sweep(h._h, 4, None, 0, None, -INF, INF, None, obj.ctypes.data_as(p), None, None, None,
                                    C_.byref(best), None, None, None) == 0
    assert 1 <= best.value <= 4 and np.all(np.isfinite(obj))
    eng.close()
    data, Rt0, _ = make_case(sp, sp.problems.lovasz_theta, 1, 8, 0.4, 2)
    eng = engine_with_R(sp, gpu_handle_factory, "default", data, Rt0)
    with pytest.raises(sp.SdplrpError) as e:
        eng.round_sweep(8)
    assert e.value.code == -2
    eng.close()
