"""Hyperplane rounding on the GPU (sdplrp_round_hyperplane, csrc/rounding.cu) against NumPy / SciPy: the signs of R g_k,
the objective x'Cx of every candidate (exact for unit-weight MaxCut, whose sums are multiples of 1/4), the imbalance,
the best candidate and its +-1 vector, seeding, and that rounding leaves the solver state untouched."""
import numpy as np
import pytest
import scipy.sparse as sps

from conftest import GPU_CONFIG_PARAMS
from helpers import COMBOS, families, g1_graph, make_case
from rounding_reference import check_exact, numpy_rounding

pytestmark = pytest.mark.gpu


def engine_for(sp, gpu_handle_factory, config, C, As, bs):
    return sp.B200Engine(sp.SDPData(C, As, bs), handle=gpu_handle_factory(config))


@pytest.mark.parametrize("config", GPU_CONFIG_PARAMS)
def test_maxcut_exact_random_R(sp, gpu_handle_factory, config):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    eng = engine_for(sp, gpu_handle_factory, config, C, As, bs)
    rng = np.random.default_rng(7)
    r = 10
    R = 2.0 * rng.random((A.shape[0], r)) - 1.0
    eng.init_vars(r, R, np.zeros(A.shape[0]), 2.0, 4)
    G = rng.standard_normal((100, r))   # one full batch of 64 and a partial one
    res = eng.round_hyperplane(100, G)
    check_exact(res, R, G, C, A)
    eng.close()


@pytest.mark.parametrize("config", GPU_CONFIG_PARAMS)
def test_maxcut_exact_after_solve(sp, gpu_handle_factory, config):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    ans = sp.sdplr(C, As, bs, 10, engine_factory=lambda d: sp.B200Engine(d, handle=gpu_handle_factory(config)), printlevel=0,
                   prior_trace_bound=800.0, seed=0, objtol=float("inf"), maxtime=120.0)
    R = ans["Rt"]
    G = np.random.default_rng(3).standard_normal((100, R.shape[1]))
    res = ans["engine"].round_hyperplane(100, G)
    check_exact(res, R, G, C, A)
    ans["engine"].close()


@pytest.mark.parametrize("config", ["default", "relabel"])
def test_families_match_numpy(sp, gpu_handle_factory, config):
    for name, fam in families(sp):
        for seed, n, p, r in COMBOS:
            data, Rt0, rng = make_case(sp, fam, seed, n, p, r)
            h = gpu_handle_factory(config)
            eng = sp.B200Engine(data, handle=h)
            eng.init_vars(r, Rt0, np.zeros(data.m), 2.0, 4)
            G = rng.standard_normal((70, r))
            if name == "lovasz_theta":
                with pytest.raises(sp.SdplrpError) as e:
                    eng.round_hyperplane(70, G)
                assert e.value.code == -2
                eng.close()
                continue
            res = eng.round_hyperplane(70, G)
            X, obj, tot, amb = numpy_rounding(Rt0, G, data.C)
            ok = ~amb
            scale = max(1.0, float(np.max(np.abs(obj))))
            assert np.all(np.abs(res["obj"][ok] - obj[ok]) <= 1e-12 * scale), (name, seed, n, p, r)
            np.testing.assert_array_equal(res["sum"][ok], tot[ok])
            eng.close()


def test_argument_and_state_errors(sp, gpu_handle_factory):
    C, As, bs = sp.problems.maxcut(g1_graph())
    h = gpu_handle_factory()
    eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=h)
    with pytest.raises(sp.SdplrpError) as e:   # no rank yet
        eng.round_hyperplane(4)
    assert e.value.code == -3
    eng.init_vars(3, np.ones((C.shape[0], 3)), np.zeros(C.shape[0]), 2.0, 4)
    with pytest.raises(sp.SdplrpError) as e:
        eng.round_hyperplane(0)
    assert e.value.code == -2
    eng.close()


def test_zero_rows_round_to_plus_one(sp, gpu_handle_factory):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    eng = engine_for(sp, gpu_handle_factory, "relabel", C, As, bs)
    rng = np.random.default_rng(11)
    R = 2.0 * rng.random((A.shape[0], 4)) - 1.0
    zero = rng.choice(A.shape[0], 50, replace=False)
    R[zero] = 0.0
    eng.init_vars(4, R, np.zeros(A.shape[0]), 2.0, 4)
    G = rng.standard_normal((64, 4))
    res = eng.round_hyperplane(64, G)
    assert np.all(res["best_x"][zero] == 1.0)
    X = np.where(R @ G.T >= 0, 1.0, -1.0)
    np.testing.assert_array_equal(res["sum"], X.sum(axis=0))
    np.testing.assert_array_equal(res["obj"], np.einsum("ik,ik->k", X, sps.csr_matrix(C) @ X))
    eng.close()


def test_seeding_and_determinism(sp, gpu_handle_factory):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    R = 2.0 * np.random.default_rng(5).random((A.shape[0], 6)) - 1.0
    outs = {}
    for config in ("default", "relabel"):
        eng = engine_for(sp, gpu_handle_factory, config, C, As, bs)
        eng.init_vars(6, R, np.zeros(A.shape[0]), 2.0, 4)
        outs[config] = (eng.round_hyperplane(100, seed=9), eng.round_hyperplane(64, seed=9), eng.round_hyperplane(64, seed=10))
        eng.close()
    eng2 = engine_for(sp, gpu_handle_factory, "default", C, As, bs)
    eng2.init_vars(6, R, np.zeros(A.shape[0]), 2.0, 4)
    again = eng2.round_hyperplane(100, seed=9)
    eng2.close()
    a100, a64, b64 = outs["default"]
    for other in (outs["relabel"][0], again):
        np.testing.assert_array_equal(other["G_used"], a100["G_used"])
        np.testing.assert_array_equal(other["obj"], a100["obj"])
        np.testing.assert_array_equal(other["best_x"], a100["best_x"])
    np.testing.assert_array_equal(a100["G_used"][:64], a64["G_used"])
    np.testing.assert_array_equal(a100["obj"][:64], a64["obj"])
    np.testing.assert_array_equal(a100["sum"][:64], a64["sum"])
    assert not np.any(np.all(b64["G_used"] == a64["G_used"], axis=1))
    g = a100["G_used"].reshape(-1)   # standard normals
    assert abs(g.mean()) < 0.1 and abs(g.std() - 1.0) < 0.1
    check_exact(a100, R, a100["G_used"], C, A)


@pytest.mark.parametrize("config", ["default", "relabel"])
def test_rounding_changes_no_solver_state(sp, gpu_handle_factory, config):
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    n, r = A.shape[0], 8
    R0 = 2.0 * np.random.default_rng(2).random((n, r)) - 1.0
    got = []
    for do_round in (False, True):
        eng = engine_for(sp, gpu_handle_factory, config, C, As, bs)
        eng.init_vars(r, R0, np.zeros(n), 2.0, 4)
        eng.fg()
        eng.iterate(5)
        if do_round:
            eng.round_hyperplane(100, seed=1)
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
    out = sp.hyperplane_rounding(ans, trials=64, seed=0)
    assert out["obj"] == out["objs"][out["trial"]] == out["objs"].min()
    assert set(np.unique(out["x"])) <= {-1.0, 1.0}
    assert float(out["x"] @ (sps.csr_matrix(C) @ out["x"])) == out["obj"]
    assert -out["obj"] >= 0.878 * -ans["obj"]
    assert out["obj"] >= ans["max_dual_value"]
    ans["engine"].close()


def test_powerlaw_million_vertices(sp, gpu_handle_factory):
    n, r, K = 1_000_000, 10, 64
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
    res = eng.round_hyperplane(K, G)
    X, obj, tot, amb = numpy_rounding(R, G, C)
    ok = ~amb
    assert ok.sum() >= K - 2
    np.testing.assert_array_equal(res["obj"][ok], obj[ok])
    np.testing.assert_array_equal(res["sum"][ok], tot[ok])
    b = res["best"]
    if ok[b]:
        np.testing.assert_array_equal(res["best_x"], X[:, b])
    eng.close()


def _gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.mark.parametrize("world", [2, 4, 8])
def test_rounding_on_several_gpus(world):
    """hyperplane rounding, local search and sweep rounding on 2 / 4 / 8 ranks, every rank exact against NumPy"""
    if _gpus() < world:
        pytest.skip(f"needs {world} GPUs on one node (have {_gpus()})")
    from test_gpu_multi import _torchrun
    out = _torchrun(world, "check_multigpu_rounding.py", 29660 + world)
    tail = out.stdout[-3000:] + "\n" + out.stderr[-3000:]
    assert out.returncode == 0, tail
    for method in ("ROUNDING", "LOCAL SEARCH", "SWEEP"):
        assert f"MULTIGPU {method} OK" in out.stdout, tail
