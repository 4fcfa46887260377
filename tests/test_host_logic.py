"""Host-side logic that stays outside the kernels: root selection of the exact line search,
constraint assembly order, problem generators, SymLowRankMatrix norms, utilities."""
import numpy as np
import pytest
import scipy.sparse as sps

from helpers import dense_of, k2_graph, p3_graph


def test_pick_alpha_matches_grid_search(sp):
    rng = np.random.default_rng(0)
    for _ in range(200):
        bq = rng.standard_normal(5)
        bq[1] = -abs(bq[1]); bq[4] = abs(bq[4]) + 0.05
        a, f = sp.pick_alpha(bq, 1.0)
        xs = np.linspace(0, 1, 20001)
        vals = np.polynomial.polynomial.polyval(xs, bq)
        assert 0.0 <= a <= 1.0
        assert f <= vals.min() + 1e-7 * max(1.0, abs(vals.min()))


def test_pick_alpha_edge_cases(sp):
    with pytest.raises(ArithmeticError):
        sp.pick_alpha([0.0, 1.0, 1.0, 0.0, 1.0])                     # src/linesearch.jl:60-62
    a, f = sp.pick_alpha([1.0, -2.0, 1.0, 0.0, 0.0])                  # quadratic fallback :70-83, minimiser at 1
    assert abs(a - 1.0) < 1e-12 and abs(f) < 1e-12
    a, f = sp.pick_alpha([1.0, -1.0, 5.0, 0.0, 0.0])
    assert abs(a - 0.1) < 1e-12
    a, f = sp.pick_alpha([3.0, 0.0, 0.0, 0.0, 0.0])                   # flat: alpha stays 0 (Appendix A.4)
    assert a == 0.0 and f == 3.0


def test_assemble_order_and_global_ids(sp):
    """SolverAuxiliary classification (src/structs.jl:303-332): sparse/diagonal in order, then C; low-rank separate."""
    C, As, bs = sp.problems.minimum_bisection(p3_graph())
    asm = sp.assemble_sparse(sp.SDPData(C, As, bs))
    assert asm.gids.tolist() == [1, 2, 3, 5] and [g for g, _ in asm.lowrank] == [4]
    assert asm.mat_off.tolist()[:4] == [0, 1, 2, 3]
    C, As, bs = sp.problems.lovasz_theta(p3_graph())
    asm = sp.assemble_sparse(sp.SDPData(C, As, bs))
    assert asm.gids.tolist() == [1, 2, 3] and [g for g, _ in asm.lowrank] == [4]
    assert asm.I.tolist()[:4] == [1, 2, 2, 3] and asm.J.tolist()[:4] == [2, 1, 3, 2]   # COO {(i,j),(j,i)} per edge, (j,i)-ordered


def test_generators_match_definitions(sp):
    P = sp.problems
    A = P.erdos_renyi(12, 0.4, 1)
    Ad = A.toarray(); n = 12; d = Ad.sum(1); L = np.diag(d) - Ad
    C, As, bs = P.maxcut(A)
    assert np.allclose(C.toarray(), -0.25 * L) and np.all(bs == 1) and len(As[0]) == n
    C, As, bs = P.minimum_bisection(A)
    assert np.allclose(C.toarray(), 0.25 * L) and np.allclose(As[1].toarray(), np.ones((n, n))) and bs[-1] == 0
    C, As, bs = P.lovasz_theta(A)
    data = sp.SDPData(C, As, bs)
    mats = data.matrices()
    assert np.allclose(C.toarray(), -np.ones((n, n))) and len(mats) == A.nnz // 2 + 1
    assert all(np.allclose(dense_of(M), dense_of(M).T) and dense_of(M).sum() == 2 for M in mats[:-1])
    assert np.allclose(mats[-1].toarray(), np.eye(n)) and bs[-1] == 1 and not bs[:-1].any()
    B = sps.random(5, 7, density=0.5, random_state=1, format="csc")
    C, As, bs = P.cutnorm(B)
    Z = np.zeros((12, 12)); Z[:5, 5:] = B.toarray(); Z[5:, :5] = B.toarray().T
    assert np.allclose(C.toarray(), -Z / 2)
    C, As, bs = P.mu_conductance(A, 0.05)
    data = sp.SDPData(C, As, bs)
    assert data.n == 3 * n and data.m == 2 + 2 * n
    mats = data.matrices()
    assert np.allclose(dense_of(mats[0])[:n, :n], np.diag(d)) and np.allclose(dense_of(mats[1]), np.outer(np.r_[d, np.zeros(2 * n)], np.r_[d, np.zeros(2 * n)]))
    M = dense_of(mats[2 + n]); assert M[0, 0] == 1 and M[2 * n, 2 * n] == -1 and np.count_nonzero(M) == 2
    C, As, bs, types = P.mu_conductance_ineq(A, 0.05)
    assert types.tolist() == [False, False] + [True] * (2 * n) and np.allclose(C.toarray(), L)


def test_symlowrank_norms(sp):
    """test/symlowrank.jl:4-15"""
    rng = np.random.default_rng(0)
    for _ in range(100):
        n = int(rng.integers(50, 101)); s = int(rng.integers(1, 21))
        A = sp.SymLowRankMatrix(rng.standard_normal(s), rng.standard_normal((n, s)))
        dense = A.toarray()
        assert np.isclose(A.norm(2), np.linalg.norm(dense)) and np.isclose(A.norm(np.inf), np.abs(dense).max())


def test_oracle_symlowrank_norm_agrees(sp, oracle_mod):
    import ctypes as C
    rng = np.random.default_rng(1)
    A = sp.SymLowRankMatrix(rng.standard_normal(3), rng.standard_normal((40, 3)))
    lib = oracle_mod.load()
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    assert np.isclose(lib.orc_symlowrank_norm(40, 3, p(A.B), p(A.D), 0), A.norm(2))
    assert np.isclose(lib.orc_symlowrank_norm(40, 3, p(A.B), p(A.D), 1), A.norm(np.inf))


def test_misc(sp):
    assert sp.barvinok_pataki(800, 800) == 41 and sp.barvinok_pataki(5, 1000) == 5      # src/utils.jl:7-11
    cfg = sp.BurerMonteiroConfig()
    cfg.set("σ_0", 10.0); assert cfg.sigma_0 == 10.0
    with pytest.raises(KeyError):
        cfg.set("nonsense", 1)
    assert sp.frobenius_norm(sps.csc_matrix(np.array([[3.0, 0], [0, 4.0]]))) == 5.0


def test_rank_update_clamp(sp):
    """rank_after_update (the rank update of both drivers): always a supported rank, never above min(bp, 2r), and the
    largest supported rank at or below it; the limits are the ones include/sdplrp_b200.h states"""
    import os
    import re
    S = sp.solver
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "sdplrp_b200.h")).read()
    assert int(re.search(r"#define SDPLRP_MAX_RANK (\d+)", hdr).group(1)) == S.MAX_RANK == 256
    assert int(re.search(r"#define SDPLRP_MAX_ODD_RANK (\d+)", hdr).group(1)) == S.MAX_ODD_RANK == 128
    supported = [t for t in range(1, 600) if S.rank_supported(t)]
    assert supported == list(range(1, 129)) + list(range(130, 257, 2))
    for bp in (1, 2, 3, 41, 127, 128, 129, 130, 200, 255, 256, 257, 258, 283, 1000, 10 ** 6):
        for r in range(1, 301):
            want = min(bp, 2 * r)
            t = S.rank_after_update(bp, r)
            assert S.rank_supported(t) and t <= want, (bp, r, t)
            assert t == max(u for u in supported if u <= want), (bp, r, t)
    assert S.rank_after_update(283, 160) == 256 and S.rank_after_update(201, 128) == 200 and S.rank_after_update(41, 40) == 41


def _scaled_quartics(count, seed):
    """quartic coefficient sets over seven orders of magnitude, including the degenerate shapes of the line search"""
    rng = np.random.default_rng(seed)
    for t in range(count):
        bq = rng.standard_normal(5) * 10.0 ** rng.integers(-3, 4, 5)
        bq[1] = -abs(bq[1]); bq[4] = abs(bq[4])
        kind = t % 5
        if kind == 1: bq[4] = 0.0                       # quadratic fallback (src/linesearch.jl:70-83)
        if kind == 2: bq[3] = bq[4] = 0.0               # derivative is linear
        if kind == 3: bq[1] = 0.0                       # zero slope at 0
        if kind == 4: bq[2] = abs(bq[2]); bq[3] = abs(bq[3])
        yield bq


def test_native_pick_alpha_matches_python_and_oracle(sp, oracle_mod):
    """sdplrp_pick_alpha (the native driver's root selection, csrc/driver.cu) against the numpy.roots mirror and the
    oracle's closed-form solver: same minimum of the quartic, same step."""
    import ctypes as C
    ol = oracle_mod.load()
    for bq in _scaled_quartics(4000, 3):
        a_py, f_py = sp.pick_alpha(bq, 1.0)
        a_na, f_na = sp._lib.pick_alpha_native(bq, 1.0)
        a, f = C.c_double(), C.c_double()
        assert ol.orc_pick_alpha(bq.ctypes.data_as(C.POINTER(C.c_double)), 1.0, C.byref(a), C.byref(f)) == 0
        tol = 1e-13 * max(1.0, abs(f_na))
        assert f_na <= f_py + tol, (bq, a_py, a_na)      # numpy.roots loses tiny roots of badly scaled cubics; never the reverse
        assert abs(f_na - f.value) <= tol, (bq, a_na, a.value)
        assert abs(a_na - a.value) <= 1e-9 * max(abs(a_na), 1e-30), (bq, a_na, a.value)
    with pytest.raises(ArithmeticError):
        sp._lib.pick_alpha_native([0.0, 1.0, 1.0, 0.0, 1.0], 1.0)
    assert sp._lib.pick_alpha_native([3.0, 0.0, 0.0, 0.0, 0.0], 1.0) == (0.0, 3.0)
    a, f = sp._lib.pick_alpha_native([1.0, -1.0, 5.0, 0.0, 0.0], 1.0)
    assert abs(a - 0.1) < 1e-15


def test_native_config_defaults_match_reference_options(sp):
    """sdplrp_config_default == BurerMonteiroConfig defaults (src/options.jl:1-24); 21 fields of 8 bytes"""
    import ctypes as C
    cfg = sp._lib.default_config()
    assert C.sizeof(sp._lib.Config) == 21 * 8 and C.sizeof(sp._lib.Result) == 22 * 8
    ref = sp.BurerMonteiroConfig()
    for k in ("ptol", "gtol", "objtol", "sigma_0", "sigmafac", "maxtime", "printfreq", "fprec", "prior_trace_bound",
              "maxmajoriter", "maxiter", "numlbfgsvecs", "rankupd_tol", "printlevel"):
        assert getattr(cfg, k) == getattr(ref, k), k
    assert (cfg.gtol_relative, cfg.ptol_relative, cfg.objtol_relative) == (1, 1, 1)
    assert (cfg.eval_DIMACS_errs, cfg.eigval_highprecision, cfg.alpha_max) == (0, 0, 1.0)


def test_native_seed_stream_is_a_fixed_sequence(sp):
    from sdplrplus.jl_b200.solver import native_seed
    s = [native_seed(0, k) for k in range(1, 5)]
    assert len(set(s)) == 4 and all(0 <= x < 2 ** 64 for x in s)
    assert native_seed(7, 3) == native_seed(7, 3) != native_seed(8, 3)


def test_native_driver_needs_the_gpu_engine(sp, oracle_mod):
    C, As, bs = sp.problems.maxcut(k2_graph())
    with pytest.raises(TypeError):
        sp.sdplr(C, As, bs, 1, engine_factory=oracle_mod.OracleEngine, driver="native", printlevel=0)
