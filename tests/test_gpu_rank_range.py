"""Every rank-dependent path of the GPU kernels over the whole supported rank range (r <= 256, odd r <= 128), against the
CPU oracle and a float64 NumPy restatement of the operators taken straight from the matrices:

  a. the operators and one L-BFGS step pair at ranks on both sides of every branch that depends on r (vector width 1 / 2,
     the lane group of one to 32 lanes per row, one or up to four 32-lane units per row, the per-row constraint warp or
     tile kernel, the gather modes' own rank limits, rows per block of the low-rank projection),
  b. hyperplane rounding and one-flip local search at r > 32 (the multi-column sign pass), bit for bit,
  c. low-rank matrices B D B' with s from 1 to 17 (one to three column chunks of the projection, mixed-sign D with a zero,
     zero rows in B) as a constraint, as two constraints and as the objective, and the Lanczos eigenvalues of such an S,
  d. the rank contract of sdplrp_set_rank and the clamped rank update of both drivers."""
import math

import numpy as np
import pytest
import scipy.sparse as sps

from conftest import GPU_CONFIG_PARAMS
from helpers import dense_S, g1_graph
from rounding_reference import check_against_reference, check_exact, start_vectors

pytestmark = pytest.mark.gpu

# ranks on both sides of every rank-dependent branch: 31/32/33 (nv <= 16 / 32 lane groups, the row-constraint warp kernel,
# kSignCols), 63..66 (one -> two units per row, gather_mode 2 up to r = 64), 100 (TPB % r != 0), 127 / 128 (largest odd,
# a power of two), 130 ... 256 (up to four units per row; 256 is the largest supported rank)
RANKS = [1, 2, 3, 31, 32, 33, 63, 64, 65, 66, 100, 127, 128, 130, 192, 250, 256]
LARGE_R_CONFIGS = ["default", "relabel", "gather_bulk", "gather_async_small"]
OP_CASES = [pytest.param(c, r, id=f"{c}-r{r}") for r in RANKS for c in (GPU_CONFIG_PARAMS if r < 128 else LARGE_R_CONFIGS)]
UNSUPPORTED = [129, 131, 255, 257, 258, 300, 514]


def _relclose(a, b, tol, what=""):
    a, b = np.asarray(a, float), np.asarray(b, float)
    scale = max(1.0, float(np.max(np.abs(b))) if b.size else 1.0)
    err = float(np.max(np.abs(a - b))) if a.size else 0.0
    assert err <= tol * scale, f"{what}: err {err:.3e} scale {scale:.3e}"


def _pair(sp, oracle_mod, handle, data, Rt0, r, lam0=None, sigma=2.0, hist=4):
    lam0 = np.zeros(data.m) if lam0 is None else lam0
    ge = sp.B200Engine(data, handle=handle)
    ge.init_vars(r, Rt0, lam0, sigma, hist)
    oe = oracle_mod.OracleEngine(data)
    oe.init_vars(r, Rt0, lam0, sigma, hist)
    return ge, oe


@pytest.fixture
def handles(gpu_handle_factory):
    """gpu_handle_factory with every handle closed at the end of the test"""
    made = []

    def make(config="default", **opts):
        h = gpu_handle_factory(config)
        for k, v in opts.items():
            h.set_option(k, v)
        made.append(h)
        return h
    yield make
    for h in made:
        h.close()


# ---------------------------------------------------------------- float64 restatement of the operators
def _coo_terms(U, V, rows, cols, vals):
    """v_k (U_i.V_j + V_i.U_j) / 2 per stored entry (i, j, v_k)"""
    return vals * 0.5 * (np.einsum("ij,ij->i", U[rows], V[cols]) + np.einsum("ij,ij->i", V[rows], U[cols]))


def ref_A(sp, data, U, V=None):
    """[<A_i, (UV' + VU')/2> for every constraint ; <C, (UV' + VU')/2>]; a low-rank A = B D B' as tr(U'B D B'V)"""
    V = U if V is None else V

    def one(A):
        if isinstance(A, sp.SymLowRankMatrix):
            return float(np.sum((U.T @ A.B) * (V.T @ A.B) * A.D[None, :]))
        if isinstance(A, sp.types.SparseMatrixCOO):
            return float(_coo_terms(U, V, A.rows, A.cols, A.vals).sum())
        c = sps.coo_matrix(A)
        return float(_coo_terms(U, V, c.row, c.col, c.data).sum())
    out = []
    for A in data.As:
        if isinstance(A, sp.types.ConstraintBatch):
            idx = np.repeat(np.arange(len(A)), np.diff(A.offsets))
            out.extend(np.bincount(idx, weights=_coo_terms(U, V, A.rows, A.cols, A.vals), minlength=len(A)))
        else:
            out.append(one(A))
    out.append(one(data.C))
    return np.array(out)


def ref_S_times(sp, data, y, X):
    """(sum_i y_i A_i + y_m C) X"""
    X = np.asarray(X, float)
    out = np.zeros_like(X)

    def add(A, w):
        nonlocal out
        if isinstance(A, sp.SymLowRankMatrix):
            out += w * (A.B @ (A.D[:, None] * (A.B.T @ X)))
        elif isinstance(A, sp.types.SparseMatrixCOO):
            np.add.at(out, A.rows, (w * A.vals)[:, None] * X[A.cols])
        else:
            out += w * (sps.csr_matrix(A) @ X)
    i = 0
    for A in data.As:
        if isinstance(A, sp.types.ConstraintBatch):
            k = len(A)
            wk = y[i + np.repeat(np.arange(k), np.diff(A.offsets))] * A.vals
            np.add.at(out, A.rows, wk[:, None] * X[A.cols])
            i += k
        else:
            add(A, y[i])
            i += 1
    add(data.C, y[data.m])
    return out


# ---------------------------------------------------------------- a. operators at every supported rank
_DATA = {}


def _data(sp, which):
    if which not in _DATA:
        P = sp.problems
        if which == "powerlaw_maxcut":   # rows in all three gather row classes (<= 32, <= 512, longer)
            C, As, bs = P.maxcut(P.powerlaw_graph(4000, 60000, 3, exponent=2.1))
        else:                            # Diag(X) = 1 and the rank-one 11' constraint
            C, As, bs = P.minimum_bisection(P.erdos_renyi(120, 0.08, 11))
        _DATA[which] = sp.SDPData(C, As, bs)
    return _DATA[which]


def _operator_pass(sp, oracle_mod, h, data, r, seed):
    """seam products against the restatement, then f/g, two line-search steps with L-BFGS updates and the third direction
    against the oracle (the GPU takes the oracle's step size and, after each step, its iterate: the rank-one families
    amplify rounding noise from one step to the next)"""
    rng = np.random.default_rng(seed)
    R = 2.0 * rng.random((data.n, r)) - 1.0
    V = rng.standard_normal((data.n, r))
    lam0 = 0.1 * rng.standard_normal(data.m)
    ge, oe = _pair(sp, oracle_mod, h, data, R, r, lam0=lam0)
    L = sp._lib
    h.upload_mat(L.MAT_W1, V)
    _relclose(h.A_uu(L.MAT_R), ref_A(sp, data, R), 1e-10, "A_uu")
    _relclose(h.A_uv(L.MAT_R, L.MAT_W1), ref_A(sp, data, R, V), 1e-10, "A_uv")
    _relclose(h.A_uu(L.MAT_R), oe.o.A_uu(R), 1e-12, "A_uu vs oracle")
    y = np.concatenate([rng.standard_normal(data.m), [-0.37]])
    h.At_preprocess(y)
    h.At_left(L.MAT_R, L.MAT_W0)
    _relclose(h.download_mat(L.MAT_W0), ref_S_times(sp, data, y, R), 1e-10, "At_left")
    _relclose(h.At_right(V), ref_S_times(sp, data, y, V), 1e-10, "At_right")
    _relclose(h.At_right(V[:, 0]), ref_S_times(sp, data, y, V[:, :1])[:, 0], 1e-10, "At_right, one column")

    _relclose(ge.fg(), oe.fg(), 1e-11, "fg")
    _relclose(ge.get_pvio_raw(), oe.get_pvio_raw(), 1e-12, "pvio_raw")
    _relclose(ge.get_G(), oe.get_G(), 1e-12, "G")
    _relclose(ge.get_y(), oe.get_y(), 1e-12, "y")
    _relclose(ge.get_G(), 2.0 * ref_S_times(sp, data, oe.get_y(), R), 1e-10, "G vs 2 S R")
    for it in range(3):
        dg, do = ge.lbfgs_dir(), oe.lbfgs_dir()
        Do = oe.get_D()
        assert np.linalg.norm(ge.get_D() - Do) <= 1e-10 * np.linalg.norm(Do), f"direction it={it}"
        assert abs(dg - do) <= 1e-10 * max(1.0, abs(do)), f"descent it={it}"
        if it == 2:       # the direction after two updates
            break
        if math.isnan(do) or do >= 0:
            ge.use_gradient_direction(); oe.use_gradient_direction()
        bqg, bqo = ge.linesearch_coeffs(), oe.linesearch_coeffs()
        _relclose(bqg, bqo, 1e-11 if it == 0 else 1e-10, f"quartic coefficients it={it}")
        _relclose(h.download_vec(L.VEC_A_RD, data.m + 1), oe.o.view("A_RD"), 1e-12 if it == 0 else 1e-10, "A_RD")
        _relclose(h.download_vec(L.VEC_A_DD, data.m + 1), oe.o.view("A_DD"), 1e-12 if it == 0 else 1e-10, "A_DD")
        alpha, _ = sp.pick_alpha(bqo, 1.0)
        objg, gn2, pn2 = ge.step_g(alpha)
        objo = oe.step(alpha); ogn2, opn2 = oe.g()
        _relclose([objg, math.sqrt(gn2), math.sqrt(pn2)], [objo, math.sqrt(ogn2), math.sqrt(opn2)], 1e-10, f"step_g it={it}")
        _relclose(ge.get_R(), oe.get_R(), 1e-10, f"R it={it}")
        _relclose(ge.get_G(), oe.get_G(), 1e-10, f"G after the step it={it}")
        ge.lbfgs_update(alpha); oe.lbfgs_update(alpha)
        ge.set_R(oe.get_R()); ge.fg()    # teacher-forced: the next step starts from the oracle's iterate
        _relclose(ge.get_G(), oe.get_G(), 1e-12, f"G at the oracle's iterate it={it}")


@pytest.mark.parametrize("which", ["powerlaw_maxcut", "bisection"])
@pytest.mark.parametrize("config,r", OP_CASES)
def test_operators_at_every_rank(sp, oracle_mod, handles, config, r, which):
    _operator_pass(sp, oracle_mod, handles(config), _data(sp, which), r, 1000 + r)


@pytest.mark.parametrize("which", ["powerlaw_maxcut", "bisection"])
@pytest.mark.parametrize("r", [3, 33, 66, 128])
@pytest.mark.parametrize("knob", [{"spmm_unroll": 4}, {"spmm_g0": 0}], ids=["spmm_unroll4", "spmm_g0_off"])
def test_operators_with_gather_knobs(sp, oracle_mod, handles, knob, r, which):
    """the class-0 register kernel with 4 nonzeros per predicated block, and lane groups of the next power of two instead of
    exactly r/2 lanes: other lanes take other pieces of a row"""
    _operator_pass(sp, oracle_mod, handles("default", **knob), _data(sp, which), r, 2000 + r)


# ---------------------------------------------------------------- b. rounding and local search at r > 32
ROUND_RANKS = [33, 40, 64, 65, 100, 256]


@pytest.mark.parametrize("config", ["default", "relabel"])
@pytest.mark.parametrize("r", ROUND_RANKS)
def test_rounding_and_local_search_multi_column(sp, handles, config, r):
    """r > 32: the sign pass walks the hyperplanes in 32-column slices with a barrier per slice inside the row loop.
    K = 100: one full batch of 64 candidates and a partial one.  check_exact asserts that no candidate has a row inside
    the tie margin (the seeds are chosen so), then every objective, sum, the best candidate and its vector bit for bit."""
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    rng = np.random.default_rng(500 + r)
    R = 2.0 * rng.random((A.shape[0], r)) - 1.0
    G = rng.standard_normal((100, r))
    eng = sp.B200Engine(sp.SDPData(C, As, bs), handle=handles(config))
    eng.init_vars(r, R, np.zeros(A.shape[0]), 2.0, 4)
    check_exact(eng.round_hyperplane(100, G), R, G, C, A)
    check_against_reference(eng.round_local_search(100, G), C, start_vectors(R, G), 1000)


def test_rounding_after_a_solve_at_the_barvinok_pataki_rank(sp, handles):
    """G1: barvinok_pataki(800, 800) = 41 (odd, > 32) is the rank a solve that has reached the bound rounds at"""
    A = g1_graph()
    C, As, bs = sp.problems.maxcut(A)
    r = sp.barvinok_pataki(800, 800)
    assert r == 41
    h = handles("default")
    ans = sp.sdplr(C, As, bs, r, engine_factory=lambda d: sp.B200Engine(d, handle=h), printlevel=0, prior_trace_bound=800.0,
                   seed=0, objtol=float("inf"), maxtime=120.0)
    assert ans["r"] == 41
    R = ans["Rt"]
    G = np.random.default_rng(41).standard_normal((100, r))
    check_exact(ans["engine"].round_hyperplane(100, G), R, G, C, A)
    check_against_reference(ans["engine"].round_local_search(100, G), C, start_vectors(R, G), 1000)


# ---------------------------------------------------------------- c. low-rank matrices with general s
LR_S = [1, 2, 7, 8, 9, 16, 17]
LR_RANKS = [1, 3, 33, 100, 256]


def _lowrank(n, s, seed):
    """B D B' with D of alternating signs (a zero entry for s >= 3) and every 7th row of B zero"""
    rng = np.random.default_rng(seed)
    D = rng.uniform(0.5, 1.5, s) * (-1.0) ** np.arange(s)
    if s >= 3:
        D[s // 2] = 0.0
    B = rng.standard_normal((n, s))
    B[::7] = 0.0
    return D, B


def _lr_problem(sp, role, s):
    P = sp.problems
    G = P.erdos_renyi(150, 0.05, 21)
    n = G.shape[0]
    if role == "objective":          # the lovasz_theta shape: low-rank C, trace and edge constraints
        _, As, bs = P.lovasz_theta(G)
        return sp.SDPData(sp.SymLowRankMatrix(*_lowrank(n, s, 30 + s)), As, bs)
    C, As, bs = P.maxcut(G)
    As = list(As) + [sp.SymLowRankMatrix(*_lowrank(n, s, 40 + s))]
    bs = list(bs) + [0.7]
    if role == "two_constraints":    # a second low-rank constraint of another width
        s2 = 9 if s != 9 else 2
        As.append(sp.SymLowRankMatrix(*_lowrank(n, s2, 50 + s2)))
        bs.append(-0.4)
    return sp.SDPData(C, As, np.array(bs))


@pytest.mark.parametrize("config", ["default", "relabel"])
@pytest.mark.parametrize("r", LR_RANKS)
@pytest.mark.parametrize("s", LR_S)
@pytest.mark.parametrize("role", ["constraint", "two_constraints", "objective"])
def test_lowrank_general_s(sp, oracle_mod, handles, role, s, r, config):
    """the projection X'B in chunks of 8 columns (s > 8: two or three launches, the last one partial), the trace and apply
    kernels with s > 1; <A, UU'> = tr(U'B D B'U) and G = 2 (S R + sum_g y_g B D B' R) against dense NumPy and the oracle"""
    data = _lr_problem(sp, role, s)
    h = handles(config)
    rng = np.random.default_rng(7 * s + r)
    R = 2.0 * rng.random((data.n, r)) - 1.0
    V = rng.standard_normal((data.n, r))
    lam0 = 0.3 * rng.standard_normal(data.m)
    ge, oe = _pair(sp, oracle_mod, h, data, R, r, lam0=lam0)
    L = sp._lib
    mats = [M.toarray() if hasattr(M, "toarray") else np.asarray(M) for M in data.matrices()] + [data.C.toarray()]
    dense = lambda X: np.array([np.sum(M * X) for M in mats])
    h.upload_mat(L.MAT_W1, V)
    _relclose(h.A_uu(L.MAT_R), dense(R @ R.T), 1e-10, "A_uu vs dense")
    _relclose(h.A_uv(L.MAT_R, L.MAT_W1), dense(0.5 * (R @ V.T + V @ R.T)), 1e-10, "A_uv vs dense")
    _relclose(h.A_uu(L.MAT_R), oe.o.A_uu(R), 1e-12, "A_uu vs oracle")
    _relclose(h.A_uv(L.MAT_R, L.MAT_W1), oe.o.A_uv(R, V), 1e-12, "A_uv vs oracle")

    _relclose(ge.fg(), oe.fg(), 1e-11, "fg")
    y = ge.get_y()
    _relclose(y, oe.get_y(), 1e-12, "y")
    _relclose(ge.get_G(), 2.0 * dense_S(data, y) @ R, 1e-10, "G vs dense")
    _relclose(ge.get_G(), oe.get_G(), 1e-12, "G vs oracle")
    ge.set_D(V); oe.set_D(V)
    _relclose(ge.linesearch_coeffs(), oe.linesearch_coeffs(), 1e-11, "quartic coefficients")
    A_RD, A_DD = h.download_vec(L.VEC_A_RD, data.m + 1), h.download_vec(L.VEC_A_DD, data.m + 1)
    _relclose(A_RD, oe.o.view("A_RD"), 1e-12, "A_RD vs oracle")
    _relclose(A_DD, oe.o.view("A_DD"), 1e-12, "A_DD vs oracle")
    _relclose(A_RD, dense(R @ V.T + V @ R.T), 1e-10, "A_RD vs dense")
    _relclose(A_DD, dense(V @ V.T), 1e-10, "A_DD vs dense")

    y2 = np.concatenate([rng.standard_normal(data.m), [0.8]])
    S = dense_S(data, y2)
    h.At_preprocess(y2)
    h.At_left(L.MAT_R, L.MAT_W0)
    _relclose(h.download_mat(L.MAT_W0), S @ R, 1e-10, "At_left")
    _relclose(h.At_right(V), S @ V, 1e-10, "At_right")


def test_lanczos_eigenvalues_with_a_wide_lowrank_term(sp, oracle_mod, handles):
    """sdplrp_S_eigval (thick-restart Lanczos; its S*x includes the B D B' terms) with s = 9 against the dense spectrum"""
    data = _lr_problem(sp, "constraint", 9)
    h = handles("default")
    rng = np.random.default_rng(9)
    R = 2.0 * rng.random((data.n, 5)) - 1.0
    ge, oe = _pair(sp, oracle_mod, h, data, R, 5, lam0=0.3 * rng.standard_normal(data.m))
    ge.fg()
    lam = np.linalg.eigvalsh(dense_S(data, ge.get_y()))
    ev, bd, mv, rs = h.S_eigval(nevs=3, tol=0.0, v0=rng.standard_normal(data.n))
    np.testing.assert_allclose(ev, lam[:3], rtol=0, atol=1e-9 * max(1.0, abs(lam).max()))


# ---------------------------------------------------------------- d. the rank contract
@pytest.mark.parametrize("r", UNSUPPORTED)
def test_set_rank_rejects_unsupported_ranks(sp, oracle_mod, handles, r):
    """r > 256, or odd r > 128: SDPLRP_ERR_ARG before anything is launched, and the previous state stays usable"""
    P = sp.problems
    data = sp.SDPData(*P.maxcut(P.erdos_renyi(300, 0.03, 4)))
    h = handles("default")
    R = 2.0 * np.random.default_rng(r).random((data.n, 10)) - 1.0
    ge, oe = _pair(sp, oracle_mod, h, data, R, 10)
    launches = h.launch_count()
    with pytest.raises(sp.SdplrpError) as e:
        h.set_rank(r, 4)
    assert e.value.code == -2 and "256" in str(e.value) and "128" in str(e.value)
    assert h.launch_count() == launches
    with pytest.raises(sp.SdplrpError) as e:
        ge.init_vars(r, np.zeros((data.n, r)), np.zeros(data.m), 2.0, 4)
    assert e.value.code == -2
    assert h.launch_count() == launches
    np.testing.assert_array_equal(ge.get_R(), R)          # rank 10 and its factor are untouched
    _relclose(ge.fg(), oe.fg(), 1e-11, "fg after the rejected call")
    ge.init_vars(10, R, np.zeros(data.m), 2.0, 4)
    _relclose(ge.fg(), oe.fg(), 1e-11, "fg after set_rank(10)")
    _relclose(ge.get_G(), oe.get_G(), 1e-12, "G after set_rank(10)")


def _unit_rows(data, r):
    """feasible start for MaxCut (unit rows, lambda = 0): the primal objective sits above every dual bound"""
    R = 2.0 * np.random.default_rng(r).random((data.n, r)) - 1.0
    return R / np.linalg.norm(R, axis=1, keepdims=True), np.zeros(data.m)


@pytest.mark.parametrize("driver", ["native", "python"])
def test_rank_update_clamps_to_the_largest_supported_rank(sp, handles, driver):
    """n = 40 000: barvinok_pataki = 283 > 256.  From r = 160 the update asks for min(283, 320) = 283 (odd, unsupported)
    and must land on 256.  No inner iterations (gtol huge), every dual check counts (ptol huge), the start point is
    feasible so the gap (~1e5) stays above objtol = 1e3, and the second check improves it by less than objtol: the second
    major iteration updates the rank, and maxmajoriter = 2 ends the solve there."""
    P = sp.problems
    C, As, bs = P.maxcut(P.gnm_graph(40000, 120000, 5))
    assert sp.barvinok_pataki(40000, 40000) == 283
    h = handles("default")
    with pytest.raises(sp.SdplrpError) as e:    # an unsupported start is refused up front
        sp.sdplr(C, As, bs, 283, engine_factory=lambda d: sp.B200Engine(d, handle=h), driver=driver, printlevel=0, maxtime=60.0)
    assert e.value.code == -2
    res = sp.sdplr(C, As, bs, 160, engine_factory=lambda d: sp.B200Engine(d, handle=h), driver=driver, printlevel=0,
                   init_func=_unit_rows, gtol=1e30, ptol=1e30, objtol=1e3, objtol_mode="absolute", rankupd_tol=1,
                   maxmajoriter=2, prior_trace_bound=40000.0, seed=1, maxtime=120.0)
    assert res["r"] == 256 and res["majoriter"] == 2
    if driver == "native":
        assert res["status"] in (0, 1)
    assert res["Rt"].shape == (40000, 256)
