"""The value-free gather pass (option "obj_value_free"): when every off-diagonal value of C is the same power of two
(unweighted MaxCut: 0.25), CD = C*D sums the gathered rows of D unscaled, takes C_ii / v at the diagonal and scales each
row by v once.  Scaling by a power of two commutes with rounding, so every result must have the same bits as the pass
that reads C's values -- at every rank, through every row class (lane group, warp, chunked long rows) and both vertex
orders, for v = 0.25 and v = -0.25.  Weighted graphs and a uniform weight that is not a power of two keep the valued
pass."""
import numpy as np
import pytest
import scipy.sparse as sps

from helpers import g1_graph

pytestmark = pytest.mark.gpu

RANKS = [1, 3, 10, 33, 64, 66, 128, 256]
_DATA = {}


def _data(sp, which):
    if which not in _DATA:
        P = sp.problems
        if which == "g1":
            C, As, bs = P.maxcut(g1_graph())
        elif which == "powerlaw":        # rows in all three gather row classes (<= 32, <= 512, longer nonzeros)
            C, As, bs = P.maxcut(P.powerlaw_graph(4000, 60000, 3, exponent=2.1))
        elif which == "weighted":
            A = sps.csc_matrix(g1_graph())
            A.data = 1.0 + np.random.default_rng(5).integers(0, 4, A.nnz).astype(float)
            A = sps.csc_matrix((A + A.T) * 0.5)
            C, As, bs = P.maxcut(A)
        elif which == "uniform_0.3":     # off-diagonal -0.25 * -1.2 = 0.3: uniform, not a power of two
            C, As, bs = P.maxcut(sps.csc_matrix(g1_graph() * 1.2))
        else:                            # C = L / 4: off-diagonal -0.25, next to the low-rank constraint 11'
            C, As, bs = P.minimum_bisection(P.erdos_renyi(120, 0.08, 11))
        _DATA[which] = sp.SDPData(C, As, bs)
    return _DATA[which]


@pytest.fixture
def handles(gpu_handle_factory):
    made = []

    def make(config, **opts):
        h = gpu_handle_factory(config)
        for k, v in opts.items():
            h.set_option(k, v)
        made.append(h)
        return h
    yield make
    for h in made:
        h.close()


def _run(sp, h, data, r, steps=2):
    """f/g, then `steps` free-running iterations; everything the line search and the step produce, per iteration"""
    L = sp._lib
    rng = np.random.default_rng(100 + r)
    R0 = 2.0 * rng.random((data.n, r)) - 1.0
    e = sp.B200Engine(data, handle=h)
    e.init_vars(r, R0, np.zeros(data.m), 2.0, 4)
    out = [np.asarray(e.fg(), float)]
    for _ in range(steps):
        d = e.lbfgs_dir()
        if not d < 0:
            e.use_gradient_direction()
        bq = np.asarray(e.linesearch_coeffs(), float)
        out += [bq, h.download_mat(L.MAT_CD), h.download_vec(L.VEC_A_RD, data.m + 1), h.download_vec(L.VEC_A_DD, data.m + 1)]
        alpha, _ = sp.pick_alpha(bq, 1.0)
        out.append(np.asarray(e.step_g(alpha), float))
        e.lbfgs_update(alpha)
    out += [e.get_R(), e.get_G(), h.download_mat(L.MAT_CR)]
    return out


@pytest.mark.parametrize("r", RANKS)
@pytest.mark.parametrize("which,config,v", [("g1", "default", 0.25), ("powerlaw", "default", 0.25), ("powerlaw", "relabel", 0.25),
                                            ("bisection", "default", -0.25)])
def test_value_free_pass_gives_the_same_bits(sp, handles, which, config, v, r):
    data = _data(sp, which)
    on, off = handles(config), handles(config, obj_value_free=0)
    got = _run(sp, on, data, r)
    ref = _run(sp, off, data, r)
    assert on.value_free_weight() == v and off.value_free_weight() == 0.0
    for k, (a, b) in enumerate(zip(got, ref)):
        assert np.array_equal(a, b), f"output {k} differs: max |diff| {np.max(np.abs(a - b)):.3e}"


@pytest.mark.parametrize("which", ["weighted", "uniform_0.3"])
def test_value_free_pass_stays_off(sp, handles, which):
    h = handles("default")
    sp.B200Engine(_data(sp, which), handle=h)
    assert h.value_free_weight() == 0.0
