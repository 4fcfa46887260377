"""On-disk formats (SURVEY.md 8f/f4): the SDPA / SDPLR-1.03 writers of exps/data_utils.jl:22-152 restated in
sdplrplus.jl_b200/formats.py, their readers (round trips) and the Gset reader."""
import numpy as np
import pytest
import scipy.sparse as sps

from helpers import g1_graph, k2_graph, p3_graph


@pytest.fixture(scope="module")
def F(sp):
    import importlib
    return importlib.import_module("sdplrplus.jl_b200.formats")


def test_julia_float_printing(F):
    cases = {1.0: "1.0", -0.25: "-0.25", 0.5: "0.5", 1e-5: "1.0e-5", 0.0001: "0.0001", 0.00012: "0.00012", 123456.0: "123456.0",
             1234567.0: "1.234567e6", 1e6: "1.0e6", 999999.0: "999999.0", 0.1: "0.1", 1 / 3: "0.3333333333333333", 2.5e-7: "2.5e-7",
             1e21: "1.0e21", -3.0e10: "-3.0e10", 5e-324: "5.0e-324", 0.0: "0.0", 12.5: "12.5", 0.00125: "0.00125"}
    for x, s in cases.items():
        assert F.jl_float(x) == s
    rng = np.random.default_rng(0)
    for x in np.r_[rng.standard_normal(200) * 10.0 ** rng.integers(-12, 12, 200), 1.0 / np.arange(1, 50)]:
        assert float(F.jl_float(x)) == x          # shortest digits that round-trip


def test_sdpa_writer_k2_literal(sp, F, tmp_path):
    """K2 MaxCut (test/maxcut.jl:6-10) through write_problem_sdpa: header, `0 1 i j -C_ij` over findnz(triu(C)),
    then one `k 1 i i 1.0` line per diagonal constraint (exps/data_utils.jl:33-50)."""
    C, As, bs = sp.problems.maxcut(k2_graph())
    p = tmp_path / "k2.sdpa"
    F.write_problem_sdpa(p, C, As, bs)
    assert p.read_text() == "2\n1\n2\n1.0 1.0 \n0 1 1 1 0.25\n0 1 1 2 -0.25\n0 1 2 2 0.25\n1 1 1 1 1.0\n2 1 2 2 1.0\n"
    C2, As2, bs2 = F.read_problem_sdpa(p)
    assert abs(C2 - C).max() == 0 and np.array_equal(bs2, bs)
    assert [A.toarray().tolist() for A in As2] == [[[1.0, 0.0], [0.0, 0.0]], [[0.0, 0.0], [0.0, 1.0]]]


def test_sdplr_writer_p3_lovasz_literal(sp, F, tmp_path):
    """Lovasz theta on the path P3 (SURVEY Appendix C): C is the low-rank -11' (`0 1 l 1`), two COO edge constraints in
    stored order (triu keeps the (i<j) entry) and the identity (exps/data_utils.jl:53-124)."""
    C, As, bs = sp.problems.lovasz_theta(p3_graph())
    p = tmp_path / "p3.sdplr"
    F.write_problem_sdplr(p, C, As, bs)
    want = ("3\n1\n3\n0.0 0.0 1.0 \n1\n"
            "0 1 l 1\n-1.0\n1.0\n1.0\n1.0\n"
            "1 1 s 1\n1 2 1.0\n"
            "2 1 s 1\n2 3 1.0\n"
            "3 1 s 3\n1 1 1.0\n2 2 1.0\n3 3 1.0\n")
    assert p.read_text() == want
    C2, As2, bs2 = F.read_problem_sdplr(p)
    assert isinstance(C2, sp.SymLowRankMatrix) and np.array_equal(C2.toarray(), C.toarray()) and np.array_equal(bs2, bs)
    for A, B in zip(sp.SDPData(C, As, bs).matrices(), As2):
        np.testing.assert_array_equal(A.toarray(), B.toarray())


@pytest.mark.parametrize("fam", ["maxcut", "minimum_bisection", "cutnorm", "lovasz_theta"])
def test_problem_round_trips(sp, F, tmp_path, fam):
    P = sp.problems
    G = P.erdos_renyi(40, 0.2, 7)
    if fam == "cutnorm":
        g = np.random.default_rng(1)
        G = sps.csc_matrix(g.standard_normal((20, 20)) * (g.random((20, 20)) < 0.2))
    C, As, bs = getattr(P, fam)(G)
    data = sp.SDPData(C, As, bs)
    F.write_problem_sdplr(tmp_path / "a.sdplr", C, As, bs)
    C2, As2, bs2 = F.read_problem_sdplr(tmp_path / "a.sdplr")
    np.testing.assert_array_equal(bs2, bs)
    np.testing.assert_array_equal(C2.toarray(), C.toarray())
    assert len(As2) == data.m
    for A, B in zip(data.matrices(), As2):
        np.testing.assert_array_equal(A.toarray(), B.toarray())
    if fam in ("maxcut", "cutnorm"):                      # SDPA carries sparse matrices only
        F.write_problem_sdpa(tmp_path / "a.sdpa", C, As, bs)
        C3, As3, bs3 = F.read_problem_sdpa(tmp_path / "a.sdpa")
        np.testing.assert_array_equal(C3.toarray(), C.toarray())
        for A, B in zip(data.matrices(), As3):
            np.testing.assert_array_equal(A.toarray(), B.toarray())
    else:
        with pytest.raises(TypeError):
            F.write_problem_sdpa(tmp_path / "b.sdpa", C, As, bs)


def test_problem_from_file_solves_like_the_original(sp, oracle_mod, F, tmp_path):
    C, As, bs = sp.problems.maxcut(k2_graph())
    F.write_problem_sdplr(tmp_path / "k2.sdplr", C, As, bs)
    C2, As2, bs2 = F.read_problem_sdplr(tmp_path / "k2.sdplr")
    kw = dict(engine_factory=oracle_mod.OracleEngine, printlevel=0, fprec=0.0, gtol=1e-8, objtol=1e-8, ptol=1e-8, prior_trace_bound=2.0)
    assert sp.sdplr(C2, As2, bs2, 1, **kw)["obj"] == pytest.approx(sp.sdplr(C, As, bs, 1, **kw)["obj"], rel=1e-12)


def test_initial_solution_round_trip(F, tmp_path):
    rng = np.random.default_rng(3)
    R, lam = rng.standard_normal((7, 3)), rng.standard_normal(5)
    F.write_initial_solution(tmp_path / "x.sol", R, lam)
    text = (tmp_path / "x.sol").read_text()
    assert text.startswith("dual variable 5\n") and "primal variable 1 s 7 3 3\n" in text
    assert "special lambdaupdate 0special CG 0\n" in text      # the reference's missing newline (exps/data_utils.jl:145-146)
    assert text.endswith(f"special sigma {F.jl_float(1 / 7)}\nspecial scale 1.0\n")
    R2, lam2 = F.read_initial_solution(tmp_path / "x.sol")
    np.testing.assert_array_equal(R2, R); np.testing.assert_array_equal(lam2, lam)


def test_gset_reader(F, tmp_path):
    p = tmp_path / "g.txt"
    p.write_text("4 5\n1 2 1\n2 3 -1\n3 3 5\n1 2 1\n4 1 2\n")        # duplicate edge (summed), self-loop (dropped)
    A = F.read_gset(p).toarray()
    want = np.zeros((4, 4)); want[0, 1] = want[1, 0] = 2; want[1, 2] = want[2, 1] = -1; want[3, 0] = want[0, 3] = 2
    np.testing.assert_array_equal(A, want)
    G = g1_graph()
    F.write_gset(tmp_path / "g1.txt", G)
    assert (F.read_graph(tmp_path / "g1.txt") != G).nnz == 0
