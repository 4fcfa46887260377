"""NumPy / SciPy restatements of the three rounding methods of csrc/rounding.cu (hyperplane, one-flip local search and
sweep rounding), which the GPU tests, the multi-GPU check and the rounding benchmark compare the device results with."""
import itertools
import math

import numpy as np
import scipy.sparse as sps

def numpy_rounding(R, G, C):
    """x_k = sign(R g_k) (ties to +1), obj_k = x_k' C x_k, sum_k; plus the candidates with a dot inside a 1e-12 relative
    margin of zero (their sign is not determined by the data)."""
    D = R @ G.T
    X = np.where(D >= 0, 1.0, -1.0)
    scale = np.linalg.norm(R, axis=1)[:, None] * np.linalg.norm(G, axis=1)[None, :]
    ambiguous = np.any(np.abs(D) <= 1e-12 * scale, axis=0) & np.any(scale > 0, axis=0)
    obj = np.einsum("ik,ik->k", X, sps.csr_matrix(C) @ X)
    return X, obj, X.sum(axis=0), ambiguous


def cut_value(A, x):
    Au = sps.triu(sps.csr_matrix(A), k=1).tocoo()
    return float(np.sum(Au.data * (x[Au.row] != x[Au.col])))


def check_exact(res, R, G, C, A=None):
    """a round_hyperplane result against numpy_rounding, bit for bit (and -cut value when the graph A is given)"""
    X, obj, tot, amb = numpy_rounding(R, G, C)
    assert not amb.any(), f"{int(amb.sum())} candidates with a row inside the tie margin"
    np.testing.assert_array_equal(res["G_used"], G)
    np.testing.assert_array_equal(res["obj"], obj)
    np.testing.assert_array_equal(res["sum"], tot)
    b = res["best"]
    assert b == int(np.argmin(obj))
    np.testing.assert_array_equal(res["best_x"], X[:, b])
    if A is not None:
        for k in range(G.shape[0]):
            assert res["obj"][k] == -cut_value(A, X[:, k])
    return X


def engine_with_R(sp, gpu_handle_factory, config, *problem_and_R):
    """an engine on SDPData(C, As, bs) (or a given SDPData) whose variables start at R"""
    *problem, R = problem_and_R
    data = problem[0] if len(problem) == 1 else sp.SDPData(*problem)
    eng = sp.B200Engine(data, handle=gpu_handle_factory(config))
    eng.init_vars(R.shape[1], R, np.zeros(data.m), 2.0, 4)
    return eng


# ---- one-flip local search ----
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


# ---- sweep rounding ----
INF = math.inf


def projections(R, G):
    """P = R G' computed once per distinct row of R, so exactly repeated rows get exactly equal projections (as on the
    device, where a row's projection depends only on the row)"""
    U, inv = np.unique(R, axis=0, return_inverse=True)
    return (U @ G.T)[inv.reshape(-1)]


def assert_order_determined(R, G, P):
    """no two vertices adjacent in a sweep order (and no vertex at 0) lie within a 1e-12 relative margin unless their rows
    of R are identical: the order and the hyperplane bits are then fixed by the data, not by the summation order"""
    scale = np.linalg.norm(R, axis=1)[:, None] * np.linalg.norm(G, axis=1)[None, :]
    _, rid = np.unique(R, axis=0, return_inverse=True)
    rid = rid.reshape(-1)
    for k in range(G.shape[0]):
        p, sc = P[:, k], scale[:, k]
        o = np.lexsort((np.arange(len(p)), p))
        gap = np.abs(np.diff(p[o]))
        close = (gap <= 1e-12 * np.maximum(sc[o][1:], sc[o][:-1])) & (rid[o][1:] != rid[o][:-1])
        assert not close.any(), f"candidate {k}: {int(close.sum())} adjacent projections inside the tie margin"
        assert not np.any((np.abs(p) <= 1e-12 * sc) & (p != 0.0)), f"candidate {k}: a projection inside the margin of 0"


def numpy_sweep(C, P, w=None, window=(-INF, INF)):
    """per candidate: order, profile f(0..n), W(S_0..n), chosen t (-1 if none feasible), x and obj of the chosen vector"""
    Cs = sps.csr_matrix(C)
    n, K = P.shape
    A = Cs.copy()
    A.setdiag(0.0)
    A.eliminate_zeros()
    coo = A.tocoo()
    rows, cols, vals = coo.row, coo.col, coo.data
    total = float(Cs.sum())
    wv = np.ones(n) if w is None else np.asarray(w, dtype=np.float64)
    out = []
    for k in range(K):
        order = np.lexsort((np.arange(n), P[:, k]))
        pos = np.empty(n, np.int64)
        pos[order] = np.arange(n)
        s = np.where(pos[cols] > pos[rows], 1.0, -1.0)          # +1: the neighbour comes after the vertex
        delta = -4.0 * np.bincount(rows, weights=vals * s, minlength=n)
        prof = total + np.concatenate([[0.0], np.cumsum(delta[order])])
        W = np.concatenate([[0.0], np.cumsum(wv[order])])
        feas = (window[0] <= W) & (W <= window[1])
        t = int(np.argmin(np.where(feas, prof, INF))) if feas.any() else -1
        x = np.ones(n)
        if t >= 0:
            x[order[:t]] = -1.0
        obj = float(x @ (Cs @ x)) if t >= 0 else INF
        out.append({"order": order, "profile": prof, "W": W, "t": t, "x": x, "obj": obj})
    return out


def exact_projection(R, g, margin=1e-10):
    """R g as the device forms it (per row: fma over the columns in order, -0.0 -> +0.0).  BLAS gives it up to rounding;
    the rows whose value lies within `margin` (relative) of a neighbour in sorted order are recomputed with that exact fma
    chain (Fraction arithmetic, correctly rounded), so the order of the host restatement is the device's."""
    from fractions import Fraction
    p = R @ g
    scale = np.linalg.norm(R, axis=1) * np.linalg.norm(g)
    o = np.argsort(p, kind="stable")
    close = np.abs(np.diff(p[o])) <= margin * np.maximum(scale[o][1:], scale[o][:-1])
    rows = np.unique(np.concatenate([o[:-1][close], o[1:][close]]))
    for i in rows:
        acc = Fraction(0)
        for c in range(R.shape[1]):
            acc = Fraction(float(Fraction(float(R[i, c])) * Fraction(float(g[c])) + acc))
        p[i] = float(acc) + 0.0
    return p
