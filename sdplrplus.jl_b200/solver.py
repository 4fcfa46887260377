"""Host-side mirror of the reference's solver interface, driving the C ABI.

Reference (file:line relative to the reference checkout):
  BurerMonteiroConfig   src/options.jl:1-24
  SolverVars            src/structs.jl:194-268
  SolverAuxiliary       src/structs.jl:274-363
  f!/g!/fg!             src/coreop.jl:11-31, 305-349
  linesearch!(+armijo)  src/linesearch.jl:4-191
  lbfgs_*               src/lbfgs.jl:35-149
  dual_obj              src/coreop.jl:376-415
  sdplr / _sdplr        src/sdplr.jl:91-449

north_star keeps the outer augmented-Lagrangian loop, the L-BFGS control logic
and the rank / suboptimality logic in Julia; Julia is absent from this image,
so `_sdplr` below is the same control flow in Python, duck-typed over an
`engine` exactly like the reference is duck-typed over (data, var, aux)
(src/lowrankopt.jl:47).  The product engine is `B200Engine` (ctypes ->
libsdplrp_b200.so); tests inject the CPU oracle behind the same interface.
"""
from __future__ import annotations

import math
import time
from dataclasses import dataclass, field
from typing import Callable, Optional

import numpy as np

from . import _lib
from .types import SDPData, assemble_sparse, frobenius_norm

EPS = float(np.finfo(np.float64).eps)


@dataclass
class BurerMonteiroConfig:
    """src/options.jl:1-24 (same names; sigma for the reference's σ)."""
    ptol: float = 1e-2
    gtol: float = 0.0
    objtol: float = 1e-2
    sigma_0: float = 2.0
    sigmafac: float = 2.0
    maxtime: float = 3600.0
    printlevel: int = 1
    printfreq: float = 60.0
    numlbfgsvecs: int = 4
    maxmajoriter: int = 10 ** 5
    maxiter: int = 10 ** 7
    fprec: float = 1e8
    rankupd_tol: int = 4
    prior_trace_bound: float = 1e18
    dataset: str = ""
    eval_DIMACS_errs: bool = False
    eigval_highprecision: bool = False
    init_func: Optional[Callable] = None
    init_args: tuple = ()
    gtol_mode: str = "relative"
    ptol_mode: str = "relative"
    objtol_mode: str = "relative"
    # not in the reference: Julia's global RNG is replaced by an explicit seed
    seed: int = 0
    lanczos_host_rng: bool = True  # draw the Lanczos start vector on the host (engine-independent)
    rng_stream: str = "numpy"      # "native": eigenvalue start vectors from the device generator with the seed sequence of
                                   # the native driver (csrc/driver.cu), so that both drivers see the same random numbers
    driver: str = "python"         # "native": run the outer loop inside the library (sdplrp_solve)

    _ALIASES = {"σ_0": "sigma_0", "σfac": "sigmafac"}

    def set(self, key, value):
        key = self._ALIASES.get(key, key)
        if not hasattr(self, key) or key.startswith("_"):
            raise KeyError(f"Unrecognized keyword argument {key}")  # reference: @error and continue
        setattr(self, key, value)


_M64 = (1 << 64) - 1


def native_seed(seed, k):
    """k-th (k = 1, 2, ...) seed of the native driver's device-generator stream (csrc/driver.cu, Driver::next_seed)."""
    x = (int(seed) + 0x632BE59BD9B4E019 * int(k)) & _M64
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def barvinok_pataki(n, m):
    """src/utils.jl:7-11"""
    return min(n, int(math.floor(math.sqrt(2 * m) + 1)))


MAX_RANK = 256       # SDPLRP_MAX_RANK: the largest rank sdplrp_set_rank accepts
MAX_ODD_RANK = 128   # SDPLRP_MAX_ODD_RANK: the largest odd rank


def rank_supported(r):
    """The ranks the GPU kernels handle (include/sdplrp_b200.h, sdplrp_set_rank)."""
    return 1 <= r <= MAX_RANK and (r % 2 == 0 or r <= MAX_ODD_RANK)


def rank_after_update(bp, r):
    """rank_update! (src/coreop.jl:518-526): r <- min(bp, 2r), clamped to the largest supported rank at or below it (an odd
    rank above 128 steps down by 1).  The same rule as rank_after_update in csrc/common.cuh (the native driver)."""
    t = min(bp, 2 * r, MAX_RANK)
    return t - 1 if t % 2 == 1 and t > MAX_ODD_RANK else t


def pick_alpha(bq, alpha_max=1.0):
    """Root selection of linesearch! (src/linesearch.jl:58-112): minimise the
    quartic over the real roots of its derivative in [0, alpha_max] and alpha_max.
    numpy.roots stands in for PolynomialRoots.roots."""
    bq = np.asarray(bq, dtype=np.float64)
    cubic = np.array([bq[1], 2.0 * bq[2], 3.0 * bq[3], 4.0 * bq[4]])
    if cubic[0] > EPS:
        raise ArithmeticError(f"Error: cubic[1] = {cubic[0]} should be less than 0.")
    if abs(cubic[3]) < EPS:
        quad = cubic[:3]
        roots = np.roots(quad[::-1]) if quad[2] != 0 else (np.array([-quad[0] / quad[1]]) if quad[1] != 0 else np.array([]))
    else:
        roots = np.roots(cubic[::-1])
    cand = list(roots) + [alpha_max]
    f = np.polynomial.polynomial.polyval
    a_star, f_star = 0.0, bq[0]
    for root in cand:
        if abs(np.imag(root)) >= EPS:
            continue
        x = float(np.real(root))
        if x < 0 or x > alpha_max or not np.isfinite(x):
            continue
        fx = float(f(x, bq))
        if fx < f_star:
            f_star, a_star = fx, x
    return a_star, f_star


# ---------------------------------------------------------------------------
# engine: the hot path behind the seam
# ---------------------------------------------------------------------------
class B200Engine:
    """SolverAuxiliary + SolverVars living on the GPU (one handle)."""

    def __init__(self, data: SDPData, handle: Optional[_lib.Handle] = None, device=0, asm=None):
        """`data` needs n, m, b, constraint_types, has_inequalities (and C for the norms of
        _sdplr); `asm` may carry triplets that were assembled elsewhere (bench: on the GPU)."""
        self.data = data
        self.h = handle if handle is not None else _lib.Handle(device=device)
        t0 = time.perf_counter()
        if asm is None:
            asm = assemble_sparse(data)
        self.assemble_time = time.perf_counter() - t0
        t0 = time.perf_counter()
        dev = getattr(asm, "device_triplets", None)
        if dev is not None:   # triplets built on the GPU (problems.powerlaw_maxcut_assembled(..., keep_on_device=True)): no host round trip
            import torch
            torch.cuda.synchronize()
            self.h.preprocess_device(asm.n, asm.m, asm.mat_off, dev[0], dev[1], dev[2], asm.gids)
        else:
            self.h.preprocess(asm.n, asm.m, asm.mat_off, asm.I, asm.J, asm.V, asm.gids)
        self.preprocess_time = time.perf_counter() - t0
        for gid1, A in asm.lowrank:
            self.h.add_symlowrank(gid1, A.B, A.D)
        self.h.set_problem(data.b, data.constraint_types.astype(np.uint8) if data.has_inequalities else None)
        self.n, self.m = data.n, data.m
        trip = 0 if dev is not None else asm.I.nbytes + asm.J.nbytes + asm.V.nbytes
        self.h2d_bytes = trip + asm.mat_off.nbytes + asm.gids.nbytes + data.b.nbytes

    # state -----------------------------------------------------------------
    def init_vars(self, r, Rt0, lambda0, sigma0, numlbfgsvecs):
        """SolverVars(Rt0, lambda0, lambda_ub, r, sigma_0) + lbfgs_init."""
        self.h.set_rank(r, numlbfgsvecs)
        self.h.upload_mat_slice(_lib.MAT_R, np.ascontiguousarray(Rt0, dtype=np.float64))   # several GPUs: 1/world of the matrix per PCIe link, the rest over NVLink
        lam = np.ascontiguousarray(lambda0, dtype=np.float64)
        ct = self.data.constraint_types
        if ct is not None and np.any(ct):  # lambda_ub = 0 on inequalities (src/structs.jl:225-268); equalities: min(x, inf) = x,
            lam = np.minimum(lam, np.where(ct, 0.0, np.inf))  # so the caller's (possibly pinned) buffer is uploaded as it is
        self.h.upload_vec(_lib.VEC_LAMBDA, lam)
        self.h.sigma = sigma0
        self.r = r

    sigma = property(lambda self: self.h.sigma, lambda self, s: setattr(self.h, "sigma", s))

    def get_R(self):
        return self.h.download_mat(_lib.MAT_R)

    def get_G(self):
        return self.h.download_mat(_lib.MAT_G)

    def get_D(self):
        return self.h.download_mat(_lib.MAT_D)

    def get_lambda(self):
        return self.h.download_vec(_lib.VEC_LAMBDA, self.m)

    def get_y(self):
        return self.h.download_vec(_lib.VEC_Y, self.m + 1)

    def get_pvio_raw(self):
        return self.h.download_vec(_lib.VEC_PVIO_RAW, self.m + 1)

    def set_R(self, Rt):
        self.h.upload_mat(_lib.MAT_R, Rt)

    def set_D(self, Dt):
        self.h.upload_mat(_lib.MAT_D, Dt)

    def set_lambda(self, lam):
        self.h.upload_vec(_lib.VEC_LAMBDA, lam)

    # fused hot path ----------------------------------------------------------
    def fg(self):
        return self.h.fg()

    def f(self):
        return self.h.f()

    def g(self):
        return self.h.g()

    def lbfgs_dir(self):
        return self.h.lbfgs_dir()

    def use_gradient_direction(self):
        self.h.use_gradient_direction()

    def linesearch_coeffs(self):
        return self.h.linesearch_coeffs()

    def armijo_eval(self, alphas):
        return self.h.armijo_eval(alphas)

    def step(self, alpha):
        return self.h.step(alpha)

    def step_g(self, alpha):
        """axpy! + g! + the two norms of src/sdplr.jl:219-234 in one ABI call (fused row pass on the device)."""
        return self.h.step_g(alpha)

    def lbfgs_update(self, alpha):
        self.h.lbfgs_update(alpha)

    def lbfgs_clear(self):
        self.h.lbfgs_clear()

    def dual_obj(self, trace_bound, it, v0=None, seed=0):
        return self.h.dual_obj(trace_bound, it, v0, seed)

    def dual_obj_highprecision(self, trace_bound, v0=None, seed=0):
        """dual_obj(...; highprecision=true): SDP_S_eigval replaces the q-step Lanczos (src/coreop.jl:386-400)."""
        return self.h.dual_obj_highprecision(trace_bound, v0, seed)

    def dimacs_errors(self, normb, normC, v0=None, seed=0):
        """DIMACS_errors(data, var, aux) (src/coreop.jl:426-453)."""
        return self.h.dimacs_errors(normb, normC, v0, seed)

    def dual_update(self):
        self.h.dual_update()

    def iterate(self, k, use_armijo=False, alpha_max=1.0, update_history=True):
        """k passes of the inner loop body driven inside the library (sdplrp_iterate)."""
        return self.h.iterate(k, alpha_max, use_armijo, update_history)

    def round_hyperplane(self, K, G=None, seed=0):
        """K hyperplane roundings of the current R on the device (sdplrp_round_hyperplane); see _lib.Handle.round_hyperplane."""
        return self.h.round_hyperplane(K, G, seed)

    def round_local_search(self, K, G=None, seed=0, max_rounds=1000):
        """K hyperplane roundings refined by one-flip descent on the device (sdplrp_round_local_search); see
        _lib.Handle.round_local_search."""
        return self.h.round_local_search(K, G, seed, max_rounds)

    def close(self):
        self.h.close()


# ---------------------------------------------------------------------------
# seam-level functions with the reference's names (f!, g!, ...)
# ---------------------------------------------------------------------------
def linesearch_(engine, alpha_max=1.0):
    """linesearch!(var, aux, dirt; alpha_max) -> (alpha, L) (src/linesearch.jl:4-127)."""
    bq = engine.linesearch_coeffs()
    alpha, Lval = pick_alpha(bq, alpha_max)
    engine.step_pending = alpha
    return alpha, Lval


def linesearch_armijo_(engine, alpha_max=1.0):
    """linesearch_armijo!(...) (src/linesearch.jl:139-191): the two A passes, then
    backtracking on the sharp AL evaluated on the device for batches of step sizes."""
    engine.linesearch_coeffs()
    L0, slope = engine.armijo_eval(np.array([0.0]))
    L0 = float(L0[0])
    c = 1e-4
    alphas = alpha_max / (2.0 ** np.arange(51))
    Ls = np.empty(51)
    for s in range(0, 51, 15):
        blk = alphas[s:s + 15]
        Lb, _ = engine.armijo_eval(blk)
        Ls[s:s + blk.size] = Lb
        ok = np.nonzero(Lb <= L0 + c * blk * slope)[0]
        if ok.size:
            k = s + int(ok[0])
            return float(alphas[k]), float(Ls[k])
    return float(alphas[50]), float(Ls[50])


def _step_g(engine, alpha):
    """`axpy!(alpha, dirt, Rt); g!(var, aux)` and the two norms (src/sdplr.jl:219-234): one fused call when the
    engine offers it, the two seam calls otherwise (oracle engine)."""
    if hasattr(engine, "step_g"):
        return engine.step_g(alpha)
    obj = engine.step(alpha)
    gn2, pn2 = engine.g()
    return obj, gn2, pn2


@dataclass
class SolverStats:
    starttime: float = 0.0
    endtime: float = 0.0
    dual_time: float = 0.0
    primal_time: float = 0.0
    DIMACS_time: float = 0.0
    lanczos_steps: int = 0
    trace: list = field(default_factory=list)  # per-iteration (L, obj, gn, pn, alpha) when config asks


def _init_point(data, r, config, rng):
    """SolverVars(data, r, config) (src/structs.jl:225-240)."""
    if config.init_func is not None:
        Rt0, lam0 = config.init_func(data, r, *config.init_args)
        return np.ascontiguousarray(Rt0, dtype=np.float64), np.asarray(lam0, dtype=np.float64)
    Rt0 = 2.0 * rng.random((data.n, r)) - 1.0   # (n, r) C-order == Julia r x n column-major
    return Rt0, np.zeros(data.m)


def _sdplr(data, engine, config: BurerMonteiroConfig, stats: SolverStats, r, rng, record_trace=False):
    """_sdplr (src/sdplr.jl:140-449), line by line."""
    n, m = data.n, data.m
    stats.starttime = time.perf_counter()
    lastprint = stats.starttime

    Rt0, lam0 = _init_point(data, r, config, rng)
    engine.init_vars(r, Rt0, lam0, config.sigma_0, config.numlbfgsvecs)
    Rt0_copy, lam0_copy = Rt0.copy(), lam0.copy()

    normb = float(np.linalg.norm(data.b))
    normC = frobenius_norm(data.C)
    gscale = normC if config.gtol_mode == "relative" else 1.0
    pscale = normb if config.ptol_mode == "relative" else 1.0

    sigma = engine.sigma
    cur_gtol = max(1.0 / sigma, config.gtol)
    cur_ptol = max(1.0 / sigma ** 0.1, config.ptol)
    L_val, obj, gn2, pn2 = engine.fg()
    grad_norm, primal_vio_norm = math.sqrt(gn2) / gscale, math.sqrt(pn2) / pscale

    it = 0
    majoriter = 0
    seed_ctr = 0
    use_armijo = data.has_inequalities
    rankupd_tol_cnt = config.rankupd_tol
    duality_gap = 1e20
    min_duality_gap = 1e20
    max_dual_value = -1e20
    best_lambda = engine.get_lambda().copy()
    stop = False

    for _ in range(config.maxmajoriter):
        majoriter += 1
        localiter = 0
        while grad_norm > cur_gtol:
            localiter += 1
            it += 1
            descent = engine.lbfgs_dir()
            if math.isnan(descent) or descent >= 0:
                engine.use_gradient_direction()
            lastval = L_val
            if use_armijo:
                alpha, L_val = linesearch_armijo_(engine, 1.0)
            else:
                alpha, L_val = linesearch_(engine, 1.0)
            obj, gn2, pn2 = _step_g(engine, alpha)
            grad_norm, primal_vio_norm = math.sqrt(gn2) / gscale, math.sqrt(pn2) / pscale
            if record_trace:
                stats.trace.append((L_val, obj, grad_norm, primal_vio_norm, alpha))
            rel_delta = (lastval - L_val) / max(1.0, abs(L_val), abs(lastval))
            if rel_delta < config.fprec * EPS:
                break
            if config.numlbfgsvecs > 0:
                engine.lbfgs_update(alpha)
            now = time.perf_counter()
            if now - lastprint >= config.printfreq:
                lastprint = now
                if config.printlevel > 0:
                    _print_row(config, majoriter, localiter, it, L_val, obj, engine.sigma, cur_gtol, cur_ptol, grad_norm,
                               primal_vio_norm, min_duality_gap, max_dual_value)
            if now - stats.starttime > config.maxtime or it > config.maxiter:
                break

        now = time.perf_counter()
        if config.printlevel > 0:
            _print_row(config, majoriter, localiter, it, L_val, obj, engine.sigma, cur_gtol, cur_ptol, grad_norm,
                       primal_vio_norm, min_duality_gap, max_dual_value)
        lastprint = now
        if now - stats.starttime > config.maxtime or it > config.maxiter:
            break

        rank_double = False
        sigma = engine.sigma
        if primal_vio_norm <= cur_ptol:
            t0 = time.perf_counter()
            if config.rng_stream == "native":
                seed_ctr += 1
                v0, dev_seed = None, native_seed(config.seed, seed_ctr)
            else:
                v0 = rng.standard_normal(n) if config.lanczos_host_rng else None
                dev_seed = int(rng.integers(1 << 62))
            if config.eigval_highprecision:   # src/sdplr.jl:311-321
                dual_value, _, steps = engine.dual_obj_highprecision(config.prior_trace_bound, v0, dev_seed)
            else:
                dual_value, _, steps = engine.dual_obj(config.prior_trace_bound, it, v0, dev_seed)
            stats.lanczos_steps += int(steps)
            if dual_value > max_dual_value:
                best_lambda = -engine.get_y()
                max_dual_value = dual_value
            if config.objtol_mode == "relative":
                duality_gap = (obj - max_dual_value) / min(abs(obj), abs(max_dual_value))
            else:
                duality_gap = obj - max_dual_value
            stats.dual_time += time.perf_counter() - t0
            if primal_vio_norm <= config.ptol:
                if config.objtol == math.inf:
                    stop = True
                elif duality_gap <= config.objtol:
                    min_duality_gap = min(min_duality_gap, duality_gap)
                    stop = True
                else:
                    if min_duality_gap - duality_gap < config.objtol:
                        rankupd_tol_cnt -= 1
                    else:
                        rankupd_tol_cnt = config.rankupd_tol
                    min_duality_gap = min(min_duality_gap, duality_gap)
                    if rankupd_tol_cnt == 0:
                        rank_double = True
            if stop:
                break
            engine.dual_update()
            cur_ptol = cur_ptol / sigma ** 0.9
            cur_gtol = cur_gtol / sigma
        else:
            sigma *= config.sigmafac
            engine.sigma = sigma
            cur_ptol = 1.0 / sigma ** 0.1
            cur_gtol = 1.0 / sigma

        if rank_double:
            # rank_update! (src/coreop.jl:518-526): brand-new variables, r <- min(BP, 2r) clamped to the supported ranks, sigma <- sigma_0
            r = rank_after_update(barvinok_pataki(n, m), r)
            Rt_new, lam_new = _init_point(data, r, config, rng)
            engine.init_vars(r, Rt_new, lam_new, config.sigma_0, config.numlbfgsvecs)
            sigma = config.sigma_0
            cur_ptol = 1.0 / sigma ** 0.1
            cur_gtol = 1.0 / sigma
            min_duality_gap = 1e20
            max_dual_value = -1e20
            rankupd_tol_cnt = config.rankupd_tol
        else:
            engine.lbfgs_clear()

        cur_ptol = max(cur_ptol, config.ptol)
        cur_gtol = max(cur_gtol, config.gtol)
        L_val, obj, gn2, pn2 = engine.fg()
        grad_norm, primal_vio_norm = math.sqrt(gn2) / gscale, math.sqrt(pn2) / pscale

    L_val, obj, gn2, pn2 = engine.fg()
    grad_norm, primal_vio_norm = math.sqrt(gn2) / gscale, math.sqrt(pn2) / pscale
    stats.endtime = time.perf_counter()
    totaltime = stats.endtime - stats.starttime
    stats.primal_time = totaltime - stats.dual_time
    t0 = time.perf_counter()
    if config.eval_DIMACS_errs:   # src/sdplr.jl:419-425; not part of totaltime
        if config.rng_stream == "native":
            v0, dev_seed = None, native_seed(config.seed, seed_ctr + 1)
        else:
            v0 = rng.standard_normal(n) if config.lanczos_host_rng else None
            dev_seed = int(rng.integers(1 << 62))
        DIMACS_errs = np.asarray(engine.dimacs_errors(normb, normC, v0, dev_seed))
    else:
        DIMACS_errs = np.zeros(6)
    stats.DIMACS_time = time.perf_counter() - t0
    return {
        "Rt": engine.get_R(), "lambda": best_lambda, "Rt0": Rt0_copy, "lambda0": lam0_copy, "sigma": engine.sigma,
        "grad_norm": grad_norm, "primal_vio": primal_vio_norm, "obj": obj, "max_dual_value": max_dual_value,
        "min_duality_gap": min_duality_gap, "totaltime": totaltime, "dual_time": stats.dual_time,
        "primaltime": stats.primal_time, "iter": it, "majoriter": majoriter, "DIMACS_errs": DIMACS_errs,
        "ptol": config.ptol, "objtol": config.objtol, "fprec": config.fprec, "rankupd_tol": config.rankupd_tol,
        "r": r, "lanczos_steps": stats.lanczos_steps, "L": L_val,
    }


def _sdplr_native(data, engine, config: BurerMonteiroConfig, r, rng):
    """The same solve with the outer loop inside the library (sdplrp_solve, csrc/driver.cu); only for the GPU engine.
    Returns the reference's result dict."""
    if not isinstance(getattr(engine, "h", None), _lib.Handle):
        raise TypeError("driver='native' needs the GPU engine (sdplrp_solve runs inside libsdplrp_b200.so)")
    # R0 / lambda0 are drawn here (init_func or numpy) and uploaded, exactly as driver='python' does; the random point of a
    # rank update and the eigenvalue start vectors come from the device generator (config.seed)
    cfg = _lib.default_config()
    for k in ("ptol", "gtol", "objtol", "sigma_0", "sigmafac", "maxtime", "printfreq", "fprec", "prior_trace_bound"):
        setattr(cfg, k, float(getattr(config, k)))
    for k in ("maxmajoriter", "maxiter", "numlbfgsvecs", "rankupd_tol", "printlevel"):
        setattr(cfg, k, int(getattr(config, k)))
    cfg.gtol_relative = int(config.gtol_mode == "relative")
    cfg.ptol_relative = int(config.ptol_mode == "relative")
    cfg.objtol_relative = int(config.objtol_mode == "relative")
    cfg.eval_DIMACS_errs = int(bool(config.eval_DIMACS_errs))
    cfg.eigval_highprecision = int(bool(config.eigval_highprecision))
    cfg.seed = int(config.seed)
    Rt0, lam0 = _init_point(data, r, config, rng)
    normb = float(np.linalg.norm(data.b))
    normC = frobenius_norm(data.C)
    res, best = engine.h.solve(cfg, r, Rt0, lam0, normb, normC)
    engine.r = int(res.r)
    return {
        "Rt": engine.get_R(), "lambda": best, "Rt0": Rt0, "lambda0": lam0, "sigma": res.sigma, "grad_norm": res.grad_norm,
        "primal_vio": res.primal_vio, "obj": res.obj, "max_dual_value": res.max_dual_value,
        "min_duality_gap": res.min_duality_gap, "totaltime": res.totaltime, "dual_time": res.dual_time,
        "primaltime": res.primaltime, "iter": int(res.iter), "majoriter": int(res.majoriter),
        "DIMACS_errs": np.array(list(res.DIMACS_errs)), "ptol": config.ptol, "objtol": config.objtol, "fprec": config.fprec,
        "rankupd_tol": config.rankupd_tol, "r": int(res.r), "lanczos_steps": int(res.lanczos_steps), "L": res.L,
        "status": int(res.status),
    }


def hyperplane_rounding(ans, trials=64, seed=0, local_search_rounds=0):
    """Goemans-Williamson rounding of a solve: `trials` random hyperplanes through the factor R that `sdplr` left on the
    GPU, each cut evaluated on the device.  `ans` is the dict `sdplr` returns.  Returns {"x": the best +-1 vector (input
    vertex order), "obj": its objective <C, xx'>, "objs": every candidate's objective, "sums": every candidate's sum(x),
    "trial": the 0-based index of the best candidate}.  Only the objective and the imbalance are evaluated: constraints
    that a +-1 vector does not satisfy by construction are not checked.
    local_search_rounds > 0: every candidate is then refined by at most that many rounds of parallel one-flip descent
    on the device (sdplrp_round_local_search), and "x", "obj", "objs", "sums" describe the refined candidates; the result
    also has "objs_rounded" (before the descent), "flips" and "rounds" (per candidate; -1 = stopped by the round limit)."""
    engine = ans["engine"]
    if not hasattr(engine, "round_hyperplane"):
        raise TypeError("hyperplane_rounding needs the GPU engine (the rounding passes run inside libsdplrp_b200.so)")
    if local_search_rounds > 0:
        out = engine.round_local_search(int(trials), None, seed, int(local_search_rounds))
    else:
        out = engine.round_hyperplane(int(trials), None, seed)
    k = out["best"]
    res = {"x": out["best_x"], "obj": float(out["obj"][k]), "objs": out["obj"], "sums": out["sum"], "trial": k}
    if local_search_rounds > 0:
        res.update(objs_rounded=out["obj_round"], flips=out["flips"], rounds=out["rounds"])
    return res


def _print_row(config, T, localiter, it, L, obj, sigma, gtol, ptol, gn, pn, gap, dual):
    print(f"[{config.dataset}] T={T} iter_T={localiter} tot={it} L={L:.6e} pobj={obj:.6e} sigma={sigma:g} "
          f"eta={ptol:.2e} omega={gtol:.2e} |grad|={gn:.3e} |pinf|={pn:.3e} gap={gap:.3e} dobj={dual:.6e}", flush=True)


def sdplr(C, As, b, r, constraint_types=None, config: Optional[BurerMonteiroConfig] = None, engine_factory=None,
          record_trace=False, **kwargs):
    """sdplr(C, As, b, r; kwargs...) (src/sdplr.jl:91-138).  Returns the
    reference's result dict.  `engine_factory(data)` is a test hook; the default
    builds the GPU engine (and raises if there is no CUDA device)."""
    config = config if config is not None else BurerMonteiroConfig()
    for k, v in kwargs.items():
        config.set(k, v)
    t0 = time.perf_counter()
    data = SDPData(C, As, np.asarray(b, dtype=np.float64), constraint_types)
    engine = (engine_factory or B200Engine)(data)
    stats = SolverStats()
    preprocess_dt = time.perf_counter() - t0
    rng = np.random.default_rng(config.seed)
    if config.driver == "native":
        ans = _sdplr_native(data, engine, config, int(r), rng)
    else:
        ans = _sdplr(data, engine, config, stats, int(r), rng, record_trace=record_trace)
    ans["preprocess_time"] = preprocess_dt
    ans["totaltime"] += preprocess_dt
    if record_trace:
        ans["trace"] = stats.trace
    ans["engine"] = engine
    return ans


# ---------------------------------------------------------------------------
# the LowRankOpt `sub_solver` hook (src/lowrankopt.jl:4-53)
# ---------------------------------------------------------------------------
@dataclass
class GenericExecutionStats:
    """What SolverCore.solve! fills (src/lowrankopt.jl:47-52)."""
    status: str = "unknown"
    solution: Optional[np.ndarray] = None      # flat var.Rt (r x n column-major = C-order (n, r) raveled)
    multipliers: Optional[np.ndarray] = None   # var.lambda
    elapsed_time: float = 0.0
    objective: float = float("nan")
    solver_specific: dict = field(default_factory=dict)


class Solver:
    """`SDPLRPlus.Solver(src; config, kwargs...)` + `SolverCore.solve!(solver, model, stats; kwargs...)`.

    The reference's hook passes the LowRankOpt model itself as `data` and `aux` and lets NLPModels evaluate the operators
    (src/lowrankopt.jl:47, 80-135).  For the B200 path the model is read ONCE -- C = `LRO.grad(model, MatrixIndex(1))`,
    b = `LRO.cons_constant`, the constraint matrices, `model.dim.ranks[]` (SURVEY.md 8b) -- and routed into the same device
    engine as `sdplr`.  `src` here is any object with `C`, `As`, `b`, `rank` (and optionally `constraint_types`): the
    contents of such a model.  As in the reference: unknown keywords are reported and skipped, the start point is a flat
    vector `2*rand(n*r) - 1` with `lambda0 = randn(ncon)` (src/lowrankopt.jl:72-78), `status` is always `first_order`."""

    def __init__(self, src, config: Optional[BurerMonteiroConfig] = None, engine_factory=None, **kwargs):
        self.config = config if config is not None else BurerMonteiroConfig()
        self._apply(kwargs, "error")
        self.data = SDPData(src.C, src.As, np.asarray(src.b, dtype=np.float64), getattr(src, "constraint_types", None))
        self.r = int(src.rank)
        self.rng = np.random.default_rng(self.config.seed)
        self.Rt0 = 2.0 * self.rng.random(self.data.n * self.r) - 1.0      # flat, as SolverVars(::LRO model, r) draws it
        self.lambda0 = self.rng.standard_normal(self.data.m)
        self.engine = (engine_factory or B200Engine)(self.data)
        self.stats = SolverStats()

    def _apply(self, kwargs, level):
        for k, v in kwargs.items():
            try:
                self.config.set(k, v)
            except KeyError:
                print(f"[{level}] Unrecognized keyword argument {k}")  # @error / @warn and continue (src/lowrankopt.jl:15-21, 39-45)

    def solve(self, model=None, stats: Optional[GenericExecutionStats] = None, **kwargs):
        self._apply(kwargs, "warn")
        stats = stats if stats is not None else GenericExecutionStats()
        cfg = self.config
        keep = (cfg.init_func, cfg.init_args)
        def start_point(data, r):
            if r == self.r:
                return self.Rt0.reshape(data.n, r), self.lambda0
            # rank_update! builds brand-new random variables (src/coreop.jl:518-526)
            return 2.0 * self.rng.random((data.n, r)) - 1.0, self.rng.standard_normal(data.m)
        cfg.init_func = start_point
        cfg.init_args = ()
        try:
            ans = _sdplr(self.data, self.engine, cfg, self.stats, self.r, self.rng)
        finally:
            cfg.init_func, cfg.init_args = keep
        stats.status = "first_order"                                   # TODO of the reference: the actual status
        stats.solution = np.ascontiguousarray(ans["Rt"]).reshape(-1)
        stats.multipliers = np.asarray(self.engine.get_lambda())
        stats.elapsed_time = ans["totaltime"]
        stats.objective = ans["obj"]
        stats.solver_specific = {k: ans[k] for k in ("iter", "majoriter", "max_dual_value", "min_duality_gap", "primal_vio", "r")}
        return stats


def run_inner_iterations(engine, k, use_armijo=False, alpha_max=1.0, update_history=True, native=False):
    """k passes of the hot loop body of _sdplr (src/sdplr.jl:190-246) without the tolerance
    logic: direction, descent test, line search, step, gradient, L-BFGS update.  Used by
    bench.py and the trajectory tests.  Returns the last (L, obj, gnorm2, pnorm2, alpha).  native=True runs the same
    sequence of entry points inside the library (sdplrp_iterate) when the engine offers it."""
    if native and hasattr(engine, "iterate"):
        return engine.iterate(k, use_armijo, alpha_max, update_history)
    out = None
    for _ in range(k):
        descent = engine.lbfgs_dir()
        if math.isnan(descent) or descent >= 0:
            engine.use_gradient_direction()
        if use_armijo:
            alpha, L_val = linesearch_armijo_(engine, alpha_max)
        else:
            alpha, L_val = linesearch_(engine, alpha_max)
        obj, gn2, pn2 = _step_g(engine, alpha)
        if update_history:
            engine.lbfgs_update(alpha)
        out = (L_val, obj, gn2, pn2, alpha)
    return out
