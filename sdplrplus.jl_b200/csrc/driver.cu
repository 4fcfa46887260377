// driver.cu -- native host driver: the outer augmented-Lagrangian loop of the reference behind one ABI call.
//
// Reference: _sdplr (src/sdplr.jl:140-449): tolerance schedule, inner L-BFGS loop with the exact line search
// (src/linesearch.jl:58-112: root selection on the derivative cubic) or the Armijo backtracking for inequality
// problems (src/linesearch.jl:139-191), the dual-bound / suboptimality logic (src/sdplr.jl:300-356), the dual and
// penalty updates (:358-371), the dynamic rank update (rank_update!, src/coreop.jl:518-526; barvinok_pataki,
// src/utils.jl:7-11) and the final DIMACS errors (:419-425).
//
// north_star keeps this control plane in Julia (julia/SDPLRPlusB200.jl drives the fused entry points one by one).
// SURVEY.md 8f/f1 promotes it to a supported native driver so that hosts without the Julia loop (the bench, C/C++ and
// Python callers) pay no per-iteration interpreter overhead: the loop below is the same sequence of ABI calls
// (sdplrp_lbfgs_dir -> sdplrp_linesearch_coeffs -> sdplrp_step_g -> sdplrp_lbfgs_update) and nothing else.
// Random numbers (the start vectors of the eigenvalue iterations, the fresh R of a rank update) come from the
// counter-based device generator, seeded from config.seed; R0 / lambda0 may be injected by the caller.
#include <math.h>
#include <stdio.h>
#include <algorithm>
#include <chrono>
#include <vector>
#include "common.cuh"

extern "C" {   // internal entry points of api.cu (not part of the public header)
int32_t api_lbfgs_dir_async(sdplrp_handle *h);
int32_t api_linesearch_coeffs_descent(sdplrp_handle *h, double bq[5], double *descent);
}

namespace {

constexpr double kEps = 2.220446049250313e-16;

double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

unsigned long long mix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

double horner(const double *c, int deg, double x) {
    double v = c[deg];
    for (int k = deg - 1; k >= 0; k--) v = v * x + c[k];
    return v;
}

// g(x) = c0 + c1 x + c2 x^2 + c3 x^3 in extended precision
long double cubic_eval(const double *c, long double x) { return ((c[3] * x + c[2]) * x + c[1]) * x + c[0]; }

// the real roots of g in [0, A], by monotone pieces: the critical points of g (roots of g', stable quadratic formula)
// cut [0, A] into intervals on which g is monotone; a sign change on a piece brackets exactly one root, which is
// located by bisection to the last bit.  Independent of the scaling of the coefficients (a nearly vanishing leading
// coefficient just moves a critical point out of the interval).  Stands in for PolynomialRoots.roots followed by the
// filter "real and in [0, alpha_max]" of src/linesearch.jl:82-106; roots of even multiplicity (tangency, no sign
// change) are inflection points of the quartic, never its strict minimiser, so skipping them cannot change the choice.
int cubic_roots_in(const double *c, double A, double *out) {
    double cuts[4];
    int nc = 0;
    cuts[nc++] = 0.0;
    const double qa = 3.0 * c[3], qb = 2.0 * c[2], qc = c[1];  // g'(x) = qa x^2 + qb x + qc
    double cp[2];
    int ncp = 0;
    if (qa != 0.0) {
        const double disc = qb * qb - 4.0 * qa * qc;
        if (disc > 0.0) {
            const double t = -0.5 * (qb + (qb >= 0.0 ? 1.0 : -1.0) * sqrt(disc));
            cp[ncp++] = t / qa;
            if (t != 0.0) cp[ncp++] = qc / t;
        }
    } else if (qb != 0.0) {
        cp[ncp++] = -qc / qb;
    }
    if (ncp == 2 && cp[0] > cp[1]) std::swap(cp[0], cp[1]);
    for (int k = 0; k < ncp; k++)
        if (cp[k] > 0.0 && cp[k] < A && std::isfinite(cp[k])) cuts[nc++] = cp[k];
    cuts[nc++] = A;
    int nr = 0;
    for (int k = 0; k + 1 < nc; k++) {
        long double lo = cuts[k], hi = cuts[k + 1];
        long double flo = cubic_eval(c, lo), fhi = cubic_eval(c, hi);
        if (flo == 0.0L) { if (nr == 0 || out[nr - 1] != (double)lo) out[nr++] = (double)lo; continue; }
        if (fhi == 0.0L) { out[nr++] = (double)hi; continue; }
        if ((flo < 0.0L) == (fhi < 0.0L)) continue;
        for (int it = 0; it < 200; it++) {
            const long double mid = 0.5L * (lo + hi);
            if (mid <= lo || mid >= hi) break;
            const long double fm = cubic_eval(c, mid);
            if (fm == 0.0L) { lo = hi = mid; break; }
            if ((fm < 0.0L) == (flo < 0.0L)) { lo = mid; flo = fm; } else { hi = mid; }
        }
        out[nr++] = (double)(0.5L * (lo + hi));
    }
    return nr;
}

// root selection of linesearch! (src/linesearch.jl:58-112); returns SDPLRP_ERR_LINESEARCH for cubic[1] > eps
int32_t pick_alpha(const double bq[5], double alpha_max, double *alpha_star, double *f_star) {
    double cubic[4] = {bq[1], 2.0 * bq[2], 3.0 * bq[3], 4.0 * bq[4]};
    if (cubic[0] > kEps) return SDPLRP_ERR_LINESEARCH;
    if (fabs(cubic[3]) < kEps) cubic[3] = 0.0;  // "got a quadratic function" (:70-83)
    double roots[5];
    int nr = cubic_roots_in(cubic, alpha_max, roots);
    roots[nr++] = alpha_max;
    double a_best = 0.0, f_best = bq[0];
    for (int i = 0; i < nr; i++) {
        const double x = roots[i];
        if (!(x >= 0.0) || x > alpha_max || !std::isfinite(x)) continue;
        const double fx = horner(bq, 4, x);
        if (fx < f_best) { f_best = fx; a_best = x; }
    }
    *alpha_star = a_best;
    *f_star = f_best;
    return SDPLRP_OK;
}

// R[i, :] = 2u - 1, u ~ U[0,1) from a counter-based hash of (seed, reference vertex, column): identical for every
// rank count and vertex relabeling
__global__ void k_fill_uniform(i64 n, int r, unsigned long long seed, const int *__restrict__ iperm, double *__restrict__ X) {
    const i64 total = n * r;
    for (i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x; e < total; e += (i64)gridDim.x * blockDim.x) {
        const i64 i = e / r, c = e - i * r;
        const unsigned long long v = (unsigned long long)(iperm ? iperm[i] : i);
        unsigned long long x = seed ^ (v * (unsigned long long)r + (unsigned long long)c) * 0xD6E8FEB86659FD93ull;
        x += 0x9E3779B97F4A7C15ull;
        x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
        x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
        x ^= x >> 31;
        X[e] = 2.0 * ((double)(x >> 11) * (1.0 / 9007199254740992.0)) - 1.0;
    }
}

struct Driver {
    sdplrp_handle *h;
    const sdplrp_config &cfg;
    unsigned long long seed_ctr = 0;
    unsigned long long next_seed() { return mix64((unsigned long long)cfg.seed + 0x632BE59BD9B4E019ull * (++seed_ctr)); }
};

// both ranks of a multi-GPU run must take the same time-based decisions: 1 if ANY rank says so
int32_t agree(sdplrp_handle *h, bool mine, bool *all) {
    if (h->world <= 1) { *all = mine; return SDPLRP_OK; }
    h->hscal[SC_LANCZOS + 11] = mine ? 1.0 : 0.0;
    CUDA_TRY(h, cudaMemcpyAsync(h->dscal + SC_LANCZOS + 11, h->hscal + SC_LANCZOS + 11, sizeof(double), cudaMemcpyHostToDevice, h->stream));
    SDP_CHECK(comm_reduce_scalars(h, SC_LANCZOS + 11, 1));
    SDP_CHECK(fetch_scalars(h, SC_LANCZOS + 11, 1));
    *all = h->hscal[SC_LANCZOS + 11] != 0.0;
    return SDPLRP_OK;
}

void print_row(const sdplrp_config &cfg, i64 T, i64 localiter, i64 it, double L, double obj, double sigma, double gtol, double ptol,
               double gn, double pn, double gap, double dual) {
    printf("T=%lld iter_T=%lld tot=%lld L=%.6e pobj=%.6e sigma=%g eta=%.2e omega=%.2e |grad|=%.3e |pinf|=%.3e gap=%.3e dobj=%.6e\n",
           (long long)T, (long long)localiter, (long long)it, L, obj, sigma, ptol, gtol, gn, pn, gap, dual);
    fflush(stdout);
}

// one pass of the inner loop body of _sdplr (src/sdplr.jl:194-236): L-BFGS direction, descent test with the gradient
// fallback, line search (exact quartic, or Armijo backtracking for inequality problems), step + gradient + norms.
// L_val <- the line search's AL value, alpha <- the step, sg <- {obj, ||G||^2, ||pvio||^2}.
int32_t inner_iteration(sdplrp_handle *h, bool use_armijo, double alpha_max, double *L_val, double *alpha_out, double sg[3]) {
    // The descent test (src/sdplr.jl:201-205) is taken SPECULATIVELY: the line-search pass is enqueued for the L-BFGS direction
    // right away and `descent` comes back in the same host round trip as the five coefficients; only when the direction turns
    // out not to be a descent direction (rare) the pass is redone for the gradient direction.  One synchronisation less per
    // iteration, same decisions and results.
    double descent = 0.0, alpha = 0.0, bq[5];
    SDP_CHECK(api_lbfgs_dir_async(h));
    SDP_CHECK(api_linesearch_coeffs_descent(h, bq, &descent));
    if (std::isnan(descent) || descent >= 0.0) {
        SDP_CHECK(sdplrp_use_gradient_direction(h));
        SDP_CHECK(sdplrp_linesearch_coeffs(h, bq));
    }
    if (!use_armijo) {
        if (pick_alpha(bq, alpha_max, &alpha, L_val) != SDPLRP_OK)
            return fail(h, SDPLRP_ERR_LINESEARCH, "Error: cubic[1] = " + std::to_string(bq[1]) + " should be less than 0.");
    } else {
        // linesearch_armijo! (src/linesearch.jl:139-191): sharp AL at alpha_max / 2^k, k = 0..50, c = 1e-4
        double L0 = 0.0, slope = 0.0, zero = 0.0;
        SDP_CHECK(sdplrp_armijo_eval(h, &zero, 1, &L0, &slope));
        double alphas[51], Ls[51];
        for (int k = 0; k < 51; k++) alphas[k] = alpha_max / pow(2.0, (double)k);
        int pick = 50;
        bool found = false;
        for (int s = 0; s < 51 && !found; s += 15) {
            const int cnt = std::min(15, 51 - s);
            SDP_CHECK(sdplrp_armijo_eval(h, alphas + s, cnt, Ls + s, nullptr));
            for (int k = s; k < s + cnt; k++)
                if (Ls[k] <= L0 + 1e-4 * alphas[k] * slope) { pick = k; found = true; break; }
        }
        alpha = alphas[pick]; *L_val = Ls[pick];
    }
    SDP_CHECK(sdplrp_step_g(h, alpha, sg));
    *alpha_out = alpha;
    return SDPLRP_OK;
}

}  // namespace

extern "C" {

int32_t sdplrp_config_default(sdplrp_config *c) {
    if (!c) return SDPLRP_ERR_ARG;
    // src/options.jl:1-24
    c->ptol = 1e-2; c->gtol = 0.0; c->objtol = 1e-2; c->sigma_0 = 2.0; c->sigmafac = 2.0; c->maxtime = 3600.0;
    c->printfreq = 60.0; c->fprec = 1e8; c->prior_trace_bound = 1e18; c->alpha_max = 1.0;
    c->maxmajoriter = 100000; c->maxiter = 10000000; c->numlbfgsvecs = 4; c->rankupd_tol = 4; c->printlevel = 1;
    c->gtol_relative = 1; c->ptol_relative = 1; c->objtol_relative = 1; c->eval_DIMACS_errs = 0; c->eigval_highprecision = 0;
    c->seed = 0;
    return SDPLRP_OK;
}

int32_t sdplrp_pick_alpha(const double biquadratic[5], double alpha_max, double *alpha, double *value) {
    if (!biquadratic || !alpha || !value) return SDPLRP_ERR_ARG;
    return pick_alpha(biquadratic, alpha_max, alpha, value);
}

int32_t sdplrp_fill_uniform(sdplrp_handle *h, int32_t mat_id, uint64_t seed) {
    if (!h) return SDPLRP_ERR_ARG;
    if (!h->preprocessed || h->r <= 0) return fail(h, SDPLRP_ERR_STATE, "fill_uniform: call sdplrp_set_rank first");
    double *X = mat_id == SDPLRP_MAT_R ? h->R : mat_id == SDPLRP_MAT_G ? h->G : mat_id == SDPLRP_MAT_D ? h->D : nullptr;
    if (!X) return fail(h, SDPLRP_ERR_ARG, "fill_uniform: R, G or D only");
    CUDA_TRY(h, cudaSetDevice(h->device));
    k_fill_uniform<<<grid_for(h->n * h->r, 256, 8 * kNumSM), 256, 0, h->stream>>>(h->n, h->r, seed, h->relabeled ? h->iperm : nullptr, X);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    comm_mark_full(h, mat_id);
    if (mat_id == SDPLRP_MAT_R) { h->CR_valid = false; h->ls_valid = false; }
    if (mat_id == SDPLRP_MAT_D) { h->CD_valid = false; h->ls_valid = false; }
    if (mat_id == SDPLRP_MAT_G) h->gram_g_valid = false;
    return SDPLRP_OK;
}

int32_t sdplrp_iterate(sdplrp_handle *h, int64_t k, double alpha_max, int32_t use_armijo, int32_t update_history, double out[5]) {
    if (!h) return SDPLRP_ERR_ARG;
    if (!h->preprocessed || h->r <= 0) return fail(h, SDPLRP_ERR_STATE, "iterate: no problem / rank set");
    if (k < 0 || !out) return fail(h, SDPLRP_ERR_ARG, "iterate: bad argument");
    double L_val = 0.0, alpha = 0.0, sg[3] = {0.0, 0.0, 0.0};
    for (int64_t i = 0; i < k; i++) {
        SDP_CHECK(inner_iteration(h, use_armijo != 0, alpha_max, &L_val, &alpha, sg));
        if (update_history && h->hist > 0) SDP_CHECK(sdplrp_lbfgs_update(h, alpha));
    }
    out[0] = L_val; out[1] = sg[0]; out[2] = sg[1]; out[3] = sg[2]; out[4] = alpha;
    return SDPLRP_OK;
}

int32_t sdplrp_solve(sdplrp_handle *h, const sdplrp_config *cfgp, int64_t r0, const double *Rt0, const double *lambda0, double normb,
                     double normC, sdplrp_result *res, double *best_lambda) {
    if (!h) return SDPLRP_ERR_ARG;
    if (!h->preprocessed) return fail(h, SDPLRP_ERR_STATE, "solve: sdplrp_preprocess / sdplrp_set_problem first");
    if (!cfgp || !res || r0 < 1) return fail(h, SDPLRP_ERR_ARG, "solve: bad argument");
    if (!rank_supported(r0)) return fail(h, SDPLRP_ERR_ARG, "solve: initial rank " + std::to_string(r0) + " is not supported (see sdplrp_set_rank)");
    const sdplrp_config &cfg = *cfgp;
    Driver drv{h, cfg};
    const i64 n = h->n, m = h->m;
    const double t_start = now_s();
    double lastprint = t_start, dual_time = 0.0;
    const int hist = (int)cfg.numlbfgsvecs;

    // SolverVars(data, r, config) (src/structs.jl:225-240): injected point, or R ~ U(-1,1), lambda = 0
    auto init_point = [&](i64 r, const double *R_in, const double *lam_in) -> int32_t {
        SDP_CHECK(sdplrp_set_rank(h, (int32_t)r, hist));
        if (R_in) SDP_CHECK(sdplrp_upload_mat(h, SDPLRP_MAT_R, R_in));
        else SDP_CHECK(sdplrp_fill_uniform(h, SDPLRP_MAT_R, drv.next_seed()));
        std::vector<double> lam((size_t)std::max<i64>(m, 1), 0.0);
        if (lam_in) for (i64 i = 0; i < m; i++) lam[(size_t)i] = lam_in[i];
        if (h->has_ineq) {  // lambda <- min(lambda, lambda_ub) (src/structs.jl:248-249)
            std::vector<double> ub((size_t)std::max<i64>(m, 1));
            SDP_CHECK(sdplrp_download_vec(h, SDPLRP_VEC_LAMBDA_UB, ub.data(), m));
            for (i64 i = 0; i < m; i++) lam[(size_t)i] = std::min(lam[(size_t)i], ub[(size_t)i]);
        }
        SDP_CHECK(sdplrp_upload_vec(h, SDPLRP_VEC_LAMBDA, lam.data(), m));
        return sdplrp_set_sigma(h, cfg.sigma_0);
    };
    i64 r = r0;
    SDP_CHECK(init_point(r, Rt0, lambda0));

    const double gscale = cfg.gtol_relative ? normC : 1.0, pscale = cfg.ptol_relative ? normb : 1.0;
    double sigma = h->sigma;
    double cur_gtol = std::max(1.0 / sigma, cfg.gtol), cur_ptol = std::max(1.0 / pow(sigma, 0.1), cfg.ptol);
    double fg[4];
    SDP_CHECK(sdplrp_fg(h, fg));
    double L_val = fg[0], obj = fg[1], grad_norm = sqrt(fg[2]) / gscale, pvio_norm = sqrt(fg[3]) / pscale;

    i64 it = 0, majoriter = 0, lanczos_steps = 0;
    const bool use_armijo = h->has_ineq;
    i64 rankupd_cnt = cfg.rankupd_tol;
    double duality_gap = 1e20, min_gap = 1e20, max_dual = -1e20;
    if (best_lambda) {  // best_lambda starts as lambda0 (src/sdplr.jl:183); slot m+1 is filled once a dual bound exists (:325)
        SDP_CHECK(sdplrp_download_vec(h, SDPLRP_VEC_LAMBDA, best_lambda, m));
        best_lambda[m] = 0.0;
    }
    std::vector<double> ybuf;
    bool stop = false, out_of_budget = false;

    for (i64 major = 0; major < cfg.maxmajoriter; major++) {
        majoriter++;
        i64 localiter = 0;
        while (grad_norm > cur_gtol) {
            localiter++; it++;
            const double lastval = L_val;
            double alpha = 0.0, sg[3];
            SDP_CHECK(inner_iteration(h, use_armijo, cfg.alpha_max, &L_val, &alpha, sg));
            obj = sg[0]; grad_norm = sqrt(sg[1]) / gscale; pvio_norm = sqrt(sg[2]) / pscale;
            const double rel_delta = (lastval - L_val) / std::max(1.0, std::max(fabs(L_val), fabs(lastval)));
            if (rel_delta < cfg.fprec * kEps) break;  // src/sdplr.jl:238-241
            if (hist > 0) SDP_CHECK(sdplrp_lbfgs_update(h, alpha));
            // the iteration budget is the same number on every rank: tested every iteration, as the reference does
            // (src/sdplr.jl:271-276).  Only the WALL-CLOCK decision needs an agreement among the ranks (an all-reduce),
            // which is taken every 16th iteration when there are several.
            if (it > cfg.maxiter) { out_of_budget = true; break; }
            if ((it & 15) == 0 || h->world <= 1) {
                const double now = now_s();
                if (now - lastprint >= cfg.printfreq) {
                    lastprint = now;
                    if (cfg.printlevel > 0 && h->rank == 0)
                        print_row(cfg, majoriter, localiter, it, L_val, obj, h->sigma, cur_gtol, cur_ptol, grad_norm, pvio_norm, min_gap, max_dual);
                }
                bool over = false;
                SDP_CHECK(agree(h, now - t_start > cfg.maxtime, &over));
                if (over) { out_of_budget = true; break; }
            }
        }
        if (cfg.printlevel > 0 && h->rank == 0)
            print_row(cfg, majoriter, localiter, it, L_val, obj, h->sigma, cur_gtol, cur_ptol, grad_norm, pvio_norm, min_gap, max_dual);
        lastprint = now_s();
        {
            bool over = false;
            SDP_CHECK(agree(h, out_of_budget || lastprint - t_start > cfg.maxtime || it > cfg.maxiter, &over));
            if (over) break;
        }

        bool rank_double = false;
        sigma = h->sigma;
        if (pvio_norm <= cur_ptol) {
            const double t0 = now_s();
            double dual_value = 0.0, mineig = 0.0;
            int64_t steps = 0;
            if (cfg.eigval_highprecision) SDP_CHECK(sdplrp_dual_obj_highprecision(h, cfg.prior_trace_bound, nullptr, drv.next_seed(), &dual_value, &mineig, &steps));
            else SDP_CHECK(sdplrp_dual_obj(h, cfg.prior_trace_bound, it, nullptr, drv.next_seed(), &dual_value, &mineig, &steps));
            lanczos_steps += steps;
            if (dual_value > max_dual) {
                if (best_lambda) {  // best_lambda = -y (src/sdplr.jl:325)
                    SDP_CHECK(sdplrp_download_vec(h, SDPLRP_VEC_Y, best_lambda, m + 1));
                    for (i64 i = 0; i <= m; i++) best_lambda[i] = -best_lambda[i];
                }
                max_dual = dual_value;
            }
            duality_gap = cfg.objtol_relative ? (obj - max_dual) / std::min(fabs(obj), fabs(max_dual)) : obj - max_dual;
            dual_time += now_s() - t0;
            if (pvio_norm <= cfg.ptol) {
                if (std::isinf(cfg.objtol) && cfg.objtol > 0) stop = true;
                else if (duality_gap <= cfg.objtol) { min_gap = std::min(min_gap, duality_gap); stop = true; }
                else {
                    if (min_gap - duality_gap < cfg.objtol) rankupd_cnt--;
                    else rankupd_cnt = cfg.rankupd_tol;
                    min_gap = std::min(min_gap, duality_gap);
                    if (rankupd_cnt == 0) rank_double = true;
                }
            }
            if (stop) break;
            SDP_CHECK(sdplrp_dual_update(h));
            cur_ptol = cur_ptol / pow(sigma, 0.9);
            cur_gtol = cur_gtol / sigma;
        } else {
            sigma *= cfg.sigmafac;
            SDP_CHECK(sdplrp_set_sigma(h, sigma));
            cur_ptol = 1.0 / pow(sigma, 0.1);
            cur_gtol = 1.0 / sigma;
        }

        if (rank_double) {
            // rank_update! (src/coreop.jl:518-526): brand-new random variables, r <- min(barvinok_pataki, 2r), sigma <- sigma_0;
            // r is clamped to the supported ranks (<= 256, odd <= 128), and may stay the same
            const i64 bp = std::min<i64>(n, (i64)floor(sqrt(2.0 * (double)m) + 1.0));
            r = rank_after_update(bp, r);
            SDP_CHECK(init_point(r, nullptr, nullptr));
            sigma = cfg.sigma_0;
            cur_ptol = 1.0 / pow(sigma, 0.1);
            cur_gtol = 1.0 / sigma;
            min_gap = 1e20; max_dual = -1e20; rankupd_cnt = cfg.rankupd_tol;
        } else {
            SDP_CHECK(sdplrp_lbfgs_clear(h));
        }
        cur_ptol = std::max(cur_ptol, cfg.ptol);
        cur_gtol = std::max(cur_gtol, cfg.gtol);
        SDP_CHECK(sdplrp_fg(h, fg));
        L_val = fg[0]; obj = fg[1]; grad_norm = sqrt(fg[2]) / gscale; pvio_norm = sqrt(fg[3]) / pscale;
    }

    SDP_CHECK(sdplrp_fg(h, fg));
    L_val = fg[0]; obj = fg[1]; grad_norm = sqrt(fg[2]) / gscale; pvio_norm = sqrt(fg[3]) / pscale;
    const double t_end = now_s();
    res->sigma = h->sigma; res->grad_norm = grad_norm; res->primal_vio = pvio_norm; res->obj = obj; res->L = L_val;
    res->max_dual_value = max_dual; res->min_duality_gap = min_gap;
    res->totaltime = t_end - t_start; res->dual_time = dual_time; res->primaltime = res->totaltime - dual_time;
    res->iter = it; res->majoriter = majoriter; res->lanczos_steps = lanczos_steps; res->r = r;
    res->status = stop ? 0 : 1;
    for (int k = 0; k < 6; k++) res->DIMACS_errs[k] = 0.0;
    res->DIMACS_time = 0.0;
    if (cfg.eval_DIMACS_errs) {  // src/sdplr.jl:419-425 (not part of totaltime)
        const double t0 = now_s();
        SDP_CHECK(sdplrp_dimacs_errors(h, normb, normC, nullptr, drv.next_seed(), res->DIMACS_errs));
        res->DIMACS_time = now_s() - t0;
    }
    return SDPLRP_OK;
}

}  // extern "C"
