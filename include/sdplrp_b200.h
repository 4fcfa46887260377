/*
 * sdplrp_b200.h -- C ABI of the B200-native SDPLRPlus hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b): the entry points a Julia
 * `ccall` shim binds to replace the reference's operator seam
 *   A!(out,aux,Ut) / A!(out,aux,Ut,Vt)         src/coreop.jl:36-70
 *   At_preprocess!(var,aux)                    src/coreop.jl:248-258
 *   At!(Y,X,aux,var) / At!(y,aux,x,var)        src/coreop.jl:260-300
 *   f! / g! / fg!                              src/coreop.jl:11-31,305-349
 *   linesearch! / linesearch_armijo!           src/linesearch.jl:4-191
 *   lbfgs_dir! / lbfgs_update! / lbfgs_clear!  src/lbfgs.jl:52-149
 *   approx_mineigval_lanczos / dual_obj        src/coreop.jl:376-415,461-514
 *   SDP_S_eigval / DIMACS_errors               src/coreop.jl:351-374,417-453
 *   preprocess_sparsecons / SolverAuxiliary    src/preprocess.jl:24-169, src/structs.jl:296-361
 * (file:line relative to the reference checkout).
 *
 * Conventions
 *  - plain C: pointers and sizes only; no torch / C++ types.
 *  - every function returns an int32 status: 0 = OK, <0 = error (enum below);
 *    sdplrp_last_error(h) gives the message.  Nothing throws or calls back.
 *  - all host pointers are caller-owned and only touched during the call; all
 *    device memory is owned by the handle.
 *  - index arrays crossing the ABI are Julia-style 1-based int64; reals are
 *    IEEE double.  "Rt" matrices are r x n column-major (Julia), which is the
 *    n x r row-major layout kept in HBM.
 *  - one handle drives one GPU.  Multi-GPU = one handle per process/rank
 *    (world > 1), NCCL communicator bootstrapped from an id made by rank 0.
 *  - calls enqueue on the handle's stream and synchronise only when they
 *    return host scalars or fill host buffers.
 */
#ifndef SDPLRP_B200_H
#define SDPLRP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sdplrp_handle sdplrp_handle;

enum {
    SDPLRP_OK = 0,
    SDPLRP_ERR_CUDA = -1,        /* CUDA runtime error (message has the call) */
    SDPLRP_ERR_ARG = -2,         /* bad argument / index out of range */
    SDPLRP_ERR_STATE = -3,       /* call order violated (e.g. no preprocess yet) */
    SDPLRP_ERR_ASYMMETRIC = -4,  /* lower entry with no upper mirror (src/preprocess.jl:138-158) */
    SDPLRP_ERR_NCCL = -5,
    SDPLRP_ERR_NO_DEVICE = -6,   /* no CUDA device: there is no CPU fallback */
    SDPLRP_ERR_LINESEARCH = -7   /* cubic[1] > eps (src/linesearch.jl:60-62) */
};

/* dense device matrices (n x r), addressed by id */
enum {
    SDPLRP_MAT_R = 0,   /* var.Rt */
    SDPLRP_MAT_G = 1,   /* var.Gt */
    SDPLRP_MAT_D = 2,   /* dirt   */
    SDPLRP_MAT_W0 = 3,  /* scratch (operator tests) */
    SDPLRP_MAT_W1 = 4,
    SDPLRP_MAT_CR = 5,  /* introspection (download only): C*R as kept by the recurrence CR += alpha*CD, and CD = C*dirt */
    SDPLRP_MAT_CD = 6,
    SDPLRP_MAT_S0 = 16, /* L-BFGS s_j = S0 + j, j in [0,h) (0-based slot) */
    SDPLRP_MAT_Y0 = 48  /* L-BFGS y_j = Y0 + j */
};

/* device vectors, addressed by id (length in parentheses) */
enum {
    SDPLRP_VEC_LAMBDA = 0,     /* (m)   var.lambda */
    SDPLRP_VEC_LAMBDA_UB = 1,  /* (m)   var.lambda_ub */
    SDPLRP_VEC_B = 2,          /* (m)   data.b */
    SDPLRP_VEC_PVIO_RAW = 3,   /* (m+1) var.primal_vio_raw */
    SDPLRP_VEC_Y = 4,          /* (m+1) var.y */
    SDPLRP_VEC_PVIO_LB = 5,    /* (m)   var.primal_vio_lb */
    SDPLRP_VEC_A_RD = 6,       /* (m+1) var.A_RD (already x2) */
    SDPLRP_VEC_A_DD = 7,       /* (m+1) var.A_DD */
    SDPLRP_VEC_S_NZVAL = 8,    /* (nnzF) aux.sparse_S.nzval */
    SDPLRP_VEC_TRIUS_NZVAL = 9 /* (nnzT) aux.triu_sparse_S.nzval (materialised on demand) */
};

/* ---- lifecycle -------------------------------------------------------- */
int32_t sdplrp_version(void);
const char *sdplrp_error_string(int32_t code);
/* rank 0 makes the 128-byte NCCL id; the host runtime broadcasts it */
int32_t sdplrp_nccl_unique_id(void *out128);
/* world == 1: nccl_id may be NULL and NCCL is never touched */
int32_t sdplrp_create(int32_t device, int32_t rank, int32_t world, const void *nccl_id, sdplrp_handle **out);
int32_t sdplrp_destroy(sdplrp_handle *h);
const char *sdplrp_last_error(sdplrp_handle *h);
int32_t sdplrp_synchronize(sdplrp_handle *h);
/* the CUDA stream the handle launches on (a cudaStream_t), for event timing */
void *sdplrp_stream(sdplrp_handle *h);

/* tuning knobs (all optional; defaults are the product configuration):
 *   "relabel"     -1 auto (default) / 0 off / 1 on: internal hub-first vertex order, set BEFORE
 *                 sdplrp_preprocess.  Invisible at the ABI (every upload/download converts).
 *   "hot_rows"    leading rows of the gathered factor pinned in L2 (evict_last); -1 = sized from L2
 *   "spmm_phases" 0 = one sweep per gather pass (default); 1 = two sweeps, hub columns (an L2-sized prefix of the
 *                 hub-first order) then tail columns; k > 1 = k hub columns.  One GPU, relabelled patterns only (experimental)
 *   "lanczos_dist" several GPUs: 1 = rows of S and of the Lanczos vectors are divided among the ranks (one all-gather of n
 *                 doubles + two scalar all-reduces per step; default), 0 = the q-step Lanczos operator is replicated on every
 *                 rank.  Only without re-orthogonalisation
 *   "row_group_max" rows with at most this many nonzeros are taken by one lane group each (default 64: measured 24 / 32 / 48 / 64 -> 4.27 / 4.14 / 4.06 / 4.02 ms for the C5 pass), longer ones by one
 *                 warp each; set BEFORE sdplrp_preprocess
 *   "spmm_unroll" nonzeros per block of the short-row kernels: 8 (default) or 4
 *   "spmm_g0"     1 = lane groups of exactly r/2 lanes per short row (default: 6 rows per warp at r = 10), 0 = next power of two
 *   "obj_value_free" 1 = when every off-diagonal value of C is the same +-2^k (unweighted MaxCut: 0.25) the gather pass
 *                 CD = C*D reads only C's pattern and scales each row once (default; same bits), 0 = it always reads C's values
 *   "rowc_kernel" pass over the per-row (single-diagonal-entry) constraints: 1 = barrier-free warp kernel, 32/(r/2) whole rows per
 *                 warp step (default on one GPU; rows of at most 32 pieces), 0 = shared-memory tile kernel (always on several GPUs).  Same bits either way
 *   "tail_ctas"   CTAs per SM of the fused step + gradient pass (1..8; 0 = auto, the default: 6 on one GPU, 4 on several.  Measured on C5, one GPU:
 *                 4 / 5 / 6 / 7 / 8 -> 1.16 / 1.10 / 0.98 / 1.31 / 1.20 ms)
 *   "halo"        several GPUs: every rank keeps the objective pattern of its own rows and the gather pass exchanges only the
 *                 factor rows that are actually gathered, hub class first.  1 = the tail class travels under a two-phase pass;
 *                 2 = the same exchange, then ONE sweep over whole rows (nothing overlaps the tail class, no second visit of
 *                 the rows); 3 = auto: 1 or 2 from the sizes of the plan (default); 0 = one all-gather of the whole
 *                 direction per iteration (round-1 path)
 *   "gather_mode" gather pass CD = C*D (gather.cu): 0 = row-binned register kernels, 1 = asynchronous tile pipeline with one
 *                 cp.async.bulk per gathered row, 2 = the same pipeline with 16-byte cp.async row pieces (even ranks <= 64)
 *   "gather_tile", "gather_stages", "gather_warps"  geometry of that pipeline (nonzeros per tile, stages of the
 *                 gathered-rows ring, warps per CTA); 0 = automatic
 *   "gather_hints" 1 = L2 evict_last / evict_first policies on the bulk row gathers of "gather_mode" 1
 *   "fused_tail"  1 = sdplrp_step_g uses the fused row pass (default), 0 = step and g separately
 *   "lbfgs_kernel" 1 = two-loop recursion on coefficients over directly computed dot products (default,
 *                 numlbfgsvecs <= 8), 0 = literal vector two-loop */
int32_t sdplrp_set_option(sdplrp_handle *h, const char *key, double value);

/* ---- preprocessing: preprocess_sparsecons + SolverAuxiliary ------------
 * The nA sparse matrices (sparse / diagonal A_i in order of appearance, then
 * C if it is sparse: src/structs.jl:303-325) as concatenated 1-based triplets
 * in `findnz` order (CSC: column-major; COO: stored order). mat_off has nA+1
 * 0-based offsets into I/J/V. sparse_global_inds[k] in 1..m, or m+1 for C.
 * Builds, on the device, the aggregated upper-triangular and full patterns
 * and every index map of src/preprocess.jl:24-169 (bit-exact; see
 * sdplrp_pattern_export) plus the device-only derived layouts. */
int32_t sdplrp_preprocess(sdplrp_handle *h, int64_t n, int64_t m, int64_t nA, const int64_t *mat_off,
                          const int64_t *I, const int64_t *J, const double *V,
                          const int64_t *sparse_global_inds);
/* sdplrp_preprocess with the triplet arrays I, J, V in DEVICE memory of the handle's GPU: a problem generator that builds
 * them there (exps/problems.jl:14-341 restated on the device, SURVEY.md 8f/f2) hands them over without a host round trip
 * (4.4 GB each way at the 10M-vertex MaxCut).  mat_off and sparse_global_inds are host arrays as above.  The arrays are
 * only read; work that produced them on another stream must have completed. */
int32_t sdplrp_preprocess_device(sdplrp_handle *h, int64_t n, int64_t m, int64_t nA, const int64_t *mat_off,
                                 const int64_t *d_I, const int64_t *d_J, const double *d_V,
                                 const int64_t *sparse_global_inds);
/* ---- structured problem blocks (SURVEY.md 8f/f2) --------------------------------------------------------------------------
 * The sparse list of sdplrp_preprocess described block by block, in order of appearance (A_1 ... A_m, then C if sparse), and
 * expanded on the device into the `findnz`-order triplets -- what the reference's problem constructors build one
 * SparseMatrixCOO at a time (test/problem.jl:16-30, 50-62, 80-92, 100-110).  A block of kind
 *   TRIPLETS  one matrix, stored entries I, J (1-based), V in findnz order (nnz of them)
 *   CSC       one matrix as SparseMatrixCSC fields: I = rowval (nnz), J = colptr (n+1), both 1-based, V = nzval
 *   DIAG      `count` matrices with ONE entry each: matrix k = V[k] * e_p e_p', p = I[k] (I NULL: p = k+1; V NULL: 1.0)
 *             -- Diag(X) = 1 of MaxCut / cut-norm / minimum bisection
 *   EDGES     `count` matrices with the two stored entries (I[k], J[k]), (J[k], I[k]), both V[k] (V NULL: 1.0)
 *             -- X_ij = 0 for every edge of Lovasz theta
 *   IDENTITY  one matrix sparse(1.0I, n, n) -- the trace constraint
 * takes the global ids first_gid, first_gid+1, ... (1-based; m+1 for C).  on_device != 0: the arrays are device memory of
 * the handle's GPU.  Maps, error codes and everything downstream are those of sdplrp_preprocess on the expanded triplets. */
enum { SDPLRP_BLOCK_TRIPLETS = 0, SDPLRP_BLOCK_CSC = 1, SDPLRP_BLOCK_DIAG = 2, SDPLRP_BLOCK_EDGES = 3, SDPLRP_BLOCK_IDENTITY = 4 };
typedef struct {
    int64_t kind, on_device, count, first_gid, nnz;
    const int64_t *I, *J;
    const double *V;
} sdplrp_block;
int32_t sdplrp_preprocess_blocks(sdplrp_handle *h, int64_t n, int64_t m, int64_t nblocks, const sdplrp_block *blocks);
int32_t sdplrp_pattern_sizes(sdplrp_handle *h, int64_t *nnzT, int64_t *nnzF, int64_t *Ec);
/* the weight v that the one-sweep row kernels of the gather pass CD = C*D factor out of C ("obj_value_free"), 0 when they
 * read C's values.  The asynchronous tile pipeline ("gather_mode"), the two-phase pass ("spmm_phases") and the halo pass of
 * several GPUs always read the values */
int32_t sdplrp_value_free_weight(sdplrp_handle *h, double *v);
/* 1-based, exactly the seven outputs of preprocess_sparsecons (SURVEY Appendix B) */
int32_t sdplrp_pattern_export(sdplrp_handle *h, int64_t *triu_colptr, int64_t *triu_rowval, int64_t *matptr,
                              int64_t *nzind, double *nzval_one, double *nzval_two, int64_t *full_colptr,
                              int64_t *full_rowval, int64_t *mappedto_triu);
/* SymLowRankMatrix(Diagonal(D), B): B is n x s column-major; global_id in 1..m+1
 * (src/structs.jl:11-24, 310-312, 326-328). Call after sdplrp_preprocess
 * (with nA = 0 when there is no sparse matrix). */
int32_t sdplrp_add_symlowrank(sdplrp_handle *h, int64_t global_id, int64_t s, const double *B, const double *D);
/* data.b and constraint types (1 = inequality <=) -> lambda_ub / primal_vio_lb
 * (src/structs.jl:228, 248-249). is_ineq may be NULL (all equalities). */
int32_t sdplrp_set_problem(sdplrp_handle *h, const double *b, const uint8_t *is_ineq);

/* ---- state: SolverVars / LBFGSHistory --------------------------------- */
/* (re)allocates R,G,D and the 2*numlbfgsvecs history for rank r and clears the
 * history (lbfgs_init, src/lbfgs.jl:35-47; rank_update!, src/coreop.jl:518-526).
 * Supported ranks: 1 <= r <= SDPLRP_MAX_RANK (256), and r <= SDPLRP_MAX_ODD_RANK (128)
 * when r is odd -- the sparse row kernels hold at most 4 x 32 lanes of 2 (even r) or
 * 1 (odd r) columns per row.  Any other r returns SDPLRP_ERR_ARG before anything is
 * allocated or launched; the previous rank and state stay valid.  sdplrp_solve's rank
 * update clamps min(barvinok_pataki, 2r) to this range (an odd r > 128 steps down by 1). */
#define SDPLRP_MAX_RANK 256
#define SDPLRP_MAX_ODD_RANK 128
int32_t sdplrp_set_rank(sdplrp_handle *h, int32_t r, int32_t numlbfgsvecs);
int32_t sdplrp_set_sigma(sdplrp_handle *h, double sigma);
int32_t sdplrp_get_sigma(sdplrp_handle *h, double *sigma);
int32_t sdplrp_get_obj(sdplrp_handle *h, double *obj);
int32_t sdplrp_upload_mat(sdplrp_handle *h, int32_t mat_id, const double *src /* r*n */);
int32_t sdplrp_download_mat(sdplrp_handle *h, int32_t mat_id, double *dst /* r*n */);
/* Several GPUs (one process per GPU), CONTIGUOUS slices: rank q reads / writes rows [q*S, min(n, (q+1)*S)) of the caller's matrix, S = ceil(n / world).
 * Upload: the slices are exchanged over NVLink, every rank ends up with the whole matrix.  Download: the matrix is completed
 * over NVLink and each rank writes its slice; the union over the ranks is the result. */
int32_t sdplrp_upload_mat_slice(sdplrp_handle *h, int32_t mat_id, const double *src /* r*n */);
int32_t sdplrp_download_mat_slice(sdplrp_handle *h, int32_t mat_id, double *dst /* r*n */);
int32_t sdplrp_upload_vec(sdplrp_handle *h, int32_t vec_id, const double *src, int64_t len);
int32_t sdplrp_download_vec(sdplrp_handle *h, int32_t vec_id, double *dst, int64_t len);

/* ---- seam-level operators (parity with test/coreop.jl) ---------------- */
/* A!(out, aux, Ut): out (m+1 doubles, host, may be NULL) also lands in the
 * device scratch vector; src/coreop.jl:36-49 */
int32_t sdplrp_A_uu(sdplrp_handle *h, int32_t U_id, double *out);
/* A!(out, aux, Ut, Vt) = A((UV'+VU')/2); src/coreop.jl:54-70 */
int32_t sdplrp_A_uv(sdplrp_handle *h, int32_t U_id, int32_t V_id, double *out);
/* At_preprocess!(var, aux): S = sum_i y_i A_i + y_{m+1} C on the aggregated
 * pattern. y (m+1, host) may be NULL to use the device var.y; src/coreop.jl:248-258 */
int32_t sdplrp_At_preprocess(sdplrp_handle *h, const double *y);
/* At!(Y, X, aux, var): Y = X*S + low-rank terms; src/coreop.jl:260-279 */
int32_t sdplrp_At_left(sdplrp_handle *h, int32_t X_id, int32_t Y_id);
/* At!(y, aux, x, var): y = S*x + low-rank terms, x and y n x ncols
 * column-major host arrays; src/coreop.jl:281-300 */
int32_t sdplrp_At_right(sdplrp_handle *h, const double *x, double *y, int64_t ncols);

/* ---- fused iteration -------------------------------------------------- */
/* f!: primal_vio_raw, obj, AL value; src/coreop.jl:11-31 */
int32_t sdplrp_f(sdplrp_handle *h, double *L, double *obj);
/* g!: y, S, G = 2*R*S (+low rank); returns ||G||_F^2 and ||max(raw,lb)||_2^2
 * (the two norms of src/sdplr.jl:224-234); src/coreop.jl:305-317 */
int32_t sdplrp_g(sdplrp_handle *h, double *gnorm2, double *pnorm2);
/* fg!: out = {L, obj, ||G||_F^2, ||pvio||_2^2}; src/coreop.jl:323-349 */
int32_t sdplrp_fg(sdplrp_handle *h, double out[4]);
/* lbfgs_dir!(dirt, his, Gt; negate=true) + descent = dot(dirt, Gt);
 * src/lbfgs.jl:77-124, src/sdplr.jl:197-201 */
int32_t sdplrp_lbfgs_dir(sdplrp_handle *h, double *descent);
/* non-descent fallback: Gt *= -1; dirt = Gt; src/sdplr.jl:202-205 */
int32_t sdplrp_use_gradient_direction(sdplrp_handle *h);
/* the two A passes of linesearch! fused (A_RD already x2, A_DD) and the five
 * quartic coefficients; src/linesearch.jl:10-16, 36-56 */
int32_t sdplrp_linesearch_coeffs(sdplrp_handle *h, double biquadratic[5]);
/* after alpha is chosen: primal_vio_raw += a(a A_DD + A_RD), obj, and
 * Rt += a*dirt; src/linesearch.jl:118-124, src/sdplr.jl:219 */
int32_t sdplrp_step(sdplrp_handle *h, double alpha, double *obj);
/* sdplrp_step followed by sdplrp_g as ONE call (the caller's `axpy!` + `g!` + the two norms, src/sdplr.jl:219-234):
 * out = {obj, ||G||_F^2, ||pvio||_2^2}.  When the line search of the current direction is still valid the library
 * runs them as a single fused row pass; results are those of the two separate calls. */
int32_t sdplrp_step_g(sdplrp_handle *h, double alpha, double out[3]);
/* lbfgs_update!(dirt, his, Gt, alpha); src/lbfgs.jl:129-149 */
int32_t sdplrp_lbfgs_update(sdplrp_handle *h, double alpha);
/* lbfgs_clear!; src/lbfgs.jl:52-59 */
int32_t sdplrp_lbfgs_clear(sdplrp_handle *h);
/* lambda_i <- min(ub_i, lambda_i - sigma*raw_i); src/sdplr.jl:358-362 */
int32_t sdplrp_dual_update(sdplrp_handle *h);
/* sharp AL at k step sizes + the slope at 0 (eval_AL closure and slope of
 * linesearch_armijo!; needs linesearch_coeffs first); src/linesearch.jl:158-172 */
int32_t sdplrp_armijo_eval(sdplrp_handle *h, const double *alphas, int32_t k, double *L, double *slope);

/* ---- dual bound ------------------------------------------------------- */
/* q-step Lanczos on the current S (set by At_preprocess / g / dual_obj):
 * alpha,beta (q doubles each, host) receive the unshifted recurrence
 * coefficients, *iters the steps done. v0 (n, host) is the unnormalised start
 * vector; NULL draws a seeded Gaussian on the device. reorth != 0 adds full
 * re-orthogonalisation (the reference has none); src/coreop.jl:461-500 */
int32_t sdplrp_lanczos(sdplrp_handle *h, int64_t q, const double *v0, uint64_t seed, int32_t reorth,
                       double *alpha, double *beta, int64_t *iters);
/* smallest eigenvalue of SymTridiagonal(d, e) (host; replaces the symeigs
 * call of src/coreop.jl:509-511) */
int32_t sdplrp_tridiag_mineig(const double *d, const double *e, int64_t k, double *out);
/* dual_obj (Lanczos branch): y, S, q = 2*ceil(sqrt(max(iter,100))*log n)
 * Lanczos steps, dual = -y'b + trace_bound*min(lambda_min,0); src/coreop.jl:376-415 */
int32_t sdplrp_dual_obj(sdplrp_handle *h, double trace_bound, int64_t iter, const double *v0, uint64_t seed,
                        double *dual_value, double *mineig, int64_t *lanczos_steps);

/* ---- high-precision eigenvalue path and DIMACS errors ------------------ */
/* SDP_S_eigval(var, aux, nevs, true; which=:SA, ncv, tol, maxiter) (src/coreop.jl:351-374): the nevs smallest
 * algebraic eigenvalues of the S last assembled (+ low-rank terms), ascending, by thick-restart Lanczos on the device
 * (the restarted-Lanczos contract of GenericArpack.symeigs: Ritz pair i is accepted when its residual bound
 * |beta_m y_m,i| <= tol * max(eps^(2/3), |theta_i + 1|); tol <= 0 means machine precision; maxiter bounds the number of
 * restarts; nevs < ncv <= min(n, 512) is enforced by clamping ncv).  v0 (n, host) is the start vector, NULL draws a
 * seeded Gaussian on the device.  bounds / matvecs / restarts may be NULL. */
int32_t sdplrp_S_eigval(sdplrp_handle *h, int64_t nevs, int64_t ncv, double tol, int64_t maxiter, const double *v0, uint64_t seed,
                        double *eigvals, double *bounds, int64_t *matvecs, int64_t *restarts);
/* dual_obj(data, var, aux, trace_bound, iter; highprecision=true): y, S, then SDP_S_eigval with ncv = min(100, n),
 * tol = 1e-6, maxiter = 10^6; src/coreop.jl:376-415 */
int32_t sdplrp_dual_obj_highprecision(sdplrp_handle *h, double trace_bound, const double *v0, uint64_t seed, double *dual_value,
                                      double *mineig, int64_t *matvecs);
/* DIMACS_errors(data, var, aux) -> errs[6] (src/coreop.jl:417-453); normb = ||b||_2, normC = ||C||_F are the caller's
 * (src/sdplr.jl:165-166).  Like the reference it overwrites y with -lambda (copy2y_lambda!) and S with the matching
 * matrix, and error 6 takes the sparse part of S only. */
int32_t sdplrp_dimacs_errors(sdplrp_handle *h, double normb, double normC, const double *v0, uint64_t seed, double errs[6]);
/* host helper: eigen-decomposition of a small dense symmetric matrix A (k x k row-major): ascending eigenvalues ev[k],
 * eigenvectors as the columns of Q (k x k row-major, may be NULL).  The projected problem of the restarted Lanczos. */
int32_t sdplrp_dense_symeig(const double *A, int64_t k, double *ev, double *Q);
/* Hyperplane rounding (Goemans-Williamson) of the current R: K candidates x_k = sign(R g_k), x_{k,i} = +1 when
 * <R_i, g_k> >= 0, else -1.  g_k in R^r: rows of G (K x r row-major, host) or, G NULL, standard normals from a
 * counter-based generator keyed by (seed, k, column) -- the same hyperplanes for every GPU count, vertex order and
 * K (candidate k of a call with K = 100 equals candidate k of a call with K = 64).  G_out (K x r, may be NULL) receives
 * the hyperplanes used.  obj[k] = <C, x_k x_k'> over the sparse objective (the quantity sdplrp_get_obj reports for R),
 * sum[k] = sum_i x_{k,i} (may be NULL; the imbalance of a bisection).  best (1-based) is the candidate with the smallest
 * obj, ties to the lowest k; best_x (n, host, reference vertex order, may be NULL) receives it as +-1.0.
 * Reads R only: no other device state (G, D, CR, CD, y, S, residuals, L-BFGS history, W0/W1) changes.
 * Several GPUs: every rank passes the same K, seed and G and receives the same results.
 * SDPLRP_ERR_ARG for K < 1, NULL obj / best, and when C has a low-rank part (or no sparse part). */
int32_t sdplrp_round_hyperplane(sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, double *G_out,
                                double *obj, double *sum, int64_t *best, double *best_x);
/* Hyperplane rounding followed by parallel one-flip descent on every candidate.  The start vectors x_k^0 are those of
 * sdplrp_round_hyperplane (same G / seed rule, ties to +1); obj_round[k] (may be NULL) is the objective of x_k^0, bit for
 * bit the obj[k] of sdplrp_round_hyperplane.  Round t = 0, 1, ... on every candidate k independently: with
 * h_ik = sum_{j != i} C_ij x_jk, vertex i wants to flip iff x_ik h_ik > 0 (flipping it changes the objective by
 * -4 x_ik h_ik).  The neighbours of i are the j != i with C_ij != 0.  Priority key(i, t) = mix64(i ^ mix64(0xD1B54A32D192ED03
 * * (t + 1))) (splitmix64 finalizer, mod 2^64) on the 0-based input vertex index i; j beats i iff key(j, t) > key(i, t), or
 * the keys are equal and j < i.  Vertex i flips iff it wants to and no neighbour that beats it also wants to: the flipped
 * vertices are pairwise non-adjacent, their gains add up and the objective falls every round.  A batch of 64 candidates
 * stops when none of its vertices wants to flip, or after max_rounds rounds.
 * Outputs: obj[k] = <C, x_k x_k'> of the final vector, sum[k] = sum_i x_{k,i}, flips[k] = single-vertex flips,
 * rounds[k] = the last (1-based) round that flipped something in candidate k, 0 when x_k^0 is a one-flip local optimum,
 * -1 when x_k still had a vertex that wanted to flip after max_rounds rounds (not a local optimum).  best (1-based) is the
 * smallest obj, ties to the lowest k; best_x (reference vertex order) its final vector.  obj_round, sum, flips, rounds,
 * G_out and best_x may be NULL.  With max_rounds = 0 and rounds NULL this is sdplrp_round_hyperplane.
 * Candidate k's result does not depend on K or on the other candidates.  Reads R only, like sdplrp_round_hyperplane.
 * Where the gains are exactly representable (unit-weight MaxCut, +-1-weight cut-norm, integer Laplacians) the results are
 * bit-identical across vertex orders and GPU counts; with general real weights a gain within rounding of 0 may be decided
 * differently under a different summation order.
 * Several GPUs: every rank passes the same K, seed, G and max_rounds and receives the same results.
 * Errors as sdplrp_round_hyperplane, and SDPLRP_ERR_ARG for max_rounds < 0. */
int32_t sdplrp_round_local_search(sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, int64_t max_rounds,
                                  double *G_out, double *obj_round, double *obj, double *sum, int64_t *flips,
                                  int64_t *rounds, int64_t *best, double *best_x);

/* ---- native host driver (SURVEY.md 8f, f1) ------------------------------ */
/* BurerMonteiroConfig (src/options.jl:1-24); every field is 8 bytes wide so the layout is the same from C, Julia
 * (`struct` of Float64 / Int64 / UInt64) and ctypes.  *_relative: 1 = "relative" (default), 0 = "absolute". */
typedef struct {
    double ptol, gtol, objtol, sigma_0, sigmafac, maxtime, printfreq, fprec, prior_trace_bound, alpha_max;
    int64_t maxmajoriter, maxiter, numlbfgsvecs, rankupd_tol, printlevel;
    int64_t gtol_relative, ptol_relative, objtol_relative, eval_DIMACS_errs, eigval_highprecision;
    uint64_t seed; /* counter-based device generator: eigenvalue start vectors, random R of a rank update / of a NULL Rt0 */
} sdplrp_config;
/* the scalar entries of the reference's result Dict (src/sdplr.jl:426-448); Rt and the multipliers are fetched with
 * sdplrp_download_mat(SDPLRP_MAT_R) / the best_lambda argument.  status: 0 = tolerances met, 1 = iteration / time /
 * major-iteration budget exhausted. */
typedef struct {
    double sigma, grad_norm, primal_vio, obj, L, max_dual_value, min_duality_gap, totaltime, dual_time, primaltime, DIMACS_time;
    double DIMACS_errs[6];
    int64_t iter, majoriter, lanczos_steps, r, status;
} sdplrp_result;
int32_t sdplrp_config_default(sdplrp_config *cfg);
/* _sdplr (src/sdplr.jl:140-449) as one call: the same sequence of entry points a Julia host issues, driven natively.
 * Rt0 (r x n column-major) / lambda0 (m) may be NULL (R ~ U(-1,1) from the device generator, lambda = 0:
 * src/structs.jl:236-237).  normb = ||b||_2, normC = ||C||_F as computed by the caller (src/sdplr.jl:165-166).
 * best_lambda (m+1 doubles, may be NULL) receives the multipliers of the best dual bound (src/sdplr.jl:325).
 * Inequality problems (sdplrp_set_problem) use the Armijo search, as the reference does. */
int32_t sdplrp_solve(sdplrp_handle *h, const sdplrp_config *cfg, int64_t r, const double *Rt0, const double *lambda0, double normb,
                     double normC, sdplrp_result *result, double *best_lambda);
/* k passes of the inner loop body of _sdplr (src/sdplr.jl:194-246) without the tolerance logic: direction, descent test,
 * line search (use_armijo != 0: backtracking), step, gradient, and -- update_history != 0 -- the L-BFGS update.
 * out = {L, obj, ||G||_F^2, ||pvio||_2^2, alpha} of the last pass.  What bench.py times. */
int32_t sdplrp_iterate(sdplrp_handle *h, int64_t k, double alpha_max, int32_t use_armijo, int32_t update_history, double out[5]);
/* root selection of linesearch! (src/linesearch.jl:58-112) for quartic coefficients as returned by
 * sdplrp_linesearch_coeffs: the minimiser over the real roots of the derivative in [0, alpha_max] and alpha_max itself
 * (host only).  Returns SDPLRP_ERR_LINESEARCH when cubic[1] > eps. */
int32_t sdplrp_pick_alpha(const double biquadratic[5], double alpha_max, double *alpha, double *value);
/* mat (R, G or D) <- 2u - 1 with u ~ U[0,1) from the counter-based device generator, keyed by (seed, reference vertex,
 * column): the same matrix for every GPU count and internal vertex order (SolverVars' `2 .* rand(r, n) .- 1`,
 * src/structs.jl:236, without the 0.8 GB host round trip at n = 10^7) */
int32_t sdplrp_fill_uniform(sdplrp_handle *h, int32_t mat_id, uint64_t seed);

/* ---- introspection ---------------------------------------------------- */
/* kernel-group sections timed with CUDA events on the handle's stream */
enum {
    SDPLRP_SEC_LBFGS_DIR = 0,    /* two-loop recursion kernels (2h+1 launches) */
    SDPLRP_SEC_LS_PASS = 1,      /* fused {A(RD'+DR'), A(DD')} sampled-dot kernels */
    SDPLRP_SEC_LS_COEFF = 2,     /* quartic-coefficient reduction */
    SDPLRP_SEC_STEP = 3,         /* residual recurrence + R += alpha*D */
    SDPLRP_SEC_S_ASSEMBLE = 4,   /* y formation + S update */
    SDPLRP_SEC_SPMM = 5,         /* CD = C*D (objective gather pass with the fused line-search dots), CR rebuilds */
    SDPLRP_SEC_NORMS = 6,        /* ||G||^2, ||pvio||^2 */
    SDPLRP_SEC_LBFGS_UPDATE = 7,
    SDPLRP_SEC_A_UU = 8,         /* A(RR') of f! */
    SDPLRP_SEC_F_FINISH = 9,
    SDPLRP_SEC_LANCZOS = 10,
    SDPLRP_SEC_COMM = 11,        /* NCCL collectives */
    SDPLRP_SEC_GRAD = 12,        /* G = 2*(y_obj*CR + S_dyn*R + low rank) with ||G||^2 fused */
    SDPLRP_SEC_TAIL = 13,        /* fused step + y + gradient + norms row pass (sdplrp_step_g) */
    SDPLRP_SEC_COUNT = 14
};
/* on != 0: record a CUDA-event pair around every section from now on */
int32_t sdplrp_set_profiling(sdplrp_handle *h, int32_t on);
/* synchronises, adds the pending event pairs up and returns (then resets) the
 * accumulated milliseconds and launch-group counts per section (SDPLRP_SEC_COUNT each) */
int32_t sdplrp_section_times(sdplrp_handle *h, double *ms, int64_t *counts);
/* number of kernels this handle has launched since creation */
int32_t sdplrp_launch_count(sdplrp_handle *h, int64_t *count);
/* rows [lo,hi) of R/G/D owned by this rank (0-based) */
/* several GPUs: the halo plan of the gather pass on this rank: {active, own rows, own nonzeros, hub ghost rows, tail ghost rows,
 * hub rows packed per pass, tail rows packed per pass} (a packed row goes to one peer; a row needed by k peers counts k times) */
int32_t sdplrp_halo_stats(sdplrp_handle *h, int64_t out[7]);
int32_t sdplrp_row_range(sdplrp_handle *h, int64_t *lo, int64_t *hi);

#ifdef __cplusplus
}
#endif
#endif /* SDPLRP_B200_H */
