// common.cuh -- handle, error plumbing and device-side reduction helpers shared
// by every translation unit of libsdplrp_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/sdplrp_b200.h"

typedef long long i64;

constexpr int kNumSM = 148;          // B200: 2 dies x 74 SMs
constexpr int kMaxHist = 32;         // numlbfgsvecs upper bound (ids S0..S0+31)
constexpr int kRedBlocks = 4 * kNumSM;  // persistent grid of streaming/reduction kernels
constexpr int kRedThreads = 256;
constexpr int kMaxRedK = 64;         // max simultaneous sums of one reduction kernel
constexpr int kLbSmallLen = 17 * 17 + 3 * 17 + 17 + 7;  // Gram (17x17) + three probe rows + coefficients
constexpr long long kPartialsLen = (long long)kRedBlocks * kMaxRedK * 8;  // doubles in h->partials
constexpr int kLongMatThreshold = 64;   // matrices with more triu entries go to the chunked path
constexpr int kChunkEntries = 2048;     // entries per chunk (one CTA) of a long matrix
constexpr int kRowGroupMax = 64;        // rows with <= this many nonzeros: one sub-warp lane group per row
constexpr int kRowWarpMax = 512;        // rows with <= this many: one warp per row; longer: chunks of this size, one warp each

// the ranks every kernel handles (include/sdplrp_b200.h, sdplrp_set_rank): at most 4 units of 32 lanes per row in the sparse
// row kernels (gradient.cu, launch_csr), each lane holding 2 columns for even r and 1 for odd r
static inline bool rank_supported(long long r) {
    return r >= 1 && r <= SDPLRP_MAX_RANK && (r % 2 == 0 || r <= SDPLRP_MAX_ODD_RANK);
}
// rank_update! (src/coreop.jl:518-526) r <- min(bp, 2r), clamped to the largest supported rank at or below it
// (solver.py rank_after_update is the same rule)
static inline long long rank_after_update(long long bp, long long r) {
    long long t = std::min(std::min(bp, 2 * r), (long long)SDPLRP_MAX_RANK);
    if (t % 2 == 1 && t > SDPLRP_MAX_ODD_RANK) t -= 1;
    return t;
}

// rows of a CSR pattern binned by length (compacted lists, natural order inside a bin);
// list[c] == nullptr with cnt[c] == n means "all rows" (identity, keeps streaming access)
struct RowClasses {
    int *list[3] = {nullptr, nullptr, nullptr};
    long long cnt[3] = {0, 0, 0};
    int *storage = nullptr;
};

// long rows cut into chunks (one warp each, gradient.cu)
struct TileLayout {
    long long n_long = 0, n_chunks = 0;
    int *long_rows = nullptr;    // n_long   rows with more than `chunk` nonzeros (ascending)
    int *long_cptr = nullptr;    // n_long+1 first chunk of each long row
    int *chunk_start = nullptr, *chunk_end = nullptr, *chunk_row = nullptr;  // n_chunks
};

// tile plan of the asynchronous gather pass (gather.cu): the CSR of a row range cut into tiles of whole rows with at most T
// nonzeros; rows longer than T become chunk tiles combined per row afterwards
struct GatherPlan {
    int4 *tiles = nullptr;       // {row0, nrows (< 0: chunk, slot = ~nrows), nz0, nnz}
    long long ntiles = 0, n_long = 0, n_chunks = 0;
    int *long_rows = nullptr;    // n_long
    int *long_cptr = nullptr;    // n_long+1 chunk slots of each long row
    const int *ptr_key = nullptr;
    long long row_lo = 0, row_hi = 0;
    int T = 0;
};

// Multi-GPU gather pass (world > 1, dealt equal blocks, sparse objective, constraints in per-row lists): the LOCAL view of the
// objective pattern -- only the owned rows, columns renumbered to [own rows | hub ghosts | tail ghosts] -- and the lists of
// the halo exchange that replaces the all-gather of the gathered factor (preprocess.cu: halo_build, comm.cu: halo_*).
struct HaloPlan {
    bool active = false;
    long long nloc = 0, lnnz = 0;
    long long n_ghost[2] = {0, 0};       // ghost rows per class: 0 = hub part of the other ranks' blocks, 1 = tail part
    long long n_send[2] = {0, 0};        // rows this rank packs per class (a row goes once to every peer that gathers it)
    int *lptr = nullptr, *lmid = nullptr, *lidx = nullptr;   // nloc+1, nloc, lnnz: row i = [lptr[i], lmid[i]) own + hub-ghost columns,
    double *lval = nullptr;                                   //                   [lmid[i], lptr[i+1]) tail-ghost columns
    RowClasses cls;                      // row bins of the local rows
    TileLayout longs;                    // their long rows in chunks
    int *send_rows[2] = {nullptr, nullptr};                   // local row ids to pack, grouped by destination rank
    std::vector<long long> send_off[2], recv_off[2];          // world+1 row offsets per class
    double *sendbuf = nullptr;                                // (n_send[0] + n_send[1]) x r
    double *xc = nullptr;                                     // the gathered operand of a pass, compact: [own rows | hub ghosts | tail ghosts] x r
    long long sendbuf_len = 0, xc_len = 0;
};

// hyperplane rounding (rounding.cu): buffers allocated on first use, freed with the problem
struct RoundingState {
    unsigned long long *words = nullptr;  // n: one bit per candidate of the current batch, internal vertex order
    double *x = nullptr;                  // n: the expanded +-1 vector of the best candidate
    int *chunk_row = nullptr;             // nchunks: first row of every chunk of the evaluation pass
    long long e_lo = 0, e_hi = 0, nchunks = 0;  // owned nonzeros [e_lo, e_hi) of the full pattern
    double *G = nullptr, *sums = nullptr; // K x r hyperplanes; per batch 4 x 64 sums (set bits, eval sums, first eval sums,
                                          // flips), then sum of C and 64 want counts of a local-search round
    long long G_len = 0, sums_len = 0;
    // one-flip local search (first use)
    unsigned long long *want = nullptr, *flip = nullptr;  // n: want / flip word of every vertex in the current round
    unsigned long long *best_words = nullptr;             // n: final words of the batch that holds the best candidate so far
    unsigned char *dirty = nullptr;                       // n: the row's want word must be recomputed
    int *long_rows = nullptr, *long_sptr = nullptr;       // rows of the full pattern with more than kLsLong nonzeros (ascending),
                                                          // and the first segment of each (+1)
    int *seg_row = nullptr, *seg_start = nullptr;         // n_seg: row and first nonzero of every segment
    double *seg_part = nullptr;                           // n_seg x 64 want sums of a segment
    long long n_seg = 0, l_lo = 0, l_hi = 0, s_lo = 0, s_hi = 0;  // the owned long rows [l_lo, l_hi) and their segments [s_lo, s_hi)
};

struct LowRank {
    i64 gid;     // 0-based global slot
    i64 s;
    double *dB;  // n x s column-major
    double *dD;  // s
};

// device scalar slots (h->dscal)
enum {
    SC_DOT = 0,       // running dot of the L-BFGS recursion
    SC_DESCENT = 1,
    SC_GNORM2 = 2,
    SC_PNORM2 = 3,
    SC_OBJ = 4,
    SC_LVAL = 5,
    SC_BQ = 8,        // 8 partial sums -> 5 quartic coefficients
    SC_RHO = 32,      // rho_j, j < kMaxHist
    SC_A = 64,        // a_j (alpha of the first loop)
    SC_SUMS = 16,     // 3 row classes x 2 fused sums of the sparse kernels (6 doubles)
    SC_LANCZOS = 96,  // alpha_i, beta_i, stop flag scratch
    SC_COUNT = 128
};

struct sdplrp_handle {
    int device = 0, rank = 0, world = 1;
    cudaStream_t stream = nullptr;
    std::string err;
    i64 launches = 0;
    void *nccl = nullptr;  // ncclComm_t when world > 1

    // problem sizes
    i64 n = 0, m = 0, nA = 0, nnzT = 0, nnzF = 0, Ec = 0;
    i64 row_lo = 0, row_hi = 0;  // rows of R/G/D owned by this rank
    std::vector<i64> row_starts; // world+1 block boundaries (identical on every rank)
    i64 c_lo = 0, c_hi = 0;      // internal slots of the per-row constraints of the owned rows (vecops.cu)
    std::vector<i64> c_starts;   // world+1: rowc_ptr[row_starts[q]]
    bool mat_full[8] = {true, true, true, true, true, true, true, true};  // R,G,D,W0,W1: all rows valid here?
    bool preprocessed = false;
    bool has_ineq = false;       // some constraint is an inequality (sdplrp_set_problem): the driver uses the Armijo search

    // aggregated patterns (0-based int32 on device)
    int *triu_colptr = nullptr, *triu_rowval = nullptr;  // n+1, nnzT   (CSC of triu == CSR of tril), reference labels
    int *ref_full_ptr = nullptr, *ref_full_idx = nullptr;  // n+1, nnzF  agg_sparse_A in reference labels (export only)
    int *mapped = nullptr;                               // nnzF (reference slot) -> triu slot
    // internal vertex order: rows sorted by descending degree (hubs first) so that the hot rows of the
    // gathered factor are contiguous and the row classes are ranges.  Invisible at the ABI: uploads and
    // downloads of anything indexed by vertex go through perm / iperm.
    bool relabeled = false;
    bool equal_blocks = false;                           // ... and ranks 0..P-2 hold exactly block_rows rows (in-place ncclAllGather)
    i64 block_rows = 0;
    bool dealt = false;                                  // multi-GPU: row blocks fixed by the round-robin deal of the relabeling
    int relabel_mode = -1;                               // -1 auto, 0 off, 1 on (sdplrp_set_option "relabel")
    int *perm = nullptr, *iperm = nullptr;               // n: internal label of reference vertex / its inverse
    int *i2r = nullptr, *r2i = nullptr;                  // nnzF: internal full slot <-> reference full slot
    int *full_ptr = nullptr, *full_idx = nullptr;        // n+1, nnzF   the symmetric pattern as CSR in INTERNAL labels
    double *S = nullptr;                                 // nnzF  sparse_S.nzval (internal slot order)
    double *stage = nullptr;                             // n x r staging buffer of the permuting copies
    i64 stage_len = 0;
    i64 l2_persist_bytes = 0;                            // cudaLimitPersistingL2CacheSize set at creation
    i64 hot_rows = -1;                                   // leading (hub) rows of a gathered factor kept in L2; -1 = auto
    int row_group_max = kRowGroupMax;                    // rows with <= this many nonzeros go to the lane-group-per-row kernels (set before preprocessing)
    int spmm_unroll = 8;                                 // nonzeros per predicated block of the class-0 register kernel (4 or 8)
    int tail_ctas = 0;                                   // CTAs per SM of the fused tail kernel k_step_grad (gradient.cu); 0 = auto (6 on one GPU, 4 on several)
    int rowc_kernel = 1;                                 // row-list constraint pass: 1 = barrier-free warp kernel (r/2 <= 32 pieces), 0 = shared-memory tile kernel (aop.cu)
    int spmm_g0 = 1;                                     // class-0 lane groups of exactly r/2 lanes (0: next power of two)
    int spmm_phases = 0;                                 // 0 = one sweep per gather pass (default); 1 = hub | tail two-phase pass with an
                                                         // L2-sized hub prefix; > 1 = that many hub columns (gradient.cu, grad_obj_spmm)
    int lanczos_dist = 1;                                // world > 1: 1 = row-partitioned q-step Lanczos (default; measured identical to the replicated
                                                         // recurrence on 2 GPUs and 2.5x faster), 0 = replicated operator (lanczos.cu: lz_run_dist)
    cudaStream_t class_streams[2] = {nullptr, nullptr};  // side streams of the medium / long row classes of a gather pass (gradient.cu)
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    bool fork_open = false;                              // a caller forked the side streams around several launches of one pass
    // multi-GPU halo exchange of the gather pass (preprocess.cu: halo_build, comm.cu)
    int halo_mode = 3;                                   // 0 = all-gather of the whole factor (round-1 path), 1 = halo exchange under a two-phase pass,
                                                         // 2 = halo exchange, then one sweep, 3 = auto (1 or 2 from the plan's sizes; default)
    HaloPlan halo;
    void *nccl_halo = nullptr;                           // second communicator (ncclCommSplit) for the exchange on comm_stream
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t ev_pack = nullptr, ev_class[2] = {nullptr, nullptr};
    // asynchronous tile pipeline of the gather pass (gather.cu)
    int gather_mode = 0;                                 // 0 = register kernels of gradient.cu, 1 = cp.async.bulk row gathers, 2 = 16-byte cp.async row gathers
    int gather_tile = 0, gather_stages = 0, gather_warps = 0;  // 0 = automatic (gather_geometry)
    int gather_hints = 0;                                // 1 = L2 evict_last / evict_first policies on the row gathers (MODE 1)
    i64 gather_attr_smem[2][5] = {{0}};                 // dynamic shared memory the kernel variants were last sized for
    GatherPlan full_plan;                                // plan of the full pattern over the owned rows
    int *row_mid = nullptr;                              // n: first tail-column position of every row (two-phase pass)
    i64 row_mid_cols = -1;                               // hub prefix row_mid was built for
    // per-entry lists in reference order (E_c)
    int *matptr = nullptr;     // nA+1
    int *mat_gid = nullptr;    // nA   0-based global slot of each sparse matrix
    int *ent_slot = nullptr;   // Ec   nzind (0-based triu slot)
    int *ent_row = nullptr, *ent_col = nullptr;  // Ec   coordinates of that slot in INTERNAL labels
    double *ent_one = nullptr, *ent_two = nullptr;  // Ec
    // chunked ("long") matrices for the A passes
    i64 n_long = 0, n_chunks = 0;
    int *long_mat = nullptr;       // n_long: matrix index
    int *long_chunk_ptr = nullptr; // n_long+1: first chunk of each long matrix
    int *chunk_mat = nullptr;      // n_chunks: index into long_mat
    double *chunk_part = nullptr;  // n_chunks*2 partial sums
    // S assembly: static (objective) part + dynamic slots
    int obj_mat = -1;              // index of the objective in the sparse list, -1 if C is not sparse
    double *triuS_static = nullptr;  // nnzT: contribution of the objective matrix (unit y)
    double S_static_scale = 0.0;     // y_{m+1} the static part of S currently carries
    bool S_static_valid = false;
    bool S_current = false;          // S (full pattern) matches the device y / was uploaded by the caller
    i64 n_dyn = 0;                 // triu slots with at least one non-objective contributor
    int *dyn_slot = nullptr;       // n_dyn: triu slot
    int *dyn_ptr = nullptr;        // n_dyn+1 into dyn_mat/dyn_val
    int *dyn_gid = nullptr;        // contributors: global slot of y
    double *dyn_val = nullptr;     //               nzval_one
    int *dyn_pos_a = nullptr, *dyn_pos_b = nullptr;  // n_dyn: the (row,col) and (col,row) slots of the full pattern
    // objective-split hot path: static objective values on the full pattern, dynamic pattern as CSR
    double *Cfull = nullptr;       // nnzF: C's value at every full-pattern slot (0 where C has no entry)
    // value-free gather pass (gradient.cu, grad_obj_spmm): every off-diagonal Cfull value is the same v = +-2^k (unweighted
    // MaxCut: 0.25), so C*X = v * (pattern*X with C_ii / v on the diagonal), bit for bit; set by pre_build
    double vf_val = 0.0;           // v, 0 = C is not of that form
    double *vf_diag = nullptr;     // n: C_ii / v (0 where the pattern has no diagonal entry)
    int obj_value_free = 1;        // sdplrp_set_option "obj_value_free": 0 = always read Cfull (A/B, tests)
    double *dynS = nullptr;        // n_dyn: constraint part of S at the dynamic slots (per iteration)
    i64 n_dynF = 0;                // dynamic slots of the full pattern
    int *dynrow_ptr = nullptr;     // n+1
    int *dynrow_col = nullptr;     // n_dynF
    int *dynrow_src = nullptr;     // n_dynF -> index into dynS
    int *dyn_diag = nullptr;       // n: index into dynS of the dynamic DIAGONAL slot of row i, -1 if none (dynrow_* holds only
                                   //    the off-diagonal dynamic slots: the diagonal part of S_dyn*R is a row scaling)
    // constraints that are a single diagonal entry (Diag(X) = 1 of MaxCut / cut-norm / bisection ...), as per-row lists in
    // internal row order: their sampled dots are a streaming pass over the factor rows (aop.cu, k_A_rowc)
    i64 n_sd = 0;
    int *rowc_ptr = nullptr;       // n+1   constraint p of row i: rowc_ptr[i] <= p < rowc_ptr[i+1]; p IS its internal slot
    double *rowc_val = nullptr;    // n_sd  its value (nzval_one == nzval_two on the diagonal)
    int *cperm = nullptr;          // m+1   internal slot of reference constraint g (slot m = objective, fixed)
    int *dyn_nsd_end = nullptr;    // n_dyn end of the contributors that are NOT single-diagonal-entry constraints
    i64 n_dyn_nsd = 0;             // their total number (0 for MaxCut-type problems: the hot loop then skips S_dyn)
    unsigned char *sd_flag = nullptr;  // nA: matrix handled by the row lists
    RowClasses full_cls, dyn_cls;  // row bins of the full / dynamic pattern
    TileLayout full_long, dyn_long; // rows of the third class cut into kRowWarpMax-nonzero chunks (gradient.cu)
    double *tile_scratch = nullptr; // chunk partial sums, max(n_chunks) x r
    i64 tile_scratch_len = 0;
    double *CR = nullptr, *CD = nullptr;  // n x r: C*R (recurrence) and C*D
    bool CR_valid = false, CD_valid = false;
    i64 state_cap = 0;             // doubles per factor array of the current allocation (sdplrp_set_rank reuses it when nothing changed)
    bool ls_valid = false;         // A_RD / A_DD (and CD) belong to the current R and D
    bool fused_tail = true;        // sdplrp_step_g may use the fused row pass

    // low-rank matrices
    std::vector<LowRank> lr;
    double *lr_tmp = nullptr;  // r*s_max*2 scratch (XB products)
    i64 lr_tmp_len = 0;

    // vectors
    double *b = nullptr, *lambda = nullptr, *lambda_ub = nullptr, *pvio_lb = nullptr;
    double *y = nullptr, *pvio_raw = nullptr, *A_RD = nullptr, *A_DD = nullptr, *A_out = nullptr;
    double *pvio_raw_alt = nullptr;  // second residual buffer: the fused step/gradient pass reads one and writes the other
    double sigma = 2.0;
    double y_obj = 0.0;  // host copy of y[m] (coefficient of the objective in S)

    // dense state
    int r = 0, hist = 0, latest = 0;  // latest is 1-based like the reference
    double *R = nullptr, *G = nullptr, *D = nullptr, *W0 = nullptr, *W1 = nullptr;
    double *Sh[kMaxHist] = {nullptr}, *Yh[kMaxHist] = {nullptr};
    // coefficient-space L-BFGS (lbfgs.cu): Gram matrix of [s_j, y_j, g], probe-row scratch, coefficients
    int lbfgs_kernel = 1;          // 0 = literal vector two-loop, 1 = coefficient two-loop on directly computed dots
    double *lb_small = nullptr;    // kLbSmallLen doubles
    bool gram_pairs_valid = false, gram_g_valid = false;
    int gram_prestored = -1;       // slot whose y was overwritten by the y = -g pre-store since the last update

    // reduction plumbing
    double *dscal = nullptr;      // SC_COUNT device scalars
    double *hscal = nullptr;      // pinned mirror
    double *partials = nullptr;   // kRedBlocks * kMaxRedK (+ chunked extras)
    unsigned *ticket = nullptr;   // last-block-done counters
    // section profiling (CUDA events on `stream`)
    bool prof = false;
    std::vector<cudaEvent_t> ev_free;
    struct Pending { int sec; cudaEvent_t a, b; };
    std::vector<Pending> ev_pending;
    double sec_ms[SDPLRP_SEC_COUNT] = {0};
    i64 sec_cnt[SDPLRP_SEC_COUNT] = {0};
    // Lanczos workspace
    double *lz_v = nullptr, *lz_w = nullptr, *lz_vp = nullptr, *lz_ab = nullptr;
    i64 lz_ab_len = 0;
    double *lz_basis = nullptr;
    i64 lz_basis_len = 0;
    RoundingState rnd;
};

#define CUDA_TRY(h, call)                                                                      \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                    \
            return SDPLRP_ERR_CUDA;                                                            \
        }                                                                                      \
    } while (0)

#define SDP_CHECK(expr)                        \
    do {                                       \
        int32_t rc__ = (expr);                 \
        if (rc__ != SDPLRP_OK) return rc__;    \
    } while (0)

#define KLAUNCH(h) ((h)->launches++)

static inline int32_t fail(sdplrp_handle *h, int32_t code, const std::string &msg) {
    h->err = msg;
    return code;
}

template <typename T>
static inline int32_t dev_alloc(sdplrp_handle *h, T **p, i64 count) {
    if (*p) { cudaFree(*p); *p = nullptr; }
    if (count <= 0) count = 1;
    CUDA_TRY(h, cudaMalloc((void **)p, (size_t)count * sizeof(T)));
    return SDPLRP_OK;
}
template <typename T>
static inline void dev_free(T **p) {
    if (*p) { cudaFree(*p); *p = nullptr; }
}

static inline int grid_for(i64 work_items, int per_block, int max_blocks = 1 << 30) {
    i64 g = (work_items + per_block - 1) / per_block;
    if (g < 1) g = 1;
    if (g > max_blocks) g = max_blocks;
    return (int)g;
}

// ---------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum K per-thread values over the CTA (blockDim.x multiple of 32, <= 1024).
// Result valid in thread 0.
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K]) {
    __shared__ double sm[K][32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < K; k++) v[k] = warp_sum(v[k]);
    __syncthreads();  // protect sm across repeated calls
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < K; k++) sm[k][wid] = v[k];
    }
    __syncthreads();
    if (wid == 0) {
#pragma unroll
        for (int k = 0; k < K; k++) {
            double t = lane < nw ? sm[k][lane] : 0.0;
            v[k] = warp_sum(t);
        }
    }
}

// Deterministic grid reduction: every CTA deposits its K sums, the last CTA to
// arrive (ticket) adds all deposits in a fixed order and calls `fin(sums)`.
// out-of-kernel state: partials[gridDim.x*K], *ticket == 0 on entry and exit.
template <int K, typename Fin>
__device__ __forceinline__ void grid_sum_finalize(double (&v)[K], double *partials, unsigned *ticket, Fin fin) {
    block_sum<K>(v);
    __shared__ bool is_last;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; k++) partials[(size_t)blockIdx.x * K + k] = v[k];
        __threadfence();
        unsigned t = atomicAdd(ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double s[K];
#pragma unroll
        for (int k = 0; k < K; k++) s[k] = 0.0;
        for (unsigned bI = threadIdx.x; bI < gridDim.x; bI += blockDim.x) {
#pragma unroll
            for (int k = 0; k < K; k++) s[k] += __ldcg(&partials[(size_t)bI * K + k]);
        }
        block_sum<K>(s);
        if (threadIdx.x == 0) {
            fin(s);
            *ticket = 0u;
        }
    }
}

// 128-bit read-only loads of two doubles
__device__ __forceinline__ double2 ldg2(const double *p) { return __ldg(reinterpret_cast<const double2 *>(p)); }

// host-visible kernels' launcher prototypes (one TU per subsystem) -----------
int32_t pre_build(sdplrp_handle *h, i64 n, i64 m, i64 nA, const int64_t *mat_off, const int64_t *I,
                  const int64_t *J, const double *V, const int64_t *gids, bool triplets_on_device = false);
int32_t pre_export(sdplrp_handle *h, int64_t *triu_colptr, int64_t *triu_rowval, int64_t *matptr,
                   int64_t *nzind, double *one, double *two, int64_t *full_colptr, int64_t *full_rowval,
                   int64_t *mapped);
void pre_free(sdplrp_handle *h);
void round_free(sdplrp_handle *h);   // rounding buffers (rounding.cu)

// A passes (aop.cu)
int32_t aop_uu(sdplrp_handle *h, const double *U, double *out_dev);                    // out = A(UU')
int32_t aop_uv(sdplrp_handle *h, const double *U, const double *V, double *out_dev);  // out = A((UV'+VU')/2)
int32_t aop_linesearch(sdplrp_handle *h, bool skip_objective);                         // A_RD (x2), A_DD fused
int32_t aop_uu_skip(sdplrp_handle *h, const double *U, double *out_dev, bool skip_objective);

int32_t lr_project(sdplrp_handle *h, const LowRank &L, const double *X, double *dst);  // dst[k*r+i] = (X'B)[i,k]
int32_t lr_scratch(sdplrp_handle *h);

// gradient (gradient.cu)
int32_t grad_form_y(sdplrp_handle *h);                          // copy2y_lambda_sub_pvio!
int32_t grad_assemble_S(sdplrp_handle *h);                      // At_preprocess! from device y
int32_t grad_spmm(sdplrp_handle *h, const double *X, double *Y, double scale, bool want_norm);  // Y = scale*X*S (+low rank)
int32_t grad_spmm_sparse(sdplrp_handle *h, const double *X, double *Y, double scale);           // Y = scale*X*S, sparse part only
int32_t grad_obj_spmm(sdplrp_handle *h, const double *X, double *Y, const double *Z, double *sums6);  // Y = C*X, sums <X,Y>, <X,Z>
inline bool obj_value_free(const sdplrp_handle *h) { return h->obj_value_free && h->vf_val != 0.0; }  // grad_obj_spmm skips Cfull
int32_t grad_obj_slots(sdplrp_handle *h, const double *sums6, double *a_rd_m, double *a_dd_m);
int32_t grad_hot(sdplrp_handle *h);                             // G = 2*(y_obj*CR + S_dyn*R + low rank), ||G||^2
int32_t grad_step_fused(sdplrp_handle *h, double alpha);        // step + y + gradient + both norms in one row pass
int32_t vec_tail_rest(sdplrp_handle *h, double alpha, const double *raw_in, double *raw_out, double *pn2_out);
int32_t grad_spmv(sdplrp_handle *h, const double *x, double *y, i64 ncols);                     // y = S*x (+low rank), n x ncols col-major
int32_t grad_triuS(sdplrp_handle *h, double *out_dev);          // materialise triu_sparse_S.nzval

// asynchronous tile pipeline of the gather pass (gather.cu)
bool gather_supported(const sdplrp_handle *h);
int gather_tile_size(const sdplrp_handle *h);
void gather_plan_free(GatherPlan &p);
int32_t gather_plan_build(sdplrp_handle *h, GatherPlan &p, const int *ptr_dev, i64 row_lo, i64 row_hi, int T);
int32_t gather_spmm(sdplrp_handle *h, const GatherPlan &plan, const int *ptr, const int *idx, const double *val, const double *Xg,
                    const double *X, const double *Z, double *Y, int epi, double scale, double *sums4);

i64 tile_hot_rows(const sdplrp_handle *h);   // hub prefix of a gathered factor (gradient.cu)

// m-vector kernels (vecops.cu)
int32_t vec_f_finish(sdplrp_handle *h);      // raw -= b, obj, AL value -> SC_OBJ, SC_LVAL
int32_t vec_biquadratic(sdplrp_handle *h);   // SC_BQ..SC_BQ+4
int32_t vec_commit(sdplrp_handle *h, double alpha);  // residual recurrence + obj
int32_t vec_pnorm2(sdplrp_handle *h);        // ||max(raw,lb)||^2 -> SC_PNORM2
int32_t vec_dual_update(sdplrp_handle *h);
int32_t vec_armijo(sdplrp_handle *h, const double *alphas, int k, double *L, double *slope);
int32_t vec_dual_dot(sdplrp_handle *h, double *out);  // -y[1:m]'b
int32_t vec_copy2y_lambda(sdplrp_handle *h);          // copy2y_lambda!: y_i = -lambda_i, y_{m+1} = 1
int32_t vec_dimacs_sums(sdplrp_handle *h, double *raw_norm2, double *lambda_b);  // ||raw[1:m]||^2, lambda'b

// dense BLAS-1 fusions (lbfgs.cu)
int32_t lb_dir(sdplrp_handle *h);                   // lbfgs_dir! + descent -> SC_DESCENT
int32_t lb_update(sdplrp_handle *h, double alpha);  // lbfgs_update!
int32_t lb_clear(sdplrp_handle *h);
int32_t lb_axpy(sdplrp_handle *h, double alpha, const double *x, double *y);  // y += alpha x over owned rows
int32_t lb_axpy2(sdplrp_handle *h, double alpha, const double *x1, double *y1, const double *x2, double *y2);
int32_t lb_neg_copy(sdplrp_handle *h);              // G = -G ; D = G
int32_t lb_norm2(sdplrp_handle *h, const double *x, int slot);
int32_t lb_dot(sdplrp_handle *h, const double *x, const double *y, int slot);   // dscal[slot] = <x,y> over the owned rows

// Lanczos (lanczos.cu)
int32_t lz_run(sdplrp_handle *h, i64 q, const double *v0_host, uint64_t seed, int reorth, double *alpha,
               double *beta, i64 *iters);
double tridiag_mineig_host(const double *d, const double *e, i64 k);
void dense_symeig_host(const double *A, i64 m, double *ev, double *Q);  // small dense symmetric eigenproblem (cyclic Jacobi)
// thick-restart Lanczos for the nev smallest eigenvalues of the current S (SDP_S_eigval)
int32_t lz_eigs(sdplrp_handle *h, i64 nev, i64 ncv, double tol, i64 maxiter, const double *v0_host, uint64_t seed, double *eigs,
                double *bounds, i64 *matvecs, i64 *restarts);

// multi-GPU plumbing (comm.cu); all no-ops when world == 1
int32_t comm_init(sdplrp_handle *h, const void *nccl_id);
void comm_destroy(sdplrp_handle *h);
int32_t comm_partition(sdplrp_handle *h);
void comm_mark_partial(sdplrp_handle *h, int mat_id);
void comm_mark_full(sdplrp_handle *h, int mat_id);
int32_t comm_require_full(sdplrp_handle *h, int mat_id);
int32_t comm_gather_rows(sdplrp_handle *h, double *p, int mat_id);
int32_t comm_reduce_mvec(sdplrp_handle *h, double *v1, double *v2);   // shared slots [n_sd, m] only
int32_t comm_gather_rowvec(sdplrp_handle *h, double *v);              // every rank's owned rows of an n-vector (internal order) to every rank
int32_t comm_gather_rowbytes(sdplrp_handle *h, void *v, size_t row_bytes);  // the same for row_bytes bytes per row, byte-exact
int32_t comm_gather_cvec(sdplrp_handle *h, double *v);                // make every per-row-constraint slot current on every rank
int32_t comm_reduce_scalars(sdplrp_handle *h, int slot, int count);
int32_t comm_check_same(sdplrp_handle *h, unsigned long long value, const char *what);  // error unless all ranks pass the same value
int32_t comm_reduce_ptr(sdplrp_handle *h, double *p, int count);
int32_t comm_step_R(sdplrp_handle *h, double alpha);
int32_t comm_allgather_bytes(sdplrp_handle *h, const void *send, void *recv, size_t bytes);       // recv = world x bytes
// halo exchange (comm.cu): pack the rows the peers gather from X (n x r, internal labels, own block valid), start the two
// class exchanges on the comm stream; halo_wait makes the compute stream wait for one class (its exposed time is the
// "comm" section)
int32_t halo_build(sdplrp_handle *h);       // preprocess.cu
void halo_free(sdplrp_handle *h);
bool halo_active(const sdplrp_handle *h);
int32_t halo_begin(sdplrp_handle *h, const double *X);
int32_t halo_wait(sdplrp_handle *h, int klass);

// reference order <-> internal order (perm.cu)
int32_t perm_stage(sdplrp_handle *h, i64 len);
int32_t perm_upload(sdplrp_handle *h, double *dst_dev, const double *src_host, i64 ncols, bool row_major);
int32_t perm_download(sdplrp_handle *h, const double *src_dev, double *dst_host, i64 ncols, bool row_major);
int32_t perm_upload_slice(sdplrp_handle *h, double *dst_dev, const double *src_host, i64 ncols);      // reference rows [rank*S, (rank+1)*S), S = ceil(n/world)
int32_t perm_download_slice(sdplrp_handle *h, const double *src_dev, double *dst_host, i64 ncols);
int32_t comm_allgather_inplace(sdplrp_handle *h, double *buf, size_t cnt);
int32_t perm_device(sdplrp_handle *h, double *dst, const double *src, i64 ncols, bool row_major, bool to_internal);
int32_t perm_slots_upload(sdplrp_handle *h, double *dst_dev, const double *src_host, i64 len);
int32_t perm_slots_download(sdplrp_handle *h, const double *src_dev, double *dst_host, i64 len);
int32_t perm_cvec_upload(sdplrp_handle *h, double *dst_dev, const double *src_host, i64 len);     // m or m+1 doubles
int32_t perm_cvec_download(sdplrp_handle *h, const double *src_dev, double *dst_host, i64 len);

// section timers (api.cu)
cudaEvent_t prof_begin(sdplrp_handle *h);
void prof_end(sdplrp_handle *h, int sec, cudaEvent_t a);
struct SectionScope {
    sdplrp_handle *h; int sec; cudaEvent_t a;
    SectionScope(sdplrp_handle *h_, int sec_) : h(h_), sec(sec_), a(h_->prof ? prof_begin(h_) : nullptr) {}
    ~SectionScope() { if (a) prof_end(h, sec, a); }
};

// scalar plumbing (api.cu)
int32_t fetch_scalars(sdplrp_handle *h, int first, int count);  // dscal -> hscal, synchronises
