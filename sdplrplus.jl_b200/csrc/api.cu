// api.cu -- the extern "C" entry points of libsdplrp_b200.so (see
// include/sdplrp_b200.h for the contract and the reference file:line each one
// replaces).  There is no CPU fallback: without a CUDA device sdplrp_create
// fails with SDPLRP_ERR_NO_DEVICE.
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include "common.cuh"

static const char *kNoHandle = "null handle";

#define REQUIRE_H(h) \
    if (!(h)) return SDPLRP_ERR_ARG
#define REQUIRE_PRE(h)                                                                   \
    if (!(h)->preprocessed) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_preprocess first")
#define REQUIRE_RANK(h)                                                                  \
    if ((h)->r <= 0) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_set_rank first")

int32_t fetch_scalars(sdplrp_handle *h, int first, int count) {
    CUDA_TRY(h, cudaMemcpyAsync(h->hscal + first, h->dscal + first, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return SDPLRP_OK;
}

cudaEvent_t prof_begin(sdplrp_handle *h) {
    cudaEvent_t e = nullptr;
    if (!h->ev_free.empty()) { e = h->ev_free.back(); h->ev_free.pop_back(); }
    else if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    cudaEventRecord(e, h->stream);
    return e;
}
void prof_end(sdplrp_handle *h, int sec, cudaEvent_t a) {
    cudaEvent_t e = nullptr;
    if (!h->ev_free.empty()) { e = h->ev_free.back(); h->ev_free.pop_back(); }
    else if (cudaEventCreate(&e) != cudaSuccess) { h->ev_free.push_back(a); return; }
    cudaEventRecord(e, h->stream);
    h->ev_pending.push_back({sec, a, e});
}
static void prof_collect(sdplrp_handle *h) {
    for (auto &p : h->ev_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) { h->sec_ms[p.sec] += ms; h->sec_cnt[p.sec] += 1; }
        h->ev_free.push_back(p.a); h->ev_free.push_back(p.b);
    }
    h->ev_pending.clear();
}

static double *mat_ptr(sdplrp_handle *h, int id) {
    switch (id) {
    case SDPLRP_MAT_R: return h->R;
    case SDPLRP_MAT_G: return h->G;
    case SDPLRP_MAT_D: return h->D;
    case SDPLRP_MAT_W0: return h->W0;
    case SDPLRP_MAT_W1: return h->W1;
    case SDPLRP_MAT_CR: return h->CR;   // introspection: the C*R recurrence of the objective split (null without a sparse C)
    case SDPLRP_MAT_CD: return h->CD;
    default: break;
    }
    if (id >= SDPLRP_MAT_S0 && id < SDPLRP_MAT_S0 + h->hist) return h->Sh[id - SDPLRP_MAT_S0];
    if (id >= SDPLRP_MAT_Y0 && id < SDPLRP_MAT_Y0 + h->hist) return h->Yh[id - SDPLRP_MAT_Y0];
    return nullptr;
}

static double *vec_ptr(sdplrp_handle *h, int id, i64 *len) {
    switch (id) {
    case SDPLRP_VEC_LAMBDA: *len = h->m; return h->lambda;
    case SDPLRP_VEC_LAMBDA_UB: *len = h->m; return h->lambda_ub;
    case SDPLRP_VEC_B: *len = h->m; return h->b;
    case SDPLRP_VEC_PVIO_RAW: *len = h->m + 1; return h->pvio_raw;
    case SDPLRP_VEC_Y: *len = h->m + 1; return h->y;
    case SDPLRP_VEC_PVIO_LB: *len = h->m; return h->pvio_lb;
    case SDPLRP_VEC_A_RD: *len = h->m + 1; return h->A_RD;
    case SDPLRP_VEC_A_DD: *len = h->m + 1; return h->A_DD;
    case SDPLRP_VEC_S_NZVAL: *len = h->nnzF; return h->S;
    default: return nullptr;
    }
}

__global__ void k_fill(i64 len, double v, double *__restrict__ x) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < len; i += (i64)gridDim.x * blockDim.x) x[i] = v;
}
// `ineq` is in reference constraint order, ub / lb in the internal order (cperm)
__global__ void k_bounds(i64 m, const unsigned char *__restrict__ ineq, const int *__restrict__ cperm, double *__restrict__ ub,
                         double *__restrict__ lb) {
    for (i64 g = blockIdx.x * (i64)blockDim.x + threadIdx.x; g < m; g += (i64)gridDim.x * blockDim.x) {
        const bool q = ineq && ineq[g];
        const i64 c = cperm ? cperm[g] : g;
        ub[c] = q ? 0.0 : INFINITY;   // src/structs.jl:228
        lb[c] = q ? 0.0 : -INFINITY;  // src/structs.jl:249
    }
}

extern "C" {

int32_t sdplrp_version(void) { return 100; }

const char *sdplrp_error_string(int32_t code) {
    switch (code) {
    case SDPLRP_OK: return "ok";
    case SDPLRP_ERR_CUDA: return "CUDA runtime error";
    case SDPLRP_ERR_ARG: return "bad argument";
    case SDPLRP_ERR_STATE: return "call order violated";
    case SDPLRP_ERR_ASYMMETRIC: return "constraint matrix not stored symmetric";
    case SDPLRP_ERR_NCCL: return "NCCL error";
    case SDPLRP_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
    case SDPLRP_ERR_LINESEARCH: return "line search slope is positive";
    default: return "unknown error";
    }
}

const char *sdplrp_last_error(sdplrp_handle *h) { return h ? h->err.c_str() : kNoHandle; }

int32_t sdplrp_create(int32_t device, int32_t rank, int32_t world, const void *nccl_id, sdplrp_handle **out) {
    if (!out) return SDPLRP_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return SDPLRP_ERR_NO_DEVICE;
    if (device < 0 || device >= ndev || world < 1 || rank < 0 || rank >= world) return SDPLRP_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return SDPLRP_ERR_CUDA;
    sdplrp_handle *h = new sdplrp_handle();
    h->device = device; h->rank = rank; h->world = world;
    if (const char *e = getenv("SDPLRP_RELABEL")) h->relabel_mode = atoi(e) < 0 ? -1 : (atoi(e) > 0 ? 1 : 0);
    if (const char *e = getenv("SDPLRP_HOT_ROWS")) h->hot_rows = atoll(e);
    if (const char *e = getenv("SDPLRP_LBFGS_KERNEL")) h->lbfgs_kernel = atoi(e);
    if (const char *e = getenv("SDPLRP_SPMM_UNROLL")) h->spmm_unroll = atoi(e);
    if (const char *e = getenv("SDPLRP_SPMM_G0")) h->spmm_g0 = atoi(e);
    if (const char *e = getenv("SDPLRP_LANCZOS_DIST")) h->lanczos_dist = atoi(e) > 0 ? 1 : 0;
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return SDPLRP_ERR_CUDA; }
    {   // side streams of the row classes of a gather pass (SDPLRP_CLASS_STREAMS=0: everything on the one stream)
        const char *e = getenv("SDPLRP_CLASS_STREAMS");
        if (!e || atoi(e) != 0) {
            bool ok = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) == cudaSuccess;
            for (int c = 0; c < 2 && ok; c++)
                ok = cudaStreamCreateWithFlags(&h->class_streams[c], cudaStreamNonBlocking) == cudaSuccess &&
                     cudaEventCreateWithFlags(&h->ev_join[c], cudaEventDisableTiming) == cudaSuccess;
            if (!ok) { cudaGetLastError(); h->class_streams[0] = nullptr; }
        }
    }
    // L2 fetch granularity (cudaLimitMaxL2FetchGranularity: 32 / 64 / 128 bytes): the gather pass reads 80-byte rows at
    // random, so everything the memory system fetches beyond the touched sectors is waste
    if (const char *e = getenv("SDPLRP_L2_FETCH")) {
        if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoll(e)) != cudaSuccess) cudaGetLastError();
    }
    // Experiment knob only: an L2 set-aside for evict_last lines (cudaLimitPersistingL2CacheSize).  Measured on C5: a
    // set-aside of the maximum 79 MB slows every streaming kernel 1.8x (1.34 -> 2.46 ms for an 8.8 GB pass) and does
    // not speed the gather pass up, so the library leaves the device default alone unless asked to.
    if (const char *e = getenv("SDPLRP_L2_PERSIST_MB")) {
        int maxp = 0;
        cudaDeviceGetAttribute(&maxp, cudaDevAttrMaxPersistingL2CacheSize, device);
        const size_t want = std::min<size_t>((size_t)maxp, (size_t)atoll(e) << 20);
        if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) h->l2_persist_bytes = (i64)want;
        else cudaGetLastError();
    }
    bool ok = cudaMalloc((void **)&h->dscal, SC_COUNT * sizeof(double)) == cudaSuccess &&
              cudaMallocHost((void **)&h->hscal, SC_COUNT * sizeof(double)) == cudaSuccess &&
              cudaMalloc((void **)&h->partials, (size_t)kPartialsLen * sizeof(double)) == cudaSuccess &&
              cudaMalloc((void **)&h->ticket, 4 * sizeof(unsigned)) == cudaSuccess;
    if (ok) ok = cudaMemset(h->dscal, 0, SC_COUNT * sizeof(double)) == cudaSuccess && cudaMemset(h->ticket, 0, 4 * sizeof(unsigned)) == cudaSuccess;
    if (!ok) { sdplrp_destroy(h); return SDPLRP_ERR_CUDA; }
    memset(h->hscal, 0, SC_COUNT * sizeof(double));
    if (world > 1) {
        int32_t rc = comm_init(h, nccl_id);
        if (rc != SDPLRP_OK) { sdplrp_destroy(h); return rc; }
    }
    *out = h;
    return SDPLRP_OK;
}

// doubles to allocate for an n x r factor: with equal row blocks the last block is padded to block_rows rows so that the
// in-place all-gather (comm.cu) stays inside the allocation
static i64 mat_capacity(const sdplrp_handle *h, int r) {
    const i64 rows = h->equal_blocks ? std::max<i64>(h->n, (i64)h->world * h->block_rows) : h->n;
    return rows * (i64)r;
}

static void free_state(sdplrp_handle *h) {
    dev_free(&h->R); dev_free(&h->G); dev_free(&h->D); dev_free(&h->W0); dev_free(&h->W1);
    dev_free(&h->CR); dev_free(&h->CD);
    h->CR_valid = h->CD_valid = false;
    for (int j = 0; j < kMaxHist; j++) { dev_free(&h->Sh[j]); dev_free(&h->Yh[j]); }
    dev_free(&h->lb_small);
    h->gram_pairs_valid = h->gram_g_valid = false; h->gram_prestored = -1;
    dev_free(&h->lr_tmp); h->lr_tmp_len = 0;
    h->r = 0; h->hist = 0;
    h->state_cap = 0;
}

static void free_problem(sdplrp_handle *h) {
    pre_free(h);
    for (LowRank &L : h->lr) { dev_free(&L.dB); dev_free(&L.dD); }
    h->lr.clear();
    dev_free(&h->b); dev_free(&h->lambda); dev_free(&h->lambda_ub); dev_free(&h->pvio_lb);
    dev_free(&h->y); dev_free(&h->pvio_raw); dev_free(&h->pvio_raw_alt); dev_free(&h->A_RD); dev_free(&h->A_DD); dev_free(&h->A_out);
    dev_free(&h->lz_v); dev_free(&h->lz_w); dev_free(&h->lz_vp); dev_free(&h->lz_ab); dev_free(&h->lz_basis);
    h->lz_ab_len = 0; h->lz_basis_len = 0;
    dev_free(&h->stage); h->stage_len = 0;
}

int32_t sdplrp_destroy(sdplrp_handle *h) {
    if (!h) return SDPLRP_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    comm_destroy(h);
    prof_collect(h);
    for (cudaEvent_t e : h->ev_free) cudaEventDestroy(e);
    h->ev_free.clear();
    free_state(h);
    free_problem(h);
    dev_free(&h->dscal); dev_free(&h->partials); dev_free(&h->ticket);
    if (h->hscal) cudaFreeHost(h->hscal);
    for (int c = 0; c < 2; c++) {
        if (h->class_streams[c]) cudaStreamDestroy(h->class_streams[c]);
        if (h->ev_join[c]) cudaEventDestroy(h->ev_join[c]);
    }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return SDPLRP_OK;
}

int32_t sdplrp_synchronize(sdplrp_handle *h) {
    REQUIRE_H(h);
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return SDPLRP_OK;
}

void *sdplrp_stream(sdplrp_handle *h) { return h ? (void *)h->stream : nullptr; }

static int32_t preprocess_common(sdplrp_handle *h, int64_t n, int64_t m, int64_t nA, const int64_t *mat_off, const int64_t *I,
                                 const int64_t *J, const double *V, const int64_t *gids, bool triplets_on_device);

int32_t sdplrp_preprocess(sdplrp_handle *h, int64_t n, int64_t m, int64_t nA, const int64_t *mat_off, const int64_t *I,
                          const int64_t *J, const double *V, const int64_t *gids) {
    return preprocess_common(h, n, m, nA, mat_off, I, J, V, gids, false);
}

// the same with I, J, V in device memory of the handle's GPU (SURVEY 8f/f2: problem generators that build on the device)
int32_t sdplrp_preprocess_device(sdplrp_handle *h, int64_t n, int64_t m, int64_t nA, const int64_t *mat_off, const int64_t *d_I,
                                 const int64_t *d_J, const double *d_V, const int64_t *gids) {
    REQUIRE_H(h);
    if (nA > 0 && mat_off && mat_off[nA] > 0) {
        if (!d_I || !d_J || !d_V) return fail(h, SDPLRP_ERR_ARG, "preprocess_device: null triplet arrays");
        cudaPointerAttributes at;
        const void *ptrs[3] = {d_I, d_J, d_V};
        for (const void *p : ptrs) {
            if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device != h->device) {
                cudaGetLastError();
                return fail(h, SDPLRP_ERR_ARG, "preprocess_device: I, J, V must be device memory of the handle's GPU");
            }
        }
    }
    return preprocess_common(h, n, m, nA, mat_off, d_I, d_J, d_V, gids, true);
}

static int32_t preprocess_common(sdplrp_handle *h, int64_t n, int64_t m, int64_t nA, const int64_t *mat_off, const int64_t *I,
                                 const int64_t *J, const double *V, const int64_t *gids, bool triplets_on_device) {
    REQUIRE_H(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    free_state(h);
    free_problem(h);
    if (nA > 0 && (!mat_off || !gids)) return fail(h, SDPLRP_ERR_ARG, "preprocess: null arrays");
    int32_t rc = pre_build(h, n, m, nA, mat_off, I, J, V, gids, triplets_on_device);
    if (rc != SDPLRP_OK && rc != SDPLRP_ERR_ASYMMETRIC) return rc;
    // vectors of SolverVars / SDPData
    SDP_CHECK(dev_alloc(h, &h->b, m)); SDP_CHECK(dev_alloc(h, &h->lambda, m)); SDP_CHECK(dev_alloc(h, &h->lambda_ub, m));
    SDP_CHECK(dev_alloc(h, &h->pvio_lb, m)); SDP_CHECK(dev_alloc(h, &h->y, m + 1)); SDP_CHECK(dev_alloc(h, &h->pvio_raw, m + 1)); SDP_CHECK(dev_alloc(h, &h->pvio_raw_alt, m + 1));
    SDP_CHECK(dev_alloc(h, &h->A_RD, m + 1)); SDP_CHECK(dev_alloc(h, &h->A_DD, m + 1)); SDP_CHECK(dev_alloc(h, &h->A_out, m + 1));
    cudaStream_t st = h->stream;
    CUDA_TRY(h, cudaMemsetAsync(h->b, 0, (size_t)std::max<i64>(m, 1) * 8, st));
    CUDA_TRY(h, cudaMemsetAsync(h->lambda, 0, (size_t)std::max<i64>(m, 1) * 8, st));
    CUDA_TRY(h, cudaMemsetAsync(h->y, 0, (size_t)(m + 1) * 8, st));
    CUDA_TRY(h, cudaMemsetAsync(h->pvio_raw, 0, (size_t)(m + 1) * 8, st));
    CUDA_TRY(h, cudaMemsetAsync(h->pvio_raw_alt, 0, (size_t)(m + 1) * 8, st));
    CUDA_TRY(h, cudaMemsetAsync(h->A_RD, 0, (size_t)(m + 1) * 8, st));
    CUDA_TRY(h, cudaMemsetAsync(h->A_DD, 0, (size_t)(m + 1) * 8, st));
    CUDA_TRY(h, cudaMemsetAsync(h->A_out, 0, (size_t)(m + 1) * 8, st));
    k_bounds<<<grid_for(m, 256, kRedBlocks), 256, 0, st>>>(m, nullptr, h->cperm, h->lambda_ub, h->pvio_lb);
    KLAUNCH(h);
    CUDA_TRY(h, cudaStreamSynchronize(st));
    h->y_obj = 0.0;
    SDP_CHECK(comm_partition(h));
    SDP_CHECK(halo_build(h));   // multi-GPU: local pattern + halo lists of the gather pass
    return rc;
}

// multi-GPU introspection: {active, own rows, own nonzeros, hub ghosts, tail ghosts, hub rows sent, tail rows sent}
int32_t sdplrp_halo_stats(sdplrp_handle *h, int64_t out[7]) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    const HaloPlan &p = h->halo;
    out[0] = halo_active(h) ? 1 : 0; out[1] = p.nloc; out[2] = p.lnnz; out[3] = p.n_ghost[0]; out[4] = p.n_ghost[1];
    out[5] = p.n_send[0]; out[6] = p.n_send[1];
    return SDPLRP_OK;
}

int32_t sdplrp_value_free_weight(sdplrp_handle *h, double *v) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    if (!v) return fail(h, SDPLRP_ERR_ARG, "value_free_weight: null pointer");
    *v = obj_value_free(h) ? h->vf_val : 0.0;
    return SDPLRP_OK;
}

int32_t sdplrp_pattern_sizes(sdplrp_handle *h, int64_t *nnzT, int64_t *nnzF, int64_t *Ec) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    if (nnzT) *nnzT = h->nnzT;
    if (nnzF) *nnzF = h->nnzF;
    if (Ec) *Ec = h->Ec;
    return SDPLRP_OK;
}

int32_t sdplrp_pattern_export(sdplrp_handle *h, int64_t *triu_colptr, int64_t *triu_rowval, int64_t *matptr, int64_t *nzind,
                              double *nzval_one, double *nzval_two, int64_t *full_colptr, int64_t *full_rowval,
                              int64_t *mappedto_triu) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    return pre_export(h, triu_colptr, triu_rowval, matptr, nzind, nzval_one, nzval_two, full_colptr, full_rowval, mappedto_triu);
}

int32_t sdplrp_add_symlowrank(sdplrp_handle *h, int64_t global_id, int64_t s, const double *B, const double *D) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    if (global_id < 1 || global_id > h->m + 1 || s < 1 || !B || !D) return fail(h, SDPLRP_ERR_ARG, "add_symlowrank: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    LowRank L;
    int gid_internal = (int)(global_id - 1);
    CUDA_TRY(h, cudaMemcpy(&gid_internal, h->cperm + (global_id - 1), sizeof(int), cudaMemcpyDeviceToHost));  // internal constraint slot
    L.gid = gid_internal; L.s = s; L.dB = nullptr; L.dD = nullptr;
    SDP_CHECK(dev_alloc(h, &L.dB, h->n * s));
    SDP_CHECK(dev_alloc(h, &L.dD, s));
    h->lr.push_back(L);  // owned by the handle from here on (freed by free_problem even if a copy fails)
    SDP_CHECK(perm_upload(h, L.dB, B, s, false));  // rows of B follow the internal vertex order
    CUDA_TRY(h, cudaMemcpy(L.dD, D, (size_t)s * 8, cudaMemcpyHostToDevice));
    return SDPLRP_OK;
}

int32_t sdplrp_set_problem(sdplrp_handle *h, const double *b, const uint8_t *is_ineq) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    const i64 m = h->m;
    if (m > 0 && !b) return fail(h, SDPLRP_ERR_ARG, "set_problem: null b");
    if (m > 0) SDP_CHECK(perm_cvec_upload(h, h->b, b, m));
    unsigned char *dq = nullptr;
    h->has_ineq = false;
    if (is_ineq) for (i64 i = 0; i < m; i++) h->has_ineq |= is_ineq[i] != 0;
    if (is_ineq && m > 0) {
        CUDA_TRY(h, cudaMalloc((void **)&dq, (size_t)m));
        CUDA_TRY(h, cudaMemcpy(dq, is_ineq, (size_t)m, cudaMemcpyHostToDevice));
    }
    k_bounds<<<grid_for(m, 256, kRedBlocks), 256, 0, h->stream>>>(m, dq, h->cperm, h->lambda_ub, h->pvio_lb);
    KLAUNCH(h);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (dq) cudaFree(dq);
    CUDA_TRY(h, e);
    return SDPLRP_OK;
}

int32_t sdplrp_set_rank(sdplrp_handle *h, int32_t r, int32_t numlbfgsvecs) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    if (r < 1 || numlbfgsvecs < 0 || numlbfgsvecs > kMaxHist) return fail(h, SDPLRP_ERR_ARG, "set_rank: bad rank / history length");
    // checked before anything is freed or launched: the sparse row kernels would fail later (r > 128 odd) or the per-row
    // constraint tile pass would get zero rows per tile (r > 256 odd, r > 512 even)
    if (!rank_supported(r))
        return fail(h, SDPLRP_ERR_ARG, "set_rank: r = " + std::to_string(r) + " is not supported (r <= " + std::to_string(SDPLRP_MAX_RANK) +
                                           ", and r <= " + std::to_string(SDPLRP_MAX_ODD_RANK) + " when r is odd)");
    CUDA_TRY(h, cudaSetDevice(h->device));
    const i64 N = mat_capacity(h, r);
    // same rank, history length and capacity as the current state (a new start point for the same problem, the e2e path of
    // bench.py): keep the 2h+5 arrays instead of paying a cudaFree + cudaMalloc for each (0.8 GB apiece at C5)
    const bool reuse = h->R && h->G && h->D && h->lb_small && h->r == r && h->hist == numlbfgsvecs && h->state_cap == N &&
                       ((h->obj_mat >= 0) == (h->CR != nullptr)) && ((h->obj_mat >= 0) == (h->CD != nullptr));
    if (reuse) {
        h->CR_valid = h->CD_valid = false;
        if (h->W0) CUDA_TRY(h, cudaMemsetAsync(h->W0, 0, (size_t)N * 8, h->stream));  // scratch ids start out zero (lazy_scratch)
        if (h->W1) CUDA_TRY(h, cudaMemsetAsync(h->W1, 0, (size_t)N * 8, h->stream));
    } else {
        free_state(h);
        SDP_CHECK(dev_alloc(h, &h->R, N)); SDP_CHECK(dev_alloc(h, &h->G, N)); SDP_CHECK(dev_alloc(h, &h->D, N));
        if (h->obj_mat >= 0) { SDP_CHECK(dev_alloc(h, &h->CR, N)); SDP_CHECK(dev_alloc(h, &h->CD, N)); }
        for (int j = 0; j < numlbfgsvecs; j++) { SDP_CHECK(dev_alloc(h, &h->Sh[j], N)); SDP_CHECK(dev_alloc(h, &h->Yh[j], N)); }
        SDP_CHECK(dev_alloc(h, &h->lb_small, kLbSmallLen));
        h->state_cap = N;
    }
    h->r = r; h->hist = numlbfgsvecs; h->latest = numlbfgsvecs;  // lbfgs_init: latest = h (src/lbfgs.jl:45)
    CUDA_TRY(h, cudaMemsetAsync(h->R, 0, (size_t)N * 8, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->G, 0, (size_t)N * 8, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->D, 0, (size_t)N * 8, h->stream));
    SDP_CHECK(lb_clear(h));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return SDPLRP_OK;
}

int32_t sdplrp_set_option(sdplrp_handle *h, const char *key, double value) {
    REQUIRE_H(h);
    if (!key) return fail(h, SDPLRP_ERR_ARG, "set_option: null key");
    const std::string k(key);
    if (k == "relabel") { h->relabel_mode = value < 0 ? -1 : (value > 0 ? 1 : 0); return SDPLRP_OK; }  // before preprocess
    if (k == "hot_rows") { h->hot_rows = (i64)value; return SDPLRP_OK; }
    if (k == "spmm_phases") { h->spmm_phases = value < 0 ? 0 : (int)value; return SDPLRP_OK; }
    if (k == "lanczos_dist") { h->lanczos_dist = value > 0 ? 1 : 0; return SDPLRP_OK; }
    if (k == "row_group_max") { h->row_group_max = std::max(1, std::min((int)value, kRowWarpMax)); return SDPLRP_OK; }   // before preprocess
    if (k == "spmm_unroll") { h->spmm_unroll = (int)value; return SDPLRP_OK; }
    if (k == "spmm_g0") { h->spmm_g0 = (int)value; return SDPLRP_OK; }
    if (k == "obj_value_free") { h->obj_value_free = value != 0 ? 1 : 0; return SDPLRP_OK; }
    if (k == "rowc_kernel") { h->rowc_kernel = value > 0 ? 1 : 0; return SDPLRP_OK; }
    if (k == "tail_ctas") { h->tail_ctas = std::max(0, std::min((int)value, 8)); return SDPLRP_OK; }
    if (k == "halo") { h->halo_mode = value < 0.5 ? 0 : (value < 1.5 ? 1 : (value < 2.5 ? 2 : 3)); return SDPLRP_OK; }
    if (k == "gather_mode") { h->gather_mode = value < 0 ? 0 : (int)value; return SDPLRP_OK; }
    if (k == "gather_tile") { h->gather_tile = (int)value; return SDPLRP_OK; }
    if (k == "gather_stages") { h->gather_stages = (int)value; return SDPLRP_OK; }
    if (k == "gather_warps") { h->gather_warps = (int)value; return SDPLRP_OK; }
    if (k == "gather_hints") { h->gather_hints = value > 0 ? 1 : 0; return SDPLRP_OK; }
    if (k == "fused_tail") { h->fused_tail = value != 0; return SDPLRP_OK; }
    if (k == "lbfgs_kernel") { h->lbfgs_kernel = (int)value; h->gram_pairs_valid = h->gram_g_valid = false; return SDPLRP_OK; }
    return fail(h, SDPLRP_ERR_ARG, "set_option: unknown key " + k);
}

int32_t sdplrp_set_sigma(sdplrp_handle *h, double sigma) { REQUIRE_H(h); h->sigma = sigma; return SDPLRP_OK; }
int32_t sdplrp_get_sigma(sdplrp_handle *h, double *sigma) { REQUIRE_H(h); *sigma = h->sigma; return SDPLRP_OK; }
int32_t sdplrp_get_obj(sdplrp_handle *h, double *obj) {
    REQUIRE_H(h);
    SDP_CHECK(fetch_scalars(h, SC_OBJ, 1));
    *obj = h->hscal[SC_OBJ];
    return SDPLRP_OK;
}

static int32_t lazy_scratch(sdplrp_handle *h, int id) {
    const i64 N = mat_capacity(h, h->r);
    if (id == SDPLRP_MAT_W0 && !h->W0) { SDP_CHECK(dev_alloc(h, &h->W0, N)); CUDA_TRY(h, cudaMemset(h->W0, 0, (size_t)N * 8)); }
    if (id == SDPLRP_MAT_W1 && !h->W1) { SDP_CHECK(dev_alloc(h, &h->W1, N)); CUDA_TRY(h, cudaMemset(h->W1, 0, (size_t)N * 8)); }
    return SDPLRP_OK;
}

int32_t sdplrp_upload_mat(sdplrp_handle *h, int32_t id, const double *src) {
    REQUIRE_H(h);
    REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lazy_scratch(h, id));
    if (id == SDPLRP_MAT_CR || id == SDPLRP_MAT_CD) return fail(h, SDPLRP_ERR_ARG, "upload_mat: CR / CD are download-only");
    double *p = mat_ptr(h, id);
    if (!p || !src) return fail(h, SDPLRP_ERR_ARG, "upload_mat: bad id");
    SDP_CHECK(perm_upload(h, p, src, h->r, true));
    comm_mark_full(h, id);
    if (id == SDPLRP_MAT_R) h->CR_valid = false;
    if (id == SDPLRP_MAT_D) { h->CD_valid = false; h->ls_valid = false; }
    if (id == SDPLRP_MAT_R) h->ls_valid = false;
    if (id == SDPLRP_MAT_G) h->gram_g_valid = false;
    if (id >= SDPLRP_MAT_S0) { h->gram_pairs_valid = false; h->gram_prestored = -1; }
    return SDPLRP_OK;
}

// several GPUs: rank q reads rows [q*S, (q+1)*S) of `src` (the caller's vertex order, S = ceil(n / world)); the slices are
// exchanged over NVLink, so every rank ends up with the WHOLE matrix while n*r/world doubles crossed its PCIe link
int32_t sdplrp_upload_mat_slice(sdplrp_handle *h, int32_t id, const double *src) {
    REQUIRE_H(h);
    REQUIRE_RANK(h);
    if (h->world <= 1) return sdplrp_upload_mat(h, id, src);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lazy_scratch(h, id));
    if (id == SDPLRP_MAT_CR || id == SDPLRP_MAT_CD) return fail(h, SDPLRP_ERR_ARG, "upload_mat: CR / CD are download-only");
    double *p = mat_ptr(h, id);
    if (!p || !src) return fail(h, SDPLRP_ERR_ARG, "upload_mat_slice: bad id");
    SDP_CHECK(perm_upload_slice(h, p, src, h->r));
    comm_mark_full(h, id);
    if (id == SDPLRP_MAT_R) { h->CR_valid = false; h->ls_valid = false; }
    if (id == SDPLRP_MAT_D) { h->CD_valid = false; h->ls_valid = false; }
    if (id == SDPLRP_MAT_G) h->gram_g_valid = false;
    if (id >= SDPLRP_MAT_S0) { h->gram_pairs_valid = false; h->gram_prestored = -1; }
    return SDPLRP_OK;
}

// several GPUs: rank q writes rows [q*S, (q+1)*S) of `dst`; the union over the ranks is the matrix
int32_t sdplrp_download_mat_slice(sdplrp_handle *h, int32_t id, double *dst) {
    REQUIRE_H(h);
    REQUIRE_RANK(h);
    if (h->world <= 1) return sdplrp_download_mat(h, id, dst);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lazy_scratch(h, id));
    double *p = mat_ptr(h, id);
    if (!p || !dst) return fail(h, SDPLRP_ERR_ARG, "download_mat_slice: bad id");
    SDP_CHECK(comm_gather_rows(h, p, id));   // the rows of the other ranks over NVLink
    return perm_download_slice(h, p, dst, h->r);
}

int32_t sdplrp_download_mat(sdplrp_handle *h, int32_t id, double *dst) {
    REQUIRE_H(h);
    REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lazy_scratch(h, id));
    double *p = mat_ptr(h, id);
    if (!p || !dst) return fail(h, SDPLRP_ERR_ARG, "download_mat: bad id");
    SDP_CHECK(comm_gather_rows(h, p, id));
    return perm_download(h, p, dst, h->r, true);
}

int32_t sdplrp_upload_vec(sdplrp_handle *h, int32_t id, const double *src, int64_t len) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    i64 want = 0;
    double *p = vec_ptr(h, id, &want);
    if (!p || !src || len != want) return fail(h, SDPLRP_ERR_ARG, "upload_vec: bad id or length");
    if (id == SDPLRP_VEC_S_NZVAL) {
        SDP_CHECK(perm_slots_upload(h, p, src, len));
    } else {
        SDP_CHECK(perm_cvec_upload(h, p, src, len));  // m-vectors live in the internal constraint order
    }
    if (id == SDPLRP_VEC_Y) { h->y_obj = src[h->m]; h->S_current = false; }
    if (id == SDPLRP_VEC_S_NZVAL) { h->S_static_valid = false; h->S_current = true; }
    return SDPLRP_OK;
}

int32_t sdplrp_download_vec(sdplrp_handle *h, int32_t id, double *dst, int64_t len) {
    REQUIRE_H(h);
    REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (id == SDPLRP_VEC_TRIUS_NZVAL) {
        if (len != h->nnzT || !dst) return fail(h, SDPLRP_ERR_ARG, "download_vec: bad length");
        double *tmp = nullptr;
        SDP_CHECK(dev_alloc(h, &tmp, h->nnzT));
        int32_t rc = grad_triuS(h, tmp);
        if (rc == SDPLRP_OK && len > 0) {
            cudaError_t e = cudaMemcpyAsync(dst, tmp, (size_t)len * 8, cudaMemcpyDeviceToHost, h->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
            if (e != cudaSuccess) { h->err = cudaGetErrorString(e); rc = SDPLRP_ERR_CUDA; }
        }
        cudaFree(tmp);
        return rc;
    }
    i64 want = 0;
    double *p = vec_ptr(h, id, &want);
    if (!p || !dst || len != want) return fail(h, SDPLRP_ERR_ARG, "download_vec: bad id or length");
    if (id == SDPLRP_VEC_S_NZVAL) return perm_slots_download(h, p, dst, len);
    SDP_CHECK(comm_gather_cvec(h, p));  // multi-GPU: per-row-constraint slots live on their owners
    return perm_cvec_download(h, p, dst, len);
}

// ---- seam-level operators ----------------------------------------------------
static int32_t copy_out(sdplrp_handle *h, double *dev, double *host, i64 len) {
    if (!host) return SDPLRP_OK;
    SDP_CHECK(comm_gather_cvec(h, dev));
    return perm_cvec_download(h, dev, host, len);  // (m+1)-vector: internal -> reference constraint order
}

int32_t sdplrp_A_uu(sdplrp_handle *h, int32_t U_id, double *out) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lazy_scratch(h, U_id));
    const double *U = mat_ptr(h, U_id);
    if (!U) return fail(h, SDPLRP_ERR_ARG, "A_uu: bad matrix id");
    SDP_CHECK(comm_require_full(h, U_id));
    SDP_CHECK(aop_uu(h, U, h->A_out));
    SDP_CHECK(comm_reduce_mvec(h, h->A_out, nullptr));
    return copy_out(h, h->A_out, out, h->m + 1);
}

int32_t sdplrp_A_uv(sdplrp_handle *h, int32_t U_id, int32_t V_id, double *out) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lazy_scratch(h, U_id)); SDP_CHECK(lazy_scratch(h, V_id));
    const double *U = mat_ptr(h, U_id), *V = mat_ptr(h, V_id);
    if (!U || !V) return fail(h, SDPLRP_ERR_ARG, "A_uv: bad matrix id");
    SDP_CHECK(comm_require_full(h, U_id)); SDP_CHECK(comm_require_full(h, V_id));
    SDP_CHECK(aop_uv(h, U, V, h->A_out));
    SDP_CHECK(comm_reduce_mvec(h, h->A_out, nullptr));
    return copy_out(h, h->A_out, out, h->m + 1);
}

int32_t sdplrp_At_preprocess(sdplrp_handle *h, const double *y) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (y) {
        SDP_CHECK(perm_cvec_upload(h, h->y, y, h->m + 1));
        h->y_obj = y[h->m];
    }
    return grad_assemble_S(h);
}

int32_t sdplrp_At_left(sdplrp_handle *h, int32_t X_id, int32_t Y_id) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lazy_scratch(h, X_id)); SDP_CHECK(lazy_scratch(h, Y_id));
    const double *X = mat_ptr(h, X_id);
    double *Y = mat_ptr(h, Y_id);
    if (!X || !Y || X == Y) return fail(h, SDPLRP_ERR_ARG, "At_left: bad matrix ids");
    SDP_CHECK(comm_require_full(h, X_id));
    if (!h->S_current) SDP_CHECK(grad_assemble_S(h));
    SDP_CHECK(grad_spmm(h, X, Y, 1.0, false));
    comm_mark_partial(h, Y_id);
    return SDPLRP_OK;
}

int32_t sdplrp_At_right(sdplrp_handle *h, const double *x, double *y, int64_t ncols) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    if (!x || !y || ncols < 1) return fail(h, SDPLRP_ERR_ARG, "At_right: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    double *dx = nullptr, *dy = nullptr;
    const i64 len = h->n * ncols;
    SDP_CHECK(dev_alloc(h, &dx, len));
    int32_t rc = dev_alloc(h, &dy, len);
    if (rc == SDPLRP_OK && !h->S_current) rc = grad_assemble_S(h);
    if (rc == SDPLRP_OK) rc = perm_upload(h, dx, x, ncols, false);
    if (rc == SDPLRP_OK) rc = grad_spmv(h, dx, dy, ncols);
    if (rc == SDPLRP_OK) rc = perm_download(h, dy, y, ncols, false);
    cudaFree(dx);
    if (dy) cudaFree(dy);
    return rc;
}

// ---- fused iteration -----------------------------------------------------------
// Multi-GPU: R is only advanced on the owned rows inside the inner loop; the rows of other ranks are needed only by
// passes that gather factor rows across the partition: C*R rebuilds, constraint matrices with off-diagonal entries or
// several entries (not in the per-row lists), low-rank projections, off-diagonal dynamic gradient parts.
static bool needs_remote_R_rows(const sdplrp_handle *h) {
    const i64 general = h->nA - h->n_sd - (h->obj_mat >= 0 ? 1 : 0);
    return general > 0 || h->n_dynF > 0;   // (low-rank terms project the owned rows and all-reduce r x s numbers)
}

// CR = C*R over the owned rows (from scratch); sums6[c][0] = <R,CR> per row class
static int32_t rebuild_CR(sdplrp_handle *h) {
    if (halo_active(h)) SDP_CHECK(halo_begin(h, h->R));   // only the ghost rows of R travel
    else SDP_CHECK(comm_require_full(h, SDPLRP_MAT_R));
    SectionScope sc(h, SDPLRP_SEC_SPMM);
    SDP_CHECK(grad_obj_spmm(h, h->R, h->CR, nullptr, h->dscal + SC_SUMS));
    h->CR_valid = true;
    return SDPLRP_OK;
}

__global__ void k_store_sum3(const double *__restrict__ sums6, double *out) { *out = sums6[0] + sums6[2] + sums6[4]; }

// f! (src/coreop.jl:11-31).  With a sparse objective the slot m+1 is <R, C*R>, a by-product
// of rebuilding CR = C*R (which resets the drift of the CR recurrence once per major iteration).
static int32_t do_f(sdplrp_handle *h) {
    if (!halo_active(h)) SDP_CHECK(comm_require_full(h, SDPLRP_MAT_R));   // halo plan: every constraint is a per-row list (own rows only)
    const bool split = h->obj_mat >= 0;
    {
        SectionScope sc(h, SDPLRP_SEC_A_UU);
        SDP_CHECK(aop_uu_skip(h, h->R, h->pvio_raw, split));
    }
    if (split) {
        SDP_CHECK(rebuild_CR(h));
        k_store_sum3<<<1, 1, 0, h->stream>>>(h->dscal + SC_SUMS, h->pvio_raw + h->m);
        KLAUNCH(h);
    }
    SDP_CHECK(comm_reduce_mvec(h, h->pvio_raw, nullptr));
    SectionScope sc(h, SDPLRP_SEC_F_FINISH);
    return vec_f_finish(h);
}

// g! (src/coreop.jl:305-317): y, then G = 2*(y_obj*CR + S_dyn(y)*R + low rank) and the two norms
static int32_t do_g(sdplrp_handle *h) {
    if (h->obj_mat >= 0 && !h->CR_valid) SDP_CHECK(rebuild_CR(h));
    if (needs_remote_R_rows(h)) SDP_CHECK(comm_require_full(h, SDPLRP_MAT_R));
    {
        SectionScope sc(h, SDPLRP_SEC_S_ASSEMBLE);
        SDP_CHECK(grad_form_y(h));
    }
    {
        SectionScope sc(h, SDPLRP_SEC_GRAD);
        SDP_CHECK(grad_hot(h));
    }
    h->gram_g_valid = false;  // G changed: its dots with the L-BFGS history are rebuilt by the update pass
    comm_mark_partial(h, SDPLRP_MAT_G);
    SectionScope sc(h, SDPLRP_SEC_NORMS);
    SDP_CHECK(comm_reduce_scalars(h, SC_GNORM2, 1));
    return vec_pnorm2(h);  // reduces its own share
}

int32_t sdplrp_f(sdplrp_handle *h, double *L, double *obj) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(do_f(h));
    SDP_CHECK(fetch_scalars(h, SC_OBJ, 2));
    if (obj) *obj = h->hscal[SC_OBJ];
    if (L) *L = h->hscal[SC_LVAL];
    return SDPLRP_OK;
}

int32_t sdplrp_g(sdplrp_handle *h, double *gnorm2, double *pnorm2) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(do_g(h));
    SDP_CHECK(fetch_scalars(h, SC_GNORM2, 2));
    if (gnorm2) *gnorm2 = h->hscal[SC_GNORM2];
    if (pnorm2) *pnorm2 = h->hscal[SC_PNORM2];
    return SDPLRP_OK;
}

int32_t sdplrp_fg(sdplrp_handle *h, double out[4]) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(do_f(h));
    SDP_CHECK(do_g(h));
    SDP_CHECK(fetch_scalars(h, SC_GNORM2, 4));
    out[0] = h->hscal[SC_LVAL]; out[1] = h->hscal[SC_OBJ]; out[2] = h->hscal[SC_GNORM2]; out[3] = h->hscal[SC_PNORM2];
    return SDPLRP_OK;
}

// the direction without the host round trip for `descent` (native loop: the value comes back with the line-search
// coefficients, api_linesearch_coeffs_descent)
int32_t api_lbfgs_dir_async(sdplrp_handle *h) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    {
        SectionScope sc(h, SDPLRP_SEC_LBFGS_DIR);
        SDP_CHECK(lb_dir(h));
    }
    h->CD_valid = false; h->ls_valid = false;
    comm_mark_partial(h, SDPLRP_MAT_D);
    return SDPLRP_OK;
}

int32_t sdplrp_lbfgs_dir(sdplrp_handle *h, double *descent) {
    SDP_CHECK(api_lbfgs_dir_async(h));
    SDP_CHECK(fetch_scalars(h, SC_DESCENT, 1));
    if (descent) *descent = h->hscal[SC_DESCENT];
    return SDPLRP_OK;
}

int32_t sdplrp_use_gradient_direction(sdplrp_handle *h) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(lb_neg_copy(h));
    h->gram_g_valid = false;
    h->CD_valid = false; h->ls_valid = false;
    comm_mark_partial(h, SDPLRP_MAT_D);
    return SDPLRP_OK;
}

// linesearch_coeffs; `descent` (may be null) receives dot(dirt, Gt) of the preceding direction call in the same host round trip
int32_t api_linesearch_coeffs_descent(sdplrp_handle *h, double bq[5], double *descent) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    const bool split = h->obj_mat >= 0;
    if (split && !h->CR_valid) SDP_CHECK(rebuild_CR(h));
    // several GPUs: the halo exchange of D starts here and runs on the comm stream under the constraint pass and the
    // [own | hub] half of the gather pass; without a halo plan the whole of D is all-gathered first
    if (halo_active(h)) SDP_CHECK(halo_begin(h, h->D));
    else SDP_CHECK(comm_require_full(h, SDPLRP_MAT_D));
    if (needs_remote_R_rows(h)) SDP_CHECK(comm_require_full(h, SDPLRP_MAT_R));
    {
        SectionScope sc(h, SDPLRP_SEC_LS_PASS);
        SDP_CHECK(aop_linesearch(h, split));  // constraints: sampled dots (A_RD already x2, A_DD)
    }
    if (split) {
        // objective: CD = C*D (the one gather pass of the iteration), <C,DD'> = <D,CD>, <C,RD'+DR'> = 2<D,CR>
        SectionScope sc(h, SDPLRP_SEC_SPMM);
        SDP_CHECK(grad_obj_spmm(h, h->D, h->CD, h->CR, h->dscal + SC_SUMS));
        SDP_CHECK(grad_obj_slots(h, h->dscal + SC_SUMS, h->A_RD + h->m, h->A_DD + h->m));
        h->CD_valid = true;
    }
    SDP_CHECK(comm_reduce_mvec(h, h->A_RD, h->A_DD));
    {
        SectionScope sc(h, SDPLRP_SEC_LS_COEFF);
        SDP_CHECK(vec_biquadratic(h));
    }
    h->ls_valid = true;
    static_assert(SC_DESCENT < SC_BQ, "one contiguous fetch covers descent and the coefficients");
    SDP_CHECK(fetch_scalars(h, SC_DESCENT, SC_BQ + 5 - SC_DESCENT));
    for (int k = 0; k < 5; k++) bq[k] = h->hscal[SC_BQ + k];
    if (descent) *descent = h->hscal[SC_DESCENT];
    return SDPLRP_OK;
}

int32_t sdplrp_linesearch_coeffs(sdplrp_handle *h, double bq[5]) { return api_linesearch_coeffs_descent(h, bq, nullptr); }


int32_t sdplrp_step(sdplrp_handle *h, double alpha, double *obj) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    {
        SectionScope sc(h, SDPLRP_SEC_STEP);
        SDP_CHECK(vec_commit(h, alpha));
        const bool recur = h->obj_mat >= 0 && h->CR_valid && h->CD_valid;
        if (recur && h->world == 1) {
            SDP_CHECK(lb_axpy2(h, alpha, h->D, h->R, h->CD, h->CR));  // Rt += a*dirt ; CR += a*CD
        } else {
            SDP_CHECK(comm_step_R(h, alpha));  // Rt += alpha*dirt (all rows when replicated)
            if (recur) SDP_CHECK(lb_axpy(h, alpha, h->CD, h->CR));
            else h->CR_valid = false;
        }
    }
    h->ls_valid = false;
    if (obj) {
        SDP_CHECK(fetch_scalars(h, SC_OBJ, 1));
        *obj = h->hscal[SC_OBJ];
    }
    return SDPLRP_OK;
}

// sdplrp_step followed by sdplrp_g, fused into one row pass when the line search of the current direction is
// still valid (single GPU); out = {obj, ||G||_F^2, ||pvio||_2^2}
int32_t sdplrp_step_g(sdplrp_handle *h, double alpha, double out[3]) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    if (!out) return fail(h, SDPLRP_ERR_ARG, "step_g: null output");
    CUDA_TRY(h, cudaSetDevice(h->device));
    const bool split = h->obj_mat >= 0;
    const bool fused = h->fused_tail && h->ls_valid && (!split || (h->CR_valid && h->CD_valid));
    if (fused) {
        SectionScope sc(h, SDPLRP_SEC_TAIL);
        SDP_CHECK(grad_step_fused(h, alpha));
        h->ls_valid = false; h->CD_valid = false;
        h->gram_g_valid = false;
    } else {
        SDP_CHECK(sdplrp_step(h, alpha, nullptr));
        SDP_CHECK(do_g(h));
    }
    SDP_CHECK(fetch_scalars(h, SC_GNORM2, 3));
    out[0] = h->hscal[SC_OBJ]; out[1] = h->hscal[SC_GNORM2]; out[2] = h->hscal[SC_PNORM2];
    return SDPLRP_OK;
}

int32_t sdplrp_lbfgs_update(sdplrp_handle *h, double alpha) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SectionScope sc(h, SDPLRP_SEC_LBFGS_UPDATE);
    return lb_update(h, alpha);
}

int32_t sdplrp_lbfgs_clear(sdplrp_handle *h) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    return lb_clear(h);
}

int32_t sdplrp_dual_update(sdplrp_handle *h) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    return vec_dual_update(h);
}

int32_t sdplrp_armijo_eval(sdplrp_handle *h, const double *alphas, int32_t k, double *L, double *slope) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    if (k < 0 || (k > 0 && (!alphas || !L))) return fail(h, SDPLRP_ERR_ARG, "armijo_eval: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    return vec_armijo(h, alphas, k, L, slope);
}

// ---- dual bound ------------------------------------------------------------------
int32_t sdplrp_lanczos(sdplrp_handle *h, int64_t q, const double *v0, uint64_t seed, int32_t reorth, double *alpha, double *beta,
                       int64_t *iters) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    if (q < 1 || !alpha || !beta || !iters) return fail(h, SDPLRP_ERR_ARG, "lanczos: bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device));
    i64 it = 0;
    if (!h->S_current) SDP_CHECK(grad_assemble_S(h));  // S for the device y (g! no longer materialises it)
    {
        SectionScope sc(h, SDPLRP_SEC_LANCZOS);
        SDP_CHECK(lz_run(h, q, v0, seed, reorth, alpha, beta, &it));
    }
    *iters = it;
    return SDPLRP_OK;
}

int32_t sdplrp_tridiag_mineig(const double *d, const double *e, int64_t k, double *out) {
    if (!d || !out || k < 1 || (k > 1 && !e)) return SDPLRP_ERR_ARG;
    *out = tridiag_mineig_host(d, e, k);
    return SDPLRP_OK;
}

int32_t sdplrp_dual_obj(sdplrp_handle *h, double trace_bound, int64_t iter, const double *v0, uint64_t seed, double *dual_value,
                        double *mineig, int64_t *lanczos_steps) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(grad_form_y(h));
    SDP_CHECK(grad_assemble_S(h));
    const double it = (double)std::max<i64>(iter, 100);
    i64 q = (i64)(2.0 * ceil(sqrt(it) * log((double)h->n)));  // src/coreop.jl:402
    q = std::max<i64>(1, std::min<i64>(q, h->n - 1));
    std::vector<double> a((size_t)q), b((size_t)q);
    i64 steps = 0;
    {
        SectionScope sc(h, SDPLRP_SEC_LANCZOS);
        SDP_CHECK(lz_run(h, q, v0, seed, 0, a.data(), b.data(), &steps));
    }
    for (i64 i = 0; i < steps; i++) a[(size_t)i] += 1.0;  // shift by I (src/coreop.jl:503)
    const double lam = (steps == 1 ? a[0] : tridiag_mineig_host(a.data(), b.data(), steps)) - 1.0;
    double yb = 0.0;
    SDP_CHECK(vec_dual_dot(h, &yb));
    if (dual_value) *dual_value = yb + trace_bound * std::min(lam, 0.0);  // src/coreop.jl:412
    if (mineig) *mineig = lam;
    if (lanczos_steps) *lanczos_steps = steps;
    return SDPLRP_OK;
}

int32_t sdplrp_dense_symeig(const double *A, int64_t k, double *ev, double *Q) {
    if (!A || !ev || k < 1 || k > 4096) return SDPLRP_ERR_ARG;
    dense_symeig_host(A, k, ev, Q);
    return SDPLRP_OK;
}

// SDP_S_eigval(var, aux, nevs, true; which=:SA, ncv, tol, maxiter) (src/coreop.jl:351-374) on the S last assembled
int32_t sdplrp_S_eigval(sdplrp_handle *h, int64_t nevs, int64_t ncv, double tol, int64_t maxiter, const double *v0, uint64_t seed,
                        double *eigvals, double *bounds, int64_t *matvecs, int64_t *restarts) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    if (!eigvals) return fail(h, SDPLRP_ERR_ARG, "S_eigval: eigvals is null");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (!h->S_current) SDP_CHECK(grad_assemble_S(h));
    i64 mv = 0, rs = 0;
    {
        SectionScope sc(h, SDPLRP_SEC_LANCZOS);
        SDP_CHECK(lz_eigs(h, nevs, ncv, tol, maxiter, v0, seed, eigvals, bounds, &mv, &rs));
    }
    if (matvecs) *matvecs = mv;
    if (restarts) *restarts = rs;
    return SDPLRP_OK;
}

// dual_obj(...; highprecision=true) (src/coreop.jl:376-415): ncv = min(100, n), tol = 1e-6, maxiter = 10^6
int32_t sdplrp_dual_obj_highprecision(sdplrp_handle *h, double trace_bound, const double *v0, uint64_t seed, double *dual_value,
                                      double *mineig, int64_t *matvecs) {
    REQUIRE_H(h); REQUIRE_PRE(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    SDP_CHECK(grad_form_y(h));
    SDP_CHECK(grad_assemble_S(h));
    double lam = 0.0;
    i64 mv = 0;
    {
        SectionScope sc(h, SDPLRP_SEC_LANCZOS);
        SDP_CHECK(lz_eigs(h, 1, std::min<i64>(100, h->n), 1e-6, 1000000, v0, seed, &lam, nullptr, &mv, nullptr));
    }
    double yb = 0.0;
    SDP_CHECK(vec_dual_dot(h, &yb));
    if (dual_value) *dual_value = yb + trace_bound * std::min(lam, 0.0);
    if (mineig) *mineig = lam;
    if (matvecs) *matvecs = mv;
    return SDPLRP_OK;
}

// DIMACS_errors (src/coreop.jl:426-453).  Leaves y = -lambda (copy2y_lambda!) and the matching S behind, as the
// reference does; err6 uses the sparse part of S only, as the reference does (`var.Rt * aux.sparse_S`).
int32_t sdplrp_dimacs_errors(sdplrp_handle *h, double normb, double normC, const double *v0, uint64_t seed, double errs[6]) {
    REQUIRE_H(h); REQUIRE_PRE(h); REQUIRE_RANK(h);
    if (!errs) return fail(h, SDPLRP_ERR_ARG, "dimacs_errors: errs is null");
    CUDA_TRY(h, cudaSetDevice(h->device));
    double raw2 = 0.0, lamb = 0.0, obj = 0.0;
    SDP_CHECK(vec_dimacs_sums(h, &raw2, &lamb));
    SDP_CHECK(fetch_scalars(h, SC_OBJ, 1));
    obj = h->hscal[SC_OBJ];
    SDP_CHECK(vec_copy2y_lambda(h));
    SDP_CHECK(grad_assemble_S(h));
    double lam = 0.0;
    {
        SectionScope sc(h, SDPLRP_SEC_LANCZOS);
        SDP_CHECK(lz_eigs(h, 1, std::min<i64>(100, h->n), 0.0, 1000000, v0, seed, &lam, nullptr, nullptr, nullptr));
    }
    SDP_CHECK(lazy_scratch(h, SDPLRP_MAT_W0));
    SDP_CHECK(comm_require_full(h, SDPLRP_MAT_R));
    SDP_CHECK(grad_spmm_sparse(h, h->R, h->W0, 1.0));
    comm_mark_partial(h, SDPLRP_MAT_W0);
    SDP_CHECK(lb_dot(h, h->R, h->W0, SC_LANCZOS + 9));
    SDP_CHECK(comm_reduce_scalars(h, SC_LANCZOS + 9, 1));
    SDP_CHECK(fetch_scalars(h, SC_LANCZOS + 9, 1));
    const double xz = h->hscal[SC_LANCZOS + 9];
    const double den = 1.0 + fabs(obj) + fabs(lamb);
    errs[0] = sqrt(raw2) / (1.0 + normb);
    errs[1] = 0.0;
    errs[2] = 0.0;  // X = RR', Z = C - A*(y): errors 2 and 3 vanish by construction
    errs[3] = std::max(0.0, -lam) / (1.0 + normC);
    errs[4] = (obj - lamb) / den;
    errs[5] = xz / den;
    return SDPLRP_OK;
}

int32_t sdplrp_set_profiling(sdplrp_handle *h, int32_t on) {
    REQUIRE_H(h);
    h->prof = on != 0;
    return SDPLRP_OK;
}

int32_t sdplrp_section_times(sdplrp_handle *h, double *ms, int64_t *counts) {
    REQUIRE_H(h);
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    prof_collect(h);
    for (int k = 0; k < SDPLRP_SEC_COUNT; k++) {
        if (ms) ms[k] = h->sec_ms[k];
        if (counts) counts[k] = h->sec_cnt[k];
        h->sec_ms[k] = 0.0; h->sec_cnt[k] = 0;
    }
    return SDPLRP_OK;
}

int32_t sdplrp_launch_count(sdplrp_handle *h, int64_t *count) {
    REQUIRE_H(h);
    if (count) *count = h->launches;
    return SDPLRP_OK;
}

int32_t sdplrp_row_range(sdplrp_handle *h, int64_t *lo, int64_t *hi) {
    REQUIRE_H(h);
    if (lo) *lo = h->row_lo;
    if (hi) *hi = h->row_hi;
    return SDPLRP_OK;
}

}  // extern "C"
