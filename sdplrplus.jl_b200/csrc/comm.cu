// comm.cu -- multi-GPU plumbing: one handle per rank, NCCL over NVLink.
//
// The reference has no distributed path at all (SURVEY.md 5, 8e); this is the
// B200-side design: rows of R/G/D/history and of the aggregated pattern are
// 1-D partitioned in contiguous blocks balanced by nonzeros.  R is kept
// replicated and advanced locally (R += alpha*D on every row), so the only
// bulk exchange per inner iteration is one all-gather of the direction D;
// dot products and the constraint vector are all-reduced.
//
// world == 1 never touches NCCL: every function below is a no-op then.
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>
#include <algorithm>
#include "common.cuh"

// NCCL is bound lazily with dlopen: a process that already carries a libnccl
// (e.g. the one bundled with PyTorch, which the host runtime imports first)
// keeps using it, and single-GPU use never loads NCCL at all.
namespace {
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommSplit)(ncclComm_t, int, int, ncclComm_t *, void *) = nullptr;   // optional (NCCL >= 2.18)
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi g_nccl;

bool nccl_bind() {
    if (g_nccl.ok) return true;
    void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return false;
#define BIND(field, sym) *(void **)(&g_nccl.field) = dlsym(lib, sym); if (!g_nccl.field) return false
    BIND(GetUniqueId, "ncclGetUniqueId");
    BIND(CommInitRank, "ncclCommInitRank");
    BIND(CommDestroy, "ncclCommDestroy");
    BIND(AllReduce, "ncclAllReduce");
    BIND(Broadcast, "ncclBroadcast");
    BIND(AllGather, "ncclAllGather");
    BIND(Send, "ncclSend");
    BIND(Recv, "ncclRecv");
    *(void **)(&g_nccl.CommSplit) = dlsym(lib, "ncclCommSplit");
    BIND(GroupStart, "ncclGroupStart");
    BIND(GroupEnd, "ncclGroupEnd");
    BIND(GetErrorString, "ncclGetErrorString");
#undef BIND
    g_nccl.ok = true;
    return true;
}
}  // namespace
#define ncclGetUniqueId g_nccl.GetUniqueId
#define ncclCommInitRank g_nccl.CommInitRank
#define ncclCommDestroy g_nccl.CommDestroy
#define ncclAllReduce g_nccl.AllReduce
#define ncclBroadcast g_nccl.Broadcast
#define ncclAllGather g_nccl.AllGather
#define ncclSend g_nccl.Send
#define ncclRecv g_nccl.Recv
#define ncclGroupStart g_nccl.GroupStart
#define ncclGroupEnd g_nccl.GroupEnd
#define ncclGetErrorString g_nccl.GetErrorString

#define NCCL_TRY(h, call)                                                        \
    do {                                                                         \
        ncclResult_t r__ = (call);                                               \
        if (r__ != ncclSuccess) {                                                \
            (h)->err = std::string(#call) + ": " + ncclGetErrorString(r__);      \
            return SDPLRP_ERR_NCCL;                                              \
        }                                                                        \
    } while (0)

extern "C" int32_t sdplrp_nccl_unique_id(void *out128) {
    if (!out128) return SDPLRP_ERR_ARG;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    if (!nccl_bind()) return SDPLRP_ERR_NCCL;
    ncclUniqueId id;
    if (ncclGetUniqueId(&id) != ncclSuccess) return SDPLRP_ERR_NCCL;
    memcpy(out128, &id, sizeof(id));
    return SDPLRP_OK;
}

int32_t comm_init(sdplrp_handle *h, const void *nccl_id) {
    if (h->world <= 1) return SDPLRP_OK;
    if (!nccl_id) return fail(h, SDPLRP_ERR_ARG, "create: world > 1 needs the NCCL unique id");
    if (!nccl_bind()) return fail(h, SDPLRP_ERR_NCCL, "cannot load libnccl.so.2");
    ncclUniqueId id;
    memcpy(&id, nccl_id, sizeof(id));
    ncclComm_t comm;
    NCCL_TRY(h, ncclCommInitRank(&comm, h->world, id, h->rank));
    h->nccl = (void *)comm;
    // the halo exchange of the gather pass runs on its own stream, concurrently with kernels (and scalar all-reduces) of the
    // compute stream: it gets its own communicator so that the two never serialise on one another
    if (g_nccl.CommSplit) {
        ncclComm_t c2 = nullptr;
        if (g_nccl.CommSplit(comm, 0, h->rank, &c2, nullptr) == ncclSuccess && c2) h->nccl_halo = (void *)c2;
    }
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->comm_stream, cudaStreamNonBlocking));
    CUDA_TRY(h, cudaEventCreateWithFlags(&h->ev_pack, cudaEventDisableTiming));
    for (int k = 0; k < 2; k++) CUDA_TRY(h, cudaEventCreateWithFlags(&h->ev_class[k], cudaEventDisableTiming));
    return SDPLRP_OK;
}

void comm_destroy(sdplrp_handle *h) {
    if (h->nccl_halo) { ncclCommDestroy((ncclComm_t)h->nccl_halo); h->nccl_halo = nullptr; }
    if (h->ev_pack) { cudaEventDestroy(h->ev_pack); h->ev_pack = nullptr; }
    for (int k = 0; k < 2; k++) if (h->ev_class[k]) { cudaEventDestroy(h->ev_class[k]); h->ev_class[k] = nullptr; }
    if (h->comm_stream) { cudaStreamDestroy(h->comm_stream); h->comm_stream = nullptr; }
    if (h->nccl) {
        ncclCommDestroy((ncclComm_t)h->nccl);
        h->nccl = nullptr;
    }
}

// contiguous row blocks with ~nnzF/world nonzeros each (prefix sum over the
// full pattern's row pointer); identical on every rank.
// the per-row-constraint slots that go with each rank's row block
static int32_t partition_constraints(sdplrp_handle *h) {
    h->c_starts.assign((size_t)h->world + 1, 0);
    for (int q = 0; q <= h->world; q++) {
        int v = 0;
        CUDA_TRY(h, cudaMemcpy(&v, h->rowc_ptr + h->row_starts[(size_t)q], sizeof(int), cudaMemcpyDeviceToHost));
        h->c_starts[(size_t)q] = v;
    }
    h->c_lo = h->c_starts[(size_t)h->rank];
    h->c_hi = h->c_starts[(size_t)h->rank + 1];
    return SDPLRP_OK;
}

int32_t comm_partition(sdplrp_handle *h) {
    const i64 n = h->n;
    for (int id = 0; id < 8; id++) h->mat_full[id] = true;
    if (h->dealt && h->world > 1) {  // blocks fixed by the hub-first relabeling (preprocess.cu, k_deal_rows)
        h->row_lo = h->row_starts[(size_t)h->rank];
        h->row_hi = h->row_starts[(size_t)h->rank + 1];
        return partition_constraints(h);
    }
    h->row_starts.assign((size_t)h->world + 1, 0);
    h->row_starts[(size_t)h->world] = n;
    if (h->world <= 1) {
        h->row_lo = 0; h->row_hi = n;
        h->c_lo = 0; h->c_hi = h->n_sd;
        h->c_starts.assign(2, 0); h->c_starts[1] = h->n_sd;
        return SDPLRP_OK;
    }
    std::vector<int> ptr((size_t)n + 1);
    CUDA_TRY(h, cudaMemcpy(ptr.data(), h->full_ptr, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost));
    // weight of a row in "gathered nonzeros": each nonzero of the gather pass costs ~128 B of DRAM granule
    // traffic; the streaming passes (L-BFGS 22N, step 6N, gradient 3N, constraint pass 2N, ...) cost ~35 rows of
    // 8r bytes per vertex = ~22 nonzero-equivalents at r = 10.  (With the hub-first order a pure nnz balance
    // would give the first rank a sliver of the rows and the last rank nearly all the BLAS-1 work.)
    const double kRowCost = 22.0;
    const double total = (double)ptr[(size_t)n] + kRowCost * (double)n;
    i64 row = 0;
    for (int p = 1; p < h->world; p++) {
        const double target = total * p / h->world;
        while (row < n && (double)ptr[(size_t)row] + kRowCost * (double)row < target) row++;
        h->row_starts[(size_t)p] = row;
    }
    h->row_lo = h->row_starts[(size_t)h->rank];
    h->row_hi = h->row_starts[(size_t)h->rank + 1];
    return partition_constraints(h);
}

static int full_slot(int mat_id) {
    switch (mat_id) {
    case SDPLRP_MAT_R: return 0;
    case SDPLRP_MAT_G: return 1;
    case SDPLRP_MAT_D: return 2;
    case SDPLRP_MAT_W0: return 3;
    case SDPLRP_MAT_W1: return 4;
    default: return -1;
    }
}

void comm_mark_partial(sdplrp_handle *h, int mat_id) {
    if (h->world <= 1) return;
    const int s = full_slot(mat_id);
    if (s >= 0) h->mat_full[s] = false;
}
void comm_mark_full(sdplrp_handle *h, int mat_id) {
    const int s = full_slot(mat_id);
    if (s >= 0) h->mat_full[s] = true;
}

// all-gather (variable block sizes) of the owned row blocks of a dense n x r matrix
static int32_t allgather_rows(sdplrp_handle *h, double *p) {
    SectionScope sc(h, SDPLRP_SEC_COMM);
    ncclComm_t comm = (ncclComm_t)h->nccl;
    if (h->equal_blocks) {
        // equal row blocks (the matrices carry world*block_rows rows of capacity): one in-place all-gather
        const size_t cnt = (size_t)h->block_rows * h->r;
        NCCL_TRY(h, ncclAllGather(p + (size_t)h->rank * cnt, p, cnt, ncclDouble, comm, h->stream));
        return SDPLRP_OK;
    }
    NCCL_TRY(h, ncclGroupStart());
    for (int q = 0; q < h->world; q++) {
        const i64 off = h->row_starts[(size_t)q] * h->r;
        const i64 len = (h->row_starts[(size_t)q + 1] - h->row_starts[(size_t)q]) * h->r;
        if (len > 0) NCCL_TRY(h, ncclBroadcast(p + off, p + off, (size_t)len, ncclDouble, q, comm, h->stream));
    }
    NCCL_TRY(h, ncclGroupEnd());
    return SDPLRP_OK;
}

int32_t comm_require_full(sdplrp_handle *h, int mat_id) {
    if (h->world <= 1) return SDPLRP_OK;
    const int s = full_slot(mat_id);
    if (s < 0) return fail(h, SDPLRP_ERR_ARG, "multi-GPU: only R/G/D/W0/W1 can be operator inputs");
    if (h->mat_full[s]) return SDPLRP_OK;
    double *p = nullptr;
    switch (s) {
    case 0: p = h->R; break;
    case 1: p = h->G; break;
    case 2: p = h->D; break;
    case 3: p = h->W0; break;
    default: p = h->W1; break;
    }
    SDP_CHECK(allgather_rows(h, p));
    h->mat_full[s] = true;
    return SDPLRP_OK;
}

// used by download_mat: history slots are only ever valid on their owners
int32_t comm_gather_rows(sdplrp_handle *h, double *p, int mat_id) {
    if (h->world <= 1) return SDPLRP_OK;
    const int s = full_slot(mat_id);
    if (s >= 0) return comm_require_full(h, mat_id);
    return allgather_rows(h, p);
}

// sum the per-rank partial constraint vectors (length m+1)
int32_t comm_reduce_mvec(sdplrp_handle *h, double *v1, double *v2) {
    if (h->world <= 1) return SDPLRP_OK;
    SectionScope sc(h, SDPLRP_SEC_COMM);
    ncclComm_t comm = (ncclComm_t)h->nccl;
    // only the shared slots [n_sd, m]: the per-row constraints are computed and consumed by their owner (vecops.cu)
    const size_t off = (size_t)h->n_sd, cnt = (size_t)(h->m + 1 - h->n_sd);
    NCCL_TRY(h, ncclGroupStart());
    NCCL_TRY(h, ncclAllReduce(v1 + off, v1 + off, cnt, ncclDouble, ncclSum, comm, h->stream));
    if (v2) NCCL_TRY(h, ncclAllReduce(v2 + off, v2 + off, cnt, ncclDouble, ncclSum, comm, h->stream));
    NCCL_TRY(h, ncclGroupEnd());
    return SDPLRP_OK;
}

// every rank receives the per-row-constraint slots of the other ranks (downloads, S assembly for Lanczos)
int32_t comm_gather_cvec(sdplrp_handle *h, double *v) {
    if (h->world <= 1) return SDPLRP_OK;
    SectionScope sc(h, SDPLRP_SEC_COMM);
    ncclComm_t comm = (ncclComm_t)h->nccl;
    NCCL_TRY(h, ncclGroupStart());
    for (int q = 0; q < h->world; q++) {
        const i64 off = h->c_starts[(size_t)q], len = h->c_starts[(size_t)q + 1] - off;
        if (len > 0) NCCL_TRY(h, ncclBroadcast(v + off, v + off, (size_t)len, ncclDouble, q, comm, h->stream));
    }
    NCCL_TRY(h, ncclGroupEnd());
    return SDPLRP_OK;
}

// every rank receives the owned row blocks of an n-vector in internal vertex order (row-partitioned Lanczos)
int32_t comm_gather_rowvec(sdplrp_handle *h, double *v) {
    if (h->world <= 1) return SDPLRP_OK;
    SectionScope sc(h, SDPLRP_SEC_COMM);
    ncclComm_t comm = (ncclComm_t)h->nccl;
    NCCL_TRY(h, ncclGroupStart());
    for (int q = 0; q < h->world; q++) {
        const i64 off = h->row_starts[(size_t)q], len = h->row_starts[(size_t)q + 1] - off;
        if (len > 0) NCCL_TRY(h, ncclBroadcast(v + off, v + off, (size_t)len, ncclDouble, q, comm, h->stream));
    }
    NCCL_TRY(h, ncclGroupEnd());
    return SDPLRP_OK;
}

// the same with row_bytes bytes per row (the packed sign words of the rounding passes)
int32_t comm_gather_rowbytes(sdplrp_handle *h, void *v, size_t row_bytes) {
    if (h->world <= 1) return SDPLRP_OK;
    SectionScope sc(h, SDPLRP_SEC_COMM);
    ncclComm_t comm = (ncclComm_t)h->nccl;
    char *p = static_cast<char *>(v);
    NCCL_TRY(h, ncclGroupStart());
    for (int q = 0; q < h->world; q++) {
        const size_t off = (size_t)h->row_starts[(size_t)q] * row_bytes;
        const size_t len = (size_t)(h->row_starts[(size_t)q + 1] - h->row_starts[(size_t)q]) * row_bytes;
        if (len > 0) NCCL_TRY(h, ncclBroadcast(p + off, p + off, len, ncclChar, q, comm, h->stream));
    }
    NCCL_TRY(h, ncclGroupEnd());
    return SDPLRP_OK;
}

// SPMD contract: every rank must have been handed the same problem.  `value` is a 64-bit checksum of this rank's input;
// the ranks agree iff max == min of both halves (all-reduced as exactly representable doubles).
int32_t comm_check_same(sdplrp_handle *h, unsigned long long value, const char *what) {
    if (h->world <= 1) return SDPLRP_OK;
    double *d = h->dscal + SC_LANCZOS + 12;
    double v[4] = {(double)(value >> 32), (double)(value & 0xFFFFFFFFull), 0.0, 0.0};
    v[2] = -v[0]; v[3] = -v[1];
    CUDA_TRY(h, cudaMemcpyAsync(d, v, sizeof(v), cudaMemcpyHostToDevice, h->stream));
    NCCL_TRY(h, ncclAllReduce(d, d, 4, ncclDouble, ncclMax, (ncclComm_t)h->nccl, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(v, d, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (v[0] != -v[2] || v[1] != -v[3])
        return fail(h, SDPLRP_ERR_ARG, std::string("multi-GPU: the ranks were given different ") + what +
                                           " (every rank must make the same calls with the same data)");
    return SDPLRP_OK;
}

int32_t comm_reduce_scalars(sdplrp_handle *h, int slot, int count) {
    if (h->world <= 1) return SDPLRP_OK;
    NCCL_TRY(h, ncclAllReduce(h->dscal + slot, h->dscal + slot, (size_t)count, ncclDouble, ncclSum, (ncclComm_t)h->nccl, h->stream));
    return SDPLRP_OK;
}

int32_t comm_reduce_ptr(sdplrp_handle *h, double *p, int count) {
    if (h->world <= 1) return SDPLRP_OK;
    NCCL_TRY(h, ncclAllReduce(p, p, (size_t)count, ncclDouble, ncclSum, (ncclComm_t)h->nccl, h->stream));
    return SDPLRP_OK;
}

// Rt += alpha * dirt on the rows this rank owns
int32_t comm_step_R(sdplrp_handle *h, double alpha) {
    // owned rows only: the rows of other ranks are fetched lazily (comm_require_full) by the passes that need them
    SDP_CHECK(lb_axpy(h, alpha, h->D, h->R));
    comm_mark_partial(h, SDPLRP_MAT_R);
    return SDPLRP_OK;
}

// every rank's `bytes` bytes to every rank (recv = world x bytes, rank order)
int32_t comm_allgather_bytes(sdplrp_handle *h, const void *send, void *recv, size_t bytes) {
    if (h->world <= 1) {
        if (recv != send) CUDA_TRY(h, cudaMemcpyAsync(recv, send, bytes, cudaMemcpyDeviceToDevice, h->stream));
        return SDPLRP_OK;
    }
    NCCL_TRY(h, ncclAllGather(send, recv, bytes, ncclChar, (ncclComm_t)h->nccl, h->stream));
    return SDPLRP_OK;
}

// in-place all-gather of equal blocks: rank q's cnt doubles sit at buf + q*cnt
int32_t comm_allgather_inplace(sdplrp_handle *h, double *buf, size_t cnt) {
    if (h->world <= 1) return SDPLRP_OK;
    NCCL_TRY(h, ncclAllGather(buf + (size_t)h->rank * cnt, buf, cnt, ncclDouble, (ncclComm_t)h->nccl, h->stream));
    return SDPLRP_OK;
}

// ---- halo exchange of the gather pass ---------------------------------------------------------------------------------
namespace {
// out[e] = X[(lo + rows[e / r]) * r + e % r]: the rows the peers gather, in destination order
__global__ void k_pack_rows(i64 n_rows, int r, const int *__restrict__ rows, const double *__restrict__ Xown, double *__restrict__ out) {
    const i64 total = n_rows * r;
    for (i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x; e < total; e += (i64)gridDim.x * blockDim.x) {
        const i64 q = e / r;
        const int c = (int)(e - q * r);
        out[e] = Xown[(size_t)rows[q] * r + c];
    }
}
}  // namespace

bool halo_active(const sdplrp_handle *h) { return h->world > 1 && h->halo.active && h->halo_mode != 0; }

// pack both classes (compute stream), then exchange the hub class and the tail class on the comm stream
int32_t halo_begin(sdplrp_handle *h, const double *X) {
    HaloPlan &p = h->halo;
    const int r = h->r, P = h->world;
    const i64 need_send = (p.n_send[0] + p.n_send[1]) * (i64)r, need_xc = (p.nloc + p.n_ghost[0] + p.n_ghost[1]) * (i64)r;
    if (p.sendbuf_len < need_send) { SDP_CHECK(dev_alloc(h, &p.sendbuf, need_send)); p.sendbuf_len = need_send; }
    if (p.xc_len < need_xc) { SDP_CHECK(dev_alloc(h, &p.xc, need_xc)); p.xc_len = need_xc; }
    const double *Xown = X + (size_t)h->row_lo * r;
    // own rows into the head of the compact operand (the ghosts are received behind them)
    CUDA_TRY(h, cudaMemcpyAsync(p.xc, Xown, (size_t)p.nloc * r * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    // Both classes are packed on the compute stream right behind the kernel that produced X; the comm stream then runs the
    // two exchanges back to back (hub class first) while the compute stream goes on with the constraint pass and -- from the
    // hub event on -- the [own | hub] half of the pass.  (Packing on the comm stream between the exchanges was measured
    // slower at 8 GPUs: 2.69 -> 2.75 ms per iteration, the tail exchange then starts later.)
    for (int k = 0; k < 2; k++) {
        if (p.n_send[k] <= 0) continue;
        double *sb = p.sendbuf + (size_t)(k == 0 ? 0 : p.n_send[0]) * r;
        k_pack_rows<<<grid_for(p.n_send[k] * r, 256, 8 * kNumSM), 256, 0, h->stream>>>(p.n_send[k], r, p.send_rows[k], Xown, sb);
        KLAUNCH(h);
    }
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaEventRecord(h->ev_pack, h->stream));
    CUDA_TRY(h, cudaStreamWaitEvent(h->comm_stream, h->ev_pack, 0));
    ncclComm_t comm = (ncclComm_t)(h->nccl_halo ? h->nccl_halo : h->nccl);
    for (int k = 0; k < 2; k++) {
        const double *sb = p.sendbuf + (size_t)(k == 0 ? 0 : p.n_send[0]) * r;
        double *gb = p.xc + (size_t)(p.nloc + (k == 0 ? 0 : p.n_ghost[0])) * r;
        NCCL_TRY(h, ncclGroupStart());
        for (int q = 0; q < P; q++) {
            if (q == h->rank) continue;
            const i64 so = p.send_off[k][(size_t)q], sc = p.send_off[k][(size_t)q + 1] - so;
            const i64 ro = p.recv_off[k][(size_t)q], rc = p.recv_off[k][(size_t)q + 1] - ro;
            if (sc > 0) NCCL_TRY(h, ncclSend(sb + (size_t)so * r, (size_t)sc * r, ncclDouble, q, comm, h->comm_stream));
            if (rc > 0) NCCL_TRY(h, ncclRecv(gb + (size_t)ro * r, (size_t)rc * r, ncclDouble, q, comm, h->comm_stream));
        }
        NCCL_TRY(h, ncclGroupEnd());
        CUDA_TRY(h, cudaEventRecord(h->ev_class[k], h->comm_stream));
    }
    return SDPLRP_OK;
}

int32_t halo_wait(sdplrp_handle *h, int klass) {
    SectionScope sc(h, SDPLRP_SEC_COMM);   // what the compute stream actually waits = the exposed part of the exchange
    CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_class[klass], 0));
    return SDPLRP_OK;
}
