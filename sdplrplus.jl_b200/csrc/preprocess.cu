// preprocess.cu -- device-side construction of the aggregated sparsity pattern
// and of every index map of preprocess_sparsecons (reference
// src/preprocess.jl:24-169), plus the device-only derived layouts (chunk lists
// for the constraint passes, static/dynamic split of S, SpMM row classes).
//
// Integer work, bit-exact against the oracle.  Sorting / scanning / unique use
// the CUB primitives shipped with the CUDA toolkit (library code, like cuBLAS
// for a plain GEMM); everything pattern-specific is hand-written below.
#include <cub/cub.cuh>
#include <algorithm>
#include <climits>
#include <cmath>
#include "common.cuh"

namespace {

struct Tmp {  // scoped device scratch
    std::vector<void *> ptrs;
    ~Tmp() {
        for (void *p : ptrs) cudaFree(p);
    }
    template <typename T>
    T *get(sdplrp_handle *h, i64 count, int32_t *rc) {
        T *p = nullptr;
        if (count <= 0) count = 1;
        cudaError_t e = cudaMalloc((void **)&p, (size_t)count * sizeof(T));
        if (e != cudaSuccess) {
            h->err = std::string("cudaMalloc(preprocess scratch): ") + cudaGetErrorString(e);
            *rc = SDPLRP_ERR_CUDA;
            return nullptr;
        }
        ptrs.push_back(p);
        return p;
    }
};

constexpr int TPB = 256;

__device__ __forceinline__ unsigned long long make_key(int row, int col) {
    return ((unsigned long long)(unsigned)col << 32) | (unsigned)row;
}

// order-sensitive 64-bit checksum of the input triplets (multi-GPU: every rank must preprocess the same problem)
__global__ void k_triplet_checksum(i64 nnz, const int64_t *__restrict__ I, const int64_t *__restrict__ J, const double *__restrict__ V,
                                   unsigned long long *__restrict__ out) {
    unsigned long long acc = 0ull;
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnz; k += (i64)gridDim.x * blockDim.x) {
        unsigned long long x = (unsigned long long)I[k] * 0x9E3779B97F4A7C15ull ^ (unsigned long long)J[k] * 0xD6E8FEB86659FD93ull ^
                               (unsigned long long)__double_as_longlong(V[k]) ^ ((unsigned long long)k << 17);
        x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
        x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
        acc += x ^ (x >> 31);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);   // integer sum: order-independent, deterministic
}

// coordinates -> sort keys + upper-triangle flags (src/preprocess.jl:4-16, 56-82)
__global__ void k_keys(i64 nnz, i64 n, const int64_t *__restrict__ I, const int64_t *__restrict__ J,
                       unsigned long long *__restrict__ keyF, int *__restrict__ flag, int *__restrict__ errw) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnz; k += (i64)gridDim.x * blockDim.x) {
        i64 i = I[k] - 1, j = J[k] - 1;
        if (i < 0 || i >= n || j < 0 || j >= n) {
            atomicOr(errw, 1);
            i = 0; j = 0;
        }
        keyF[k] = make_key((int)i, (int)j);
        flag[k] = (i <= j) ? 1 : 0;
    }
}

// stable compaction of the upper-triangular entries: this IS the concatenated
// findnz(triu(A_i)) order of src/preprocess.jl:95-135
__global__ void k_compact(i64 nnz, const int64_t *__restrict__ I, const int64_t *__restrict__ J,
                          const double *__restrict__ V, const int *__restrict__ flag, const int *__restrict__ tpos,
                          int *__restrict__ ent_row, int *__restrict__ ent_col, double *__restrict__ one,
                          double *__restrict__ two, unsigned long long *__restrict__ keyT) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnz; k += (i64)gridDim.x * blockDim.x) {
        if (!flag[k]) continue;
        int t = tpos[k];
        int i = (int)(I[k] - 1), j = (int)(J[k] - 1);
        double v = V[k];
        ent_row[t] = i;
        ent_col[t] = j;
        one[t] = v;
        two[t] = (i == j) ? v : 2.0 * v;  // src/preprocess.jl:125-132
        keyT[t] = make_key(i, j);
    }
}

// matptr[a] = number of triu entries before matrix a (src/preprocess.jl:101, 135)
__global__ void k_matptr(i64 nA, i64 nnz, i64 Ec, const int64_t *__restrict__ mat_off, const int *__restrict__ tpos,
                         int *__restrict__ matptr, const int64_t *__restrict__ gids, int *__restrict__ mat_gid) {
    for (i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x; a <= nA; a += (i64)gridDim.x * blockDim.x) {
        i64 off = (a < nA) ? mat_off[a] : nnz;
        matptr[a] = (off < nnz) ? tpos[off] : (int)Ec;
        if (a < nA) mat_gid[a] = (int)(gids[a] - 1);
    }
}

// column pointers of a sorted, de-duplicated (col,row) key list
__global__ void k_colptr(i64 n, i64 nnz, const unsigned long long *__restrict__ keys, int *__restrict__ ptr) {
    for (i64 c = blockIdx.x * (i64)blockDim.x + threadIdx.x; c <= n; c += (i64)gridDim.x * blockDim.x) {
        unsigned long long target = (unsigned long long)c << 32;
        i64 lo = 0, hi = nnz;
        while (lo < hi) {
            i64 mid = (lo + hi) >> 1;
            if (keys[mid] < target) lo = mid + 1; else hi = mid;
        }
        ptr[c] = (int)lo;
    }
}

__global__ void k_low32(i64 nnz, const unsigned long long *__restrict__ keys, int *__restrict__ out) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnz; k += (i64)gridDim.x * blockDim.x)
        out[k] = (int)(unsigned)(keys[k] & 0xffffffffull);
}

__device__ __forceinline__ int csc_find(const int *__restrict__ colptr, const int *__restrict__ rowval, int col, int row) {
    int low = colptr[col], high = colptr[col + 1] - 1;
    while (low <= high) {
        int mid = (low + high) >> 1;
        int rv = rowval[mid];
        if (rv == row) return mid;
        if (rv < row) low = mid + 1; else high = mid - 1;
    }
    return -1;
}

// nzind: slot of every entry in the triu CSC (src/preprocess.jl:104-124)
__global__ void k_nzind(i64 Ec, const int *__restrict__ ent_row, const int *__restrict__ ent_col,
                        const int *__restrict__ colptr, const int *__restrict__ rowval, int *__restrict__ slot) {
    for (i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x; t < Ec; t += (i64)gridDim.x * blockDim.x)
        slot[t] = csc_find(colptr, rowval, ent_col[t], ent_row[t]);
}

// agg_sparse_A_mappedto_triu (src/preprocess.jl:137-159)
__global__ void k_mapped(i64 nnzF, const unsigned long long *__restrict__ keyF, const int *__restrict__ colptr,
                         const int *__restrict__ rowval, int *__restrict__ mapped, int *__restrict__ errw) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnzF; k += (i64)gridDim.x * blockDim.x) {
        int row = (int)(unsigned)(keyF[k] & 0xffffffffull), col = (int)(keyF[k] >> 32);
        int rr = min(row, col), cc = max(row, col);
        int s = csc_find(colptr, rowval, cc, rr);
        mapped[k] = s;
        if (s < 0) atomicOr(errw, 2);
    }
}

// matrix index of every entry (upper_bound on matptr)
__global__ void k_ent_mat(i64 Ec, i64 nA, const int *__restrict__ matptr, int *__restrict__ ent_mat) {
    for (i64 t = blockIdx.x * (i64)blockDim.x + threadIdx.x; t < Ec; t += (i64)gridDim.x * blockDim.x) {
        i64 lo = 0, hi = nA;  // find last a with matptr[a] <= t
        while (lo < hi) {
            i64 mid = (lo + hi + 1) >> 1;
            if (matptr[mid] <= (int)t) lo = mid; else hi = mid - 1;
        }
        // skip empty matrices that share the same matptr value: take the one whose range contains t
        ent_mat[t] = (int)lo;
    }
}

__global__ void k_iota(i64 nItems, int *__restrict__ out) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nItems; k += (i64)gridDim.x * blockDim.x) out[k] = (int)k;
}

// first position of each slot in the slot-sorted entry list
__global__ void k_slot_ptr(i64 nnzT, i64 Ec, const int *__restrict__ sorted_slot, int *__restrict__ slot_ptr) {
    for (i64 s = blockIdx.x * (i64)blockDim.x + threadIdx.x; s <= nnzT; s += (i64)gridDim.x * blockDim.x) {
        i64 lo = 0, hi = Ec;
        while (lo < hi) {
            i64 mid = (lo + hi) >> 1;
            if (sorted_slot[mid] < (int)s) lo = mid + 1; else hi = mid;
        }
        slot_ptr[s] = (int)lo;
    }
}

// per triu slot: static (objective) value and number of non-objective contributors
__global__ void k_slot_classify(i64 nnzT, const int *__restrict__ slot_ptr, const int *__restrict__ sorted_t,
                                const int *__restrict__ ent_mat, const double *__restrict__ one, int obj_mat,
                                double *__restrict__ triuS_static, int *__restrict__ dyn_cnt, int *__restrict__ dyn_flag) {
    for (i64 s = blockIdx.x * (i64)blockDim.x + threadIdx.x; s < nnzT; s += (i64)gridDim.x * blockDim.x) {
        double st = 0.0;
        int cnt = 0;
        for (int p = slot_ptr[s]; p < slot_ptr[s + 1]; p++) {
            int t = sorted_t[p];
            if (ent_mat[t] == obj_mat) st += one[t]; else cnt++;
        }
        triuS_static[s] = st;
        dyn_cnt[s] = cnt;
        dyn_flag[s] = cnt > 0 ? 1 : 0;
    }
}

__global__ void k_dyn_fill(i64 nnzT, const int *__restrict__ slot_ptr, const int *__restrict__ sorted_t,
                           const int *__restrict__ ent_mat, const double *__restrict__ one, const int *__restrict__ mat_gid,
                           int obj_mat, const int *__restrict__ dyn_flag, const int *__restrict__ dyn_index,
                           const int *__restrict__ dyn_off, const int *__restrict__ triu_rowval,
                           const unsigned long long *__restrict__ keyT, const int *__restrict__ perm,
                           const int *__restrict__ full_ptr,
                           const int *__restrict__ full_idx, const unsigned char *__restrict__ sd_flag,
                           int *__restrict__ dyn_slot, int *__restrict__ dyn_ptr, int *__restrict__ dyn_nsd_end,
                           int *__restrict__ dyn_gid, double *__restrict__ dyn_val, int *__restrict__ pos_a,
                           int *__restrict__ pos_b) {
    for (i64 s = blockIdx.x * (i64)blockDim.x + threadIdx.x; s < nnzT; s += (i64)gridDim.x * blockDim.x) {
        if (!dyn_flag[s]) continue;
        int d = dyn_index[s];
        int o = dyn_off[s];
        dyn_slot[d] = (int)s;
        dyn_ptr[d] = o;
        // contributors that are NOT single-diagonal-entry constraints first (the hot loop only needs those:
        // the single-diagonal ones are applied from the per-row lists), then the rest; matrix order inside each part
        for (int pass = 0; pass < 2; pass++) {
            for (int p = slot_ptr[s]; p < slot_ptr[s + 1]; p++) {
                int t = sorted_t[p];
                int a = ent_mat[t];
                if (a == obj_mat) continue;
                if ((sd_flag[a] != 0) != (pass == 1)) continue;
                dyn_gid[o] = mat_gid[a];
                dyn_val[o] = one[t];
                o++;
            }
            if (pass == 0) dyn_nsd_end[d] = o;
        }
        int row = triu_rowval[s], col = (int)(keyT[s] >> 32);
        if (perm) { row = perm[row]; col = perm[col]; }  // positions in the INTERNAL full pattern
        pos_a[d] = csc_find(full_ptr, full_idx, col, row);
        pos_b[d] = csc_find(full_ptr, full_idx, row, col);
    }
}

// generic: flag items whose segment length exceeds a threshold
__global__ void k_len_flag(i64 nItems, const int *__restrict__ ptr, int thresh, int *__restrict__ flag) {
    for (i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x; a < nItems; a += (i64)gridDim.x * blockDim.x)
        flag[a] = (ptr[a + 1] - ptr[a] > thresh) ? 1 : 0;
}
__global__ void k_compact_ids(i64 nItems, const int *__restrict__ flag, const int *__restrict__ pos, int *__restrict__ out) {
    for (i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x; a < nItems; a += (i64)gridDim.x * blockDim.x)
        if (flag[a]) out[pos[a]] = (int)a;
}
__global__ void k_chunk_counts(i64 nLong, const int *__restrict__ long_mat, const int *__restrict__ matptr, int chunk,
                               int *__restrict__ cnt) {
    for (i64 l = blockIdx.x * (i64)blockDim.x + threadIdx.x; l < nLong; l += (i64)gridDim.x * blockDim.x) {
        int a = long_mat[l];
        cnt[l] = (matptr[a + 1] - matptr[a] + chunk - 1) / chunk;
    }
}
__global__ void k_chunk_mat(i64 nChunks, i64 nLong, const int *__restrict__ long_chunk_ptr, int *__restrict__ chunk_mat) {
    for (i64 c = blockIdx.x * (i64)blockDim.x + threadIdx.x; c < nChunks; c += (i64)gridDim.x * blockDim.x) {
        i64 lo = 0, hi = nLong - 1;  // last l with long_chunk_ptr[l] <= c
        while (lo < hi) {
            i64 mid = (lo + hi + 1) >> 1;
            if (long_chunk_ptr[mid] <= (int)c) lo = mid; else hi = mid - 1;
        }
        chunk_mat[c] = (int)lo;
    }
}

// export kernels: 0-based int32 -> Julia 1-based int64
__global__ void k_export_i32(i64 nItems, const int *__restrict__ in, int64_t *__restrict__ out) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nItems; k += (i64)gridDim.x * blockDim.x)
        out[k] = (int64_t)in[k] + 1;
}

template <typename F>
int32_t with_cub_temp(sdplrp_handle *h, F f) {
    size_t bytes = 0;
    CUDA_TRY(h, f((void *)nullptr, bytes));
    void *tmp = nullptr;
    CUDA_TRY(h, cudaMalloc(&tmp, bytes ? bytes : 1));
    cudaError_t e = f(tmp, bytes);
    cudaError_t e2 = cudaStreamSynchronize(h->stream);
    cudaFree(tmp);
    if (e != cudaSuccess) { h->err = std::string("cub: ") + cudaGetErrorString(e); return SDPLRP_ERR_CUDA; }
    if (e2 != cudaSuccess) { h->err = std::string("cub sync: ") + cudaGetErrorString(e2); return SDPLRP_ERR_CUDA; }
    return SDPLRP_OK;
}

// The CUB primitives below take 32-bit item counts and the device patterns are int32: inputs beyond 2^31 - 1 entries are
// refused with an error instead of being truncated.
constexpr i64 kMaxItems = 0x7fffffffLL;
#define REQUIRE_32BIT(h, count, what)                                                                                    \
    do {                                                                                                                 \
        if ((count) > kMaxItems) return fail((h), SDPLRP_ERR_ARG, std::string(what) + ": more than 2^31 - 1 entries per GPU"); \
    } while (0)

int32_t exclusive_scan(sdplrp_handle *h, const int *in, int *out, i64 count) {
    if (count <= 0) return SDPLRP_OK;
    REQUIRE_32BIT(h, count, "preprocess (scan)");
    h->launches += 2;
    return with_cub_temp(h, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, in, out, (int)count, h->stream); });
}

// sorted unique keys; returns the count
int32_t sort_unique(sdplrp_handle *h, unsigned long long *keys, unsigned long long *scratch, i64 count, int end_bit,
                    unsigned long long *out, i64 *n_out) {
    if (count <= 0) { *n_out = 0; return SDPLRP_OK; }
    REQUIRE_32BIT(h, count, "preprocess (sort)");
    h->launches += 8;
    SDP_CHECK(with_cub_temp(h, [&](void *t, size_t &b) {
        return cub::DeviceRadixSort::SortKeys(t, b, keys, scratch, (int)count, 0, end_bit, h->stream);
    }));
    int *d_n = nullptr;
    CUDA_TRY(h, cudaMalloc((void **)&d_n, sizeof(int)));
    int32_t rc = with_cub_temp(h, [&](void *t, size_t &b) {
        return cub::DeviceSelect::Unique(t, b, scratch, out, d_n, (int)count, h->stream);
    });
    int hn = 0;
    if (rc == SDPLRP_OK) {
        cudaError_t e = cudaMemcpy(&hn, d_n, sizeof(int), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { h->err = std::string("memcpy(unique count): ") + cudaGetErrorString(e); rc = SDPLRP_ERR_CUDA; }
    }
    cudaFree(d_n);
    *n_out = hn;
    return rc;
}

int32_t read_int(sdplrp_handle *h, const int *dptr, int *out) {
    CUDA_TRY(h, cudaMemcpyAsync(out, dptr, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return SDPLRP_OK;
}

int bits_for(i64 n) {
    int b = 1;
    while (((i64)1 << b) < n) b++;
    return b;
}


// Cfull[k] = value of the objective at full-pattern slot k
__global__ void k_cfull(i64 nnzF, const int *__restrict__ mapped, const int *__restrict__ i2r, const double *__restrict__ st,
                        double *__restrict__ cfull) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnzF; k += (i64)gridDim.x * blockDim.x) {
        const int t = mapped[i2r ? i2r[k] : k];
        cfull[k] = t >= 0 ? st[t] : 0.0;
    }
}
// value-free gather pass (common.cuh: vf_val): the first off-diagonal slot of the full pattern ...
__global__ void k_vf_first(i64 n, const int *__restrict__ ptr, const int *__restrict__ idx, int *__restrict__ first) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x)
        for (int k = ptr[i]; k < ptr[i + 1]; k++)
            if (idx[k] != (int)i) { atomicMin(first, k); break; }
}
// ... then every off-diagonal value must have v's bits, and every C_ii / v must be exact (*bad = 1 otherwise)
__global__ void k_vf_check(i64 n, const int *__restrict__ ptr, const int *__restrict__ idx, const double *__restrict__ cfull, double v,
                           double *__restrict__ diag, int *__restrict__ bad) {
    const unsigned long long vb = (unsigned long long)__double_as_longlong(v);
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        double d = 0.0;
        bool ok = true;
        for (int k = ptr[i]; k < ptr[i + 1]; k++) {
            if (idx[k] == (int)i) d = cfull[k];
            else ok &= (unsigned long long)__double_as_longlong(cfull[k]) == vb;
        }
        const double q = d / v;
        ok &= isfinite(q) && q * v == d;
        diag[i] = q;
        if (!ok) atomicOr(bad, 1);
    }
}
// mark the full-pattern slots (both mirrored positions) of every dynamic triu slot
__global__ void k_dyn_mark(i64 nd, const int *__restrict__ pos_a, const int *__restrict__ pos_b, const int *__restrict__ full_idx,
                           const int *__restrict__ dyn_ptr, const int *__restrict__ dyn_nsd_end,
                           int *__restrict__ flag, int *__restrict__ src, int *__restrict__ dyn_diag) {
    for (i64 d = blockIdx.x * (i64)blockDim.x + threadIdx.x; d < nd; d += (i64)gridDim.x * blockDim.x) {
        const int a = pos_a[d], b = pos_b[d];
        if (a >= 0 && a == b) {  // diagonal slot: a row scaling, not a gather (and nothing at all if only row-list constraints touch it)
            if (dyn_nsd_end[d] > dyn_ptr[d]) dyn_diag[full_idx[a]] = (int)d;
            continue;
        }
        if (a >= 0) { flag[a] = 1; src[a] = (int)d; }
        if (b >= 0) { flag[b] = 1; src[b] = (int)d; }
    }
}
__global__ void k_fill_int(i64 nItems, int v, int *__restrict__ x) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nItems; k += (i64)gridDim.x * blockDim.x) x[k] = v;
}
// single-diagonal-entry constraint matrices -> sort key = their (internal) row, n for every other matrix
__global__ void k_sd_keys(i64 nA, i64 n, int obj_mat, const int *__restrict__ matptr, const int *__restrict__ ent_row,
                          const int *__restrict__ ent_col, unsigned *__restrict__ key, int *__restrict__ val,
                          unsigned char *__restrict__ sd_flag) {
    for (i64 a = blockIdx.x * (i64)blockDim.x + threadIdx.x; a < nA; a += (i64)gridDim.x * blockDim.x) {
        const int k = matptr[a];
        const bool sd = (matptr[a + 1] - k == 1) && (int)a != obj_mat && ent_row[k] == ent_col[k];
        key[a] = sd ? (unsigned)ent_row[k] : (unsigned)n;
        val[a] = (int)a;
        sd_flag[a] = sd ? 1 : 0;
    }
}
__global__ void k_lower_bound_u32(i64 n, i64 len, const unsigned *__restrict__ sorted, int *__restrict__ ptr) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i <= n; i += (i64)gridDim.x * blockDim.x) {
        i64 lo = 0, hi = len;
        while (lo < hi) {
            i64 mid = (lo + hi) >> 1;
            if (sorted[mid] < (unsigned)i) lo = mid + 1; else hi = mid;
        }
        ptr[i] = (int)lo;
    }
}
__global__ void k_sd_fill(i64 n_sd, const int *__restrict__ sorted_a, const int *__restrict__ matptr, const int *__restrict__ mat_gid,
                          const double *__restrict__ ent_two, int *__restrict__ gid, double *__restrict__ val) {
    for (i64 p = blockIdx.x * (i64)blockDim.x + threadIdx.x; p < n_sd; p += (i64)gridDim.x * blockDim.x) {
        const int a = sorted_a[p];
        gid[p] = mat_gid[a];
        val[p] = ent_two[matptr[a]];
    }
}
__global__ void k_dyn_rows(i64 nnzF, const int *__restrict__ flag, const int *__restrict__ pos, const int *__restrict__ src,
                           const int *__restrict__ full_idx, int *__restrict__ col, int *__restrict__ osrc) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnzF; k += (i64)gridDim.x * blockDim.x)
        if (flag[k]) { col[pos[k]] = full_idx[k]; osrc[pos[k]] = src[k]; }
}
__global__ void k_gather_ptr(i64 n, const int *__restrict__ full_ptr, const int *__restrict__ pos, int *__restrict__ out) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i <= n; i += (i64)gridDim.x * blockDim.x) out[i] = pos[full_ptr[i]];
}
__global__ void k_class_flags(i64 n, int gmax, const int *__restrict__ ptr, int *__restrict__ f0, int *__restrict__ f1, int *__restrict__ f2) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        const int len = ptr[i + 1] - ptr[i];
        const int c = len <= gmax ? 0 : (len <= kRowWarpMax ? 1 : 2);
        f0[i] = c == 0; f1[i] = c == 1; f2[i] = c == 2;
    }
}


// ---- internal vertex order (descending degree) ------------------------------------
__global__ void k_deg_key(i64 n, const int *__restrict__ ptr, unsigned *__restrict__ key, int *__restrict__ val) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        key[i] = (unsigned)(n - (i64)(ptr[i + 1] - ptr[i]));  // ascending key == descending degree
        val[i] = (int)i;
    }
}
// multi-GPU: deal the degree-sorted vertices round-robin to the P ranks and lay the ranks' shares out one after the
// other, so that every rank's contiguous row block has the same mix of hub and tail rows (nonzeros AND rows balanced:
// the phases of an iteration are separated by collectives, so each phase must balance, not just their sum)
__global__ void k_deal_rows(i64 n, int P, i64 B, i64 lastT, int rem, bool equal, const int *__restrict__ sorted,
                            int *__restrict__ dealt) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < n; k += (i64)gridDim.x * blockDim.x) {
        int p = (int)(k % P);
        i64 slot = k / P;
        if (equal) {
            // equal blocks of B = ceil(n/P) rows for ranks 0..P-2 (one in-place ncclAllGather moves a factor): the ranks the
            // plain deal leaves one row short take the last (lowest-degree) rows of the last rank
            if (rem != 0 && p == P - 1 && slot >= lastT) { p = rem + (int)(slot - lastT); slot = B - 1; }
            dealt[(i64)p * B + slot] = sorted[k];
        } else {
            i64 start = 0;
            for (int q = 0; q < p; q++) start += (n - q + P - 1) / P;
            dealt[start + slot] = sorted[k];
        }
    }
}
__global__ void k_invert_perm(i64 n, const int *__restrict__ iperm, int *__restrict__ perm) {
    for (i64 p = blockIdx.x * (i64)blockDim.x + threadIdx.x; p < n; p += (i64)gridDim.x * blockDim.x) perm[iperm[p]] = (int)p;
}
// reference full slot k = (ref row = key >> 32 seen as CSR row, ref col = low 32) -> internal key
__global__ void k_internal_keys(i64 nnzF, const unsigned long long *__restrict__ keyF, const int *__restrict__ perm,
                                unsigned long long *__restrict__ ikey, int *__restrict__ payload) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnzF; k += (i64)gridDim.x * blockDim.x) {
        const int a = (int)(keyF[k] >> 32), b = (int)(unsigned)(keyF[k] & 0xffffffffull);
        ikey[k] = make_key(perm[b], perm[a]);  // (row-major key: high = internal row perm[a], low = internal col perm[b])
        payload[k] = (int)k;
    }
}
__global__ void k_scatter_inverse(i64 nItems, const int *__restrict__ fwd, int *__restrict__ inv) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nItems; k += (i64)gridDim.x * blockDim.x) inv[fwd[k]] = (int)k;
}
__global__ void k_apply_perm(i64 nItems, const int *__restrict__ perm, int *__restrict__ x) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nItems; k += (i64)gridDim.x * blockDim.x) x[k] = perm[x[k]];
}

// rows of a CSR pattern binned by length into three compacted lists
int32_t build_classes(sdplrp_handle *h, Tmp &tmp, i64 n, const int *ptr, RowClasses &cls) {
    cudaStream_t st = h->stream;
    const int GS = 8 * kNumSM;
    int32_t rc = SDPLRP_OK;
    int *f[3], *p[3];
    for (int c = 0; c < 3; c++) { f[c] = tmp.get<int>(h, n + 1, &rc); p[c] = tmp.get<int>(h, n + 1, &rc); }
    if (rc) return rc;
    for (int c = 0; c < 3; c++) CUDA_TRY(h, cudaMemsetAsync(f[c], 0, (size_t)(n + 1) * sizeof(int), st));
    k_class_flags<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, h->row_group_max, ptr, f[0], f[1], f[2]); KLAUNCH(h);
    int cnt[3];
    for (int c = 0; c < 3; c++) {
        SDP_CHECK(exclusive_scan(h, f[c], p[c], n + 1));
        SDP_CHECK(read_int(h, p[c] + n, &cnt[c]));
    }
    dev_free(&cls.storage);
    cls = RowClasses();
    if (cnt[1] == 0 && cnt[2] == 0) {  // every row is short: identity order, no list
        cls.cnt[0] = n;
        return SDPLRP_OK;
    }
    SDP_CHECK(dev_alloc(h, &cls.storage, n));
    i64 off = 0;
    for (int c = 0; c < 3; c++) {
        cls.list[c] = cls.storage + off;
        cls.cnt[c] = cnt[c];
        if (cnt[c] > 0) { k_compact_ids<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, f[c], p[c], cls.list[c]); KLAUNCH(h); }
        off += cnt[c];
    }
    return SDPLRP_OK;
}
// ---- internal constraint order: single-diagonal-entry constraints in (internal) row order first, the rest after
__global__ void k_cperm_sd(i64 n_sd, const int *__restrict__ sorted_a, const int *__restrict__ mat_gid, int *__restrict__ cperm,
                           int *__restrict__ assigned) {
    for (i64 p = blockIdx.x * (i64)blockDim.x + threadIdx.x; p < n_sd; p += (i64)gridDim.x * blockDim.x) {
        const int g = mat_gid[sorted_a[p]];
        cperm[g] = (int)p;
        assigned[g] = 1;
    }
}
__global__ void k_not(i64 nItems, const int *__restrict__ x, int *__restrict__ y) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nItems; k += (i64)gridDim.x * blockDim.x) y[k] = x[k] ? 0 : 1;
}
__global__ void k_cperm_rest(i64 m, i64 n_sd, const int *__restrict__ assigned, const int *__restrict__ rank, int *__restrict__ cperm) {
    for (i64 g = blockIdx.x * (i64)blockDim.x + threadIdx.x; g <= m; g += (i64)gridDim.x * blockDim.x) {
        if (g == m) { cperm[g] = (int)m; continue; }  // the objective keeps slot m+1
        if (!assigned[g]) cperm[g] = (int)(n_sd + rank[g]);
    }
}
__global__ void k_sd_vals(i64 n_sd, const int *__restrict__ sorted_a, const int *__restrict__ matptr, const double *__restrict__ ent_two,
                          double *__restrict__ val) {
    for (i64 p = blockIdx.x * (i64)blockDim.x + threadIdx.x; p < n_sd; p += (i64)gridDim.x * blockDim.x)
        val[p] = ent_two[matptr[sorted_a[p]]];
}

__global__ void k_tile_chunk_counts(i64 nLong, const int *__restrict__ long_rows, const int *__restrict__ ptr, int chunk,
                                    int *__restrict__ cnt) {
    for (i64 l = blockIdx.x * (i64)blockDim.x + threadIdx.x; l < nLong; l += (i64)gridDim.x * blockDim.x) {
        const int i = long_rows[l];
        cnt[l] = (ptr[i + 1] - ptr[i] + chunk - 1) / chunk;
    }
}
__global__ void k_tile_chunks(i64 nChunks, i64 nLong, const int *__restrict__ long_rows, const int *__restrict__ long_cptr,
                              const int *__restrict__ ptr, int chunk, int *__restrict__ cstart, int *__restrict__ cend,
                              int *__restrict__ crow) {
    for (i64 c = blockIdx.x * (i64)blockDim.x + threadIdx.x; c < nChunks; c += (i64)gridDim.x * blockDim.x) {
        i64 lo = 0, hi = nLong - 1;  // last l with long_cptr[l] <= c
        while (lo < hi) {
            i64 mid = (lo + hi + 1) >> 1;
            if (long_cptr[mid] <= (int)c) lo = mid; else hi = mid - 1;
        }
        const int i = long_rows[lo];
        const int s = ptr[i] + ((int)c - long_cptr[lo]) * chunk;
        cstart[c] = s;
        cend[c] = min(s + chunk, ptr[i + 1]);
        crow[c] = i;
    }
}

void tile_free(TileLayout &t) {
    dev_free(&t.long_rows); dev_free(&t.long_cptr); dev_free(&t.chunk_start); dev_free(&t.chunk_end); dev_free(&t.chunk_row);
    t.n_long = 0; t.n_chunks = 0;
}

// chunk lists of the rows that do not fit one tile of the async-copy SpMM
int32_t tile_build(sdplrp_handle *h, Tmp &tmp, i64 n, const int *ptr, TileLayout &t, int chunk) {
    cudaStream_t st = h->stream;
    const int GS = 8 * kNumSM;
    int32_t rc = SDPLRP_OK;
    tile_free(t);
    int *lflag = tmp.get<int>(h, n + 1, &rc), *lpos = tmp.get<int>(h, n + 1, &rc);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemsetAsync(lflag, 0, (size_t)(n + 1) * sizeof(int), st));
    k_len_flag<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, ptr, chunk, lflag); KLAUNCH(h);
    SDP_CHECK(exclusive_scan(h, lflag, lpos, n + 1));
    int nl = 0;
    SDP_CHECK(read_int(h, lpos + n, &nl));
    t.n_long = nl;
    if (nl == 0) return SDPLRP_OK;
    SDP_CHECK(dev_alloc(h, &t.long_rows, nl)); SDP_CHECK(dev_alloc(h, &t.long_cptr, nl + 1));
    int *ccnt = tmp.get<int>(h, nl + 1, &rc);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemsetAsync(ccnt, 0, (size_t)(nl + 1) * sizeof(int), st));
    k_compact_ids<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, lflag, lpos, t.long_rows); KLAUNCH(h);
    k_tile_chunk_counts<<<grid_for(nl, TPB, GS), TPB, 0, st>>>(nl, t.long_rows, ptr, chunk, ccnt); KLAUNCH(h);
    SDP_CHECK(exclusive_scan(h, ccnt, t.long_cptr, nl + 1));
    int nc = 0;
    SDP_CHECK(read_int(h, t.long_cptr + nl, &nc));
    t.n_chunks = nc;
    SDP_CHECK(dev_alloc(h, &t.chunk_start, nc)); SDP_CHECK(dev_alloc(h, &t.chunk_end, nc)); SDP_CHECK(dev_alloc(h, &t.chunk_row, nc));
    k_tile_chunks<<<grid_for(nc, TPB, GS), TPB, 0, st>>>(nc, nl, t.long_rows, t.long_cptr, ptr, chunk, t.chunk_start, t.chunk_end, t.chunk_row);
    KLAUNCH(h);
    return SDPLRP_OK;
}
}  // namespace

// ---- multi-GPU: local view of the objective pattern + halo lists (HaloPlan, common.cuh) -------------------------------
// The round-1 design replicated the pattern and all-gathered the whole direction D (0.7 GB received per rank at 8 GPUs,
// 1.19 ms of a 2.96 ms iteration, fully exposed).  Here every rank keeps the CSR of its OWN rows with the columns renumbered
// to [own rows | hub ghosts | tail ghosts]: a ghost is a row of another rank that some own row gathers.  Per pass each rank
// receives exactly its ghosts (about half of the other ranks' rows on the C5 graph, since most vertices have few neighbours),
// hub class first: the hub part of every block (the first Hq rows: dealt blocks are degree-sorted) is small and is what the
// [own | hub] half of every row needs, so that half of the pass runs while the tail class is still on NVLink.
__global__ void k_mark_need(i64 lnnz, const int *__restrict__ idx, unsigned char *__restrict__ need) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < lnnz; k += (i64)gridDim.x * blockDim.x) need[idx[k]] = 1;
}
// flag[c] = 1 iff label c is a ghost of class `klass` on this rank (flag has n+1 entries, the last stays 0)
__global__ void k_ghost_flags(i64 n, i64 B, int rank, i64 Hq, int klass, const unsigned char *__restrict__ need, int *__restrict__ flag) {
    for (i64 c = blockIdx.x * (i64)blockDim.x + threadIdx.x; c < n; c += (i64)gridDim.x * blockDim.x) {
        const i64 q = c / B, l = c - q * B;
        flag[c] = (need[c] && q != rank && (l < Hq ? 0 : 1) == klass) ? 1 : 0;
    }
}
// e = q * nloc + l: does rank q gather own row l (class klass)?
__global__ void k_send_flags(i64 nloc, int P, i64 n, i64 lo, int rank, i64 Hq, int klass, const unsigned char *__restrict__ need_all,
                             int *__restrict__ flag) {
    const i64 total = (i64)P * nloc;
    for (i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x; e < total; e += (i64)gridDim.x * blockDim.x) {
        const i64 q = e / nloc, l = e - q * nloc;
        flag[e] = (q != rank && need_all[(size_t)q * n + lo + l] && (l < Hq ? 0 : 1) == klass) ? 1 : 0;
    }
}
__global__ void k_send_compact(i64 total, i64 nloc, const int *__restrict__ flag, const int *__restrict__ pos, int *__restrict__ rows) {
    for (i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x; e < total; e += (i64)gridDim.x * blockDim.x)
        if (flag[e]) rows[pos[e]] = (int)(e % nloc);
}
__global__ void k_local_ptr(i64 nloc, const int *__restrict__ ptr_lo, int *__restrict__ lptr) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i <= nloc; i += (i64)gridDim.x * blockDim.x) lptr[i] = ptr_lo[i] - ptr_lo[0];
}
// one thread per own row: [own + hub-ghost columns | tail-ghost columns], each part in ascending label order
__global__ void k_local_rows(i64 nloc, i64 lo, i64 B, int rank, i64 Hq, int ngh0, const int *__restrict__ full_ptr,
                             const int *__restrict__ full_idx, const double *__restrict__ Cfull, const int *__restrict__ gid0,
                             const int *__restrict__ gid1, const int *__restrict__ lptr, int *__restrict__ lmid, int *__restrict__ lidx,
                             double *__restrict__ lval) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < nloc; i += (i64)gridDim.x * blockDim.x) {
        const int beg = full_ptr[lo + i], end = full_ptr[lo + i + 1];
        int nA = 0;
        for (int k = beg; k < end; k++) {
            const i64 c = full_idx[k], q = c / B;
            nA += (q == rank || c - q * B < Hq) ? 1 : 0;
        }
        int pa = lptr[i], pb = lptr[i] + nA;
        lmid[i] = pb;
        for (int k = beg; k < end; k++) {
            const i64 c = full_idx[k], q = c / B, l = c - q * B;
            const double v = Cfull[k];
            if (q == rank) { lidx[pa] = (int)l; lval[pa] = v; pa++; }
            else if (l < Hq) { lidx[pa] = (int)nloc + gid0[c]; lval[pa] = v; pa++; }
            else { lidx[pb] = (int)nloc + ngh0 + gid1[c]; lval[pb] = v; pb++; }
        }
    }
}

void halo_free(sdplrp_handle *h) {
    HaloPlan &p = h->halo;
    dev_free(&p.lptr); dev_free(&p.lmid); dev_free(&p.lidx); dev_free(&p.lval);
    dev_free(&p.send_rows[0]); dev_free(&p.send_rows[1]); dev_free(&p.sendbuf); dev_free(&p.xc);
    dev_free(&p.cls.storage);
    tile_free(p.longs);
    p = HaloPlan();
}

int32_t halo_build(sdplrp_handle *h) {
    halo_free(h);
    const i64 general = h->nA - h->n_sd - (h->obj_mat >= 0 ? 1 : 0);
    if (h->world <= 1 || !h->dealt || !h->equal_blocks || h->obj_mat < 0 || general > 0 || h->n_dynF > 0 || h->nnzF <= 0) return SDPLRP_OK;
    HaloPlan &p = h->halo;
    cudaStream_t st = h->stream;
    const int GS = 8 * kNumSM, P = h->world;
    const i64 n = h->n, B = h->block_rows, lo = h->row_lo, hi = h->row_hi, nloc = hi - lo;
    if (nloc <= 0) return SDPLRP_OK;
    const i64 Hq = std::max<i64>(1, std::min<i64>(B, (B + 11) / 12));   // hub part of every block: its first twelfth
    int k01[2] = {0, 0};
    SDP_CHECK(read_int(h, h->full_ptr + lo, &k01[0]));
    SDP_CHECK(read_int(h, h->full_ptr + hi, &k01[1]));
    const i64 k0 = k01[0], lnnz = (i64)k01[1] - k0;
    Tmp tmp;
    int32_t rc = SDPLRP_OK;
    unsigned char *need = tmp.get<unsigned char>(h, n, &rc), *need_all = tmp.get<unsigned char>(h, (i64)P * n, &rc);
    int *flag = tmp.get<int>(h, std::max<i64>(n + 1, (i64)P * nloc + 1), &rc);
    int *gid[2] = {tmp.get<int>(h, n + 1, &rc), tmp.get<int>(h, n + 1, &rc)};
    int *pos = tmp.get<int>(h, (i64)P * nloc + 1, &rc);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemsetAsync(need, 0, (size_t)n, st));
    if (lnnz > 0) { k_mark_need<<<grid_for(lnnz, TPB, GS), TPB, 0, st>>>(lnnz, h->full_idx + k0, need); KLAUNCH(h); }
    SDP_CHECK(comm_allgather_bytes(h, need, need_all, (size_t)n));
    // ghosts of this rank, numbered per class in label order (= by source rank, then by the source's local row)
    for (int k = 0; k < 2; k++) {
        CUDA_TRY(h, cudaMemsetAsync(flag + n, 0, sizeof(int), st));
        k_ghost_flags<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, B, h->rank, Hq, k, need, flag); KLAUNCH(h);
        SDP_CHECK(exclusive_scan(h, flag, gid[k], n + 1));
        p.recv_off[k].assign((size_t)P + 1, 0);
        for (int q = 0; q <= P; q++) {
            int v = 0;
            SDP_CHECK(read_int(h, gid[k] + std::min<i64>(n, (i64)q * B), &v));
            p.recv_off[k][(size_t)q] = v;
        }
        p.n_ghost[k] = p.recv_off[k][(size_t)P];
    }
    // rows this rank sends, per class, grouped by destination
    for (int k = 0; k < 2; k++) {
        const i64 total = (i64)P * nloc;
        CUDA_TRY(h, cudaMemsetAsync(flag + total, 0, sizeof(int), st));
        k_send_flags<<<grid_for(total, TPB, GS), TPB, 0, st>>>(nloc, P, n, lo, h->rank, Hq, k, need_all, flag); KLAUNCH(h);
        SDP_CHECK(exclusive_scan(h, flag, pos, total + 1));
        p.send_off[k].assign((size_t)P + 1, 0);
        for (int q = 0; q <= P; q++) {
            int v = 0;
            SDP_CHECK(read_int(h, pos + (i64)q * nloc, &v));
            p.send_off[k][(size_t)q] = v;
        }
        p.n_send[k] = p.send_off[k][(size_t)P];
        SDP_CHECK(dev_alloc(h, &p.send_rows[k], std::max<i64>(1, p.n_send[k])));
        if (p.n_send[k] > 0) { k_send_compact<<<grid_for(total, TPB, GS), TPB, 0, st>>>(total, nloc, flag, pos, p.send_rows[k]); KLAUNCH(h); }
    }
    // the local CSR
    SDP_CHECK(dev_alloc(h, &p.lptr, nloc + 1 + 8)); SDP_CHECK(dev_alloc(h, &p.lmid, nloc));
    SDP_CHECK(dev_alloc(h, &p.lidx, lnnz + 8)); SDP_CHECK(dev_alloc(h, &p.lval, lnnz + 8));
    k_local_ptr<<<grid_for(nloc + 1, TPB, GS), TPB, 0, st>>>(nloc, h->full_ptr + lo, p.lptr); KLAUNCH(h);
    k_local_rows<<<grid_for(nloc, 64, 32 * kNumSM), 64, 0, st>>>(nloc, lo, B, h->rank, Hq, (int)p.n_ghost[0], h->full_ptr, h->full_idx, h->Cfull,
                                                                gid[0], gid[1], p.lptr, p.lmid, p.lidx, p.lval);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    SDP_CHECK(build_classes(h, tmp, nloc, p.lptr, p.cls));
    SDP_CHECK(tile_build(h, tmp, nloc, p.lptr, p.longs, kRowWarpMax));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    p.nloc = nloc; p.lnnz = lnnz;
    p.active = true;
    return SDPLRP_OK;
}

void pre_free(sdplrp_handle *h) {
    gather_plan_free(h->full_plan);
    halo_free(h);
    round_free(h);
    tile_free(h->full_long); tile_free(h->dyn_long);
    dev_free(&h->tile_scratch); h->tile_scratch_len = 0;
    dev_free(&h->row_mid); h->row_mid_cols = -1;
    dev_free(&h->triu_colptr); dev_free(&h->triu_rowval);
    if (h->full_ptr == h->ref_full_ptr) { h->full_ptr = nullptr; h->full_idx = nullptr; }  // aliases when not relabeled
    dev_free(&h->full_ptr); dev_free(&h->full_idx); dev_free(&h->ref_full_ptr); dev_free(&h->ref_full_idx);
    dev_free(&h->perm); dev_free(&h->iperm); dev_free(&h->i2r); dev_free(&h->r2i);
    h->relabeled = false; h->dealt = false; h->equal_blocks = false;
    dev_free(&h->mapped); dev_free(&h->S); dev_free(&h->matptr); dev_free(&h->mat_gid); dev_free(&h->ent_slot);
    dev_free(&h->ent_row); dev_free(&h->ent_col); dev_free(&h->ent_one); dev_free(&h->ent_two);
    dev_free(&h->long_mat); dev_free(&h->long_chunk_ptr); dev_free(&h->chunk_mat); dev_free(&h->chunk_part);
    dev_free(&h->triuS_static); dev_free(&h->dyn_slot); dev_free(&h->dyn_ptr); dev_free(&h->dyn_gid);
    dev_free(&h->dyn_val); dev_free(&h->dyn_pos_a); dev_free(&h->dyn_pos_b);
    dev_free(&h->Cfull); dev_free(&h->vf_diag); h->vf_val = 0.0; dev_free(&h->dynS); dev_free(&h->dynrow_ptr); dev_free(&h->dynrow_col); dev_free(&h->dynrow_src);
    dev_free(&h->dyn_diag); dev_free(&h->rowc_ptr); dev_free(&h->rowc_val); dev_free(&h->sd_flag);
    dev_free(&h->cperm); dev_free(&h->dyn_nsd_end);
    h->n_sd = 0; h->n_dyn_nsd = 0;
    dev_free(&h->full_cls.storage); dev_free(&h->dyn_cls.storage);
    h->full_cls = RowClasses(); h->dyn_cls = RowClasses();
    h->CR_valid = h->CD_valid = false;
    h->preprocessed = false;
    h->S_static_valid = false;
}

// Is C = v * (its off-diagonal pattern) + diagonal, with v = +-2^k?  (Unweighted MaxCut: v = 0.25.)  Then the gather pass
// CD = C*D can sum the gathered rows unscaled and multiply by v once per row: scaling by a power of two commutes with
// rounding, so the result has the same bits as the valued sum (barring subnormal or overflowing partial sums).
static int32_t detect_value_free(sdplrp_handle *h, Tmp &tmp) {
    cudaStream_t st = h->stream;
    const i64 n = h->n;
    int32_t rc = SDPLRP_OK;
    int *flag = tmp.get<int>(h, 1, &rc);
    if (rc) return rc;
    const int none = INT_MAX;
    CUDA_TRY(h, cudaMemcpyAsync(flag, &none, sizeof(int), cudaMemcpyHostToDevice, st));
    k_vf_first<<<grid_for(n, TPB, 8 * kNumSM), TPB, 0, st>>>(n, h->full_ptr, h->full_idx, flag); KLAUNCH(h);
    int first = none;
    SDP_CHECK(read_int(h, flag, &first));
    if (first == none) return SDPLRP_OK;   // diagonal C: nothing to gather
    double v = 0.0;
    CUDA_TRY(h, cudaMemcpyAsync(&v, h->Cfull + first, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    int ex = 0;
    if (!std::isnormal(v) || std::fabs(std::frexp(v, &ex)) != 0.5) return SDPLRP_OK;
    SDP_CHECK(dev_alloc(h, &h->vf_diag, n));
    CUDA_TRY(h, cudaMemsetAsync(flag, 0, sizeof(int), st));
    k_vf_check<<<grid_for(n, TPB, 8 * kNumSM), TPB, 0, st>>>(n, h->full_ptr, h->full_idx, h->Cfull, v, h->vf_diag, flag); KLAUNCH(h);
    int bad = 1;
    SDP_CHECK(read_int(h, flag, &bad));
    if (bad) dev_free(&h->vf_diag);
    else h->vf_val = v;
    return SDPLRP_OK;
}

int32_t pre_build(sdplrp_handle *h, i64 n, i64 m, i64 nA, const int64_t *mat_off, const int64_t *I,
                  const int64_t *J, const double *V, const int64_t *gids, bool triplets_on_device) {
    pre_free(h);
    if (n <= 0 || m < 0 || nA < 0) return fail(h, SDPLRP_ERR_ARG, "preprocess: bad sizes");
    if (n >= ((i64)1 << 31) - 1) return fail(h, SDPLRP_ERR_ARG, "preprocess: n must fit int32");
    const i64 nnz = nA > 0 ? mat_off[nA] : 0;
    if (nnz >= ((i64)1 << 31) - 1) return fail(h, SDPLRP_ERR_ARG, "preprocess: total nnz must fit int32");
    for (i64 a = 0; a < nA; a++)
        if (mat_off[a] > mat_off[a + 1] || mat_off[a] < 0) return fail(h, SDPLRP_ERR_ARG, "preprocess: mat_off not monotone");
    h->n = n; h->m = m; h->nA = nA;
    h->obj_mat = -1;
    for (i64 a = 0; a < nA; a++) {
        if (gids[a] < 1 || gids[a] > m + 1) return fail(h, SDPLRP_ERR_ARG, "preprocess: sparse_global_inds out of range");
        if (gids[a] == m + 1) h->obj_mat = (int)a;
    }
    cudaStream_t st = h->stream;
    int32_t rc = SDPLRP_OK;
    Tmp tmp;
    const int GS = 8 * kNumSM;

    // ---- upload the triplets ------------------------------------------------
    int64_t *dI = tmp.get<int64_t>(h, nnz, &rc), *dJ = tmp.get<int64_t>(h, nnz, &rc);
    double *dV = tmp.get<double>(h, nnz, &rc);
    int64_t *dOff = tmp.get<int64_t>(h, nA + 1, &rc), *dG = tmp.get<int64_t>(h, nA, &rc);
    unsigned long long *keyF = tmp.get<unsigned long long>(h, nnz, &rc);
    unsigned long long *keyS = tmp.get<unsigned long long>(h, nnz, &rc);  // sort scratch
    unsigned long long *UF = tmp.get<unsigned long long>(h, nnz, &rc);
    int *flag = tmp.get<int>(h, nnz + 1, &rc), *tpos = tmp.get<int>(h, nnz + 1, &rc);
    int *errw = tmp.get<int>(h, 1, &rc);
    if (rc) return rc;
    if (nnz > 0) {
        // sdplrp_preprocess_device: the triplets were built on this GPU (a device-side problem generator); no host round trip
        const cudaMemcpyKind kind = triplets_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        CUDA_TRY(h, cudaMemcpyAsync(dI, I, (size_t)nnz * 8, kind, st));
        CUDA_TRY(h, cudaMemcpyAsync(dJ, J, (size_t)nnz * 8, kind, st));
        CUDA_TRY(h, cudaMemcpyAsync(dV, V, (size_t)nnz * 8, kind, st));
    }
    if (nA > 0) {
        CUDA_TRY(h, cudaMemcpyAsync(dOff, mat_off, (size_t)(nA + 1) * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(h, cudaMemcpyAsync(dG, gids, (size_t)nA * 8, cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(h, cudaMemsetAsync(errw, 0, sizeof(int), st));
    CUDA_TRY(h, cudaMemsetAsync(flag, 0, (size_t)(nnz + 1) * sizeof(int), st));

    if (h->world > 1) {  // SPMD contract check before anything is built from the data
        unsigned long long *dchk = tmp.get<unsigned long long>(h, 1, &rc);
        if (rc) return rc;
        CUDA_TRY(h, cudaMemsetAsync(dchk, 0, sizeof(unsigned long long), st));
        if (nnz > 0) { k_triplet_checksum<<<GS, TPB, 0, st>>>(nnz, dI, dJ, dV, dchk); KLAUNCH(h); }
        unsigned long long chk = 0ull;
        CUDA_TRY(h, cudaMemcpyAsync(&chk, dchk, sizeof(chk), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(h, cudaStreamSynchronize(st));
        chk ^= (unsigned long long)n * 0x100000001B3ull ^ (unsigned long long)nnz;
        SDP_CHECK(comm_check_same(h, chk, "problem (sdplrp_preprocess triplets)"));
    }

    // ---- keys, triu compaction ---------------------------------------------
    if (nnz > 0) { k_keys<<<GS, TPB, 0, st>>>(nnz, n, dI, dJ, keyF, flag, errw); KLAUNCH(h); }
    SDP_CHECK(exclusive_scan(h, flag, tpos, nnz + 1));
    int Ec_i = 0;
    SDP_CHECK(read_int(h, tpos + nnz, &Ec_i));
    const i64 Ec = Ec_i;
    h->Ec = Ec;
    int herr = 0;
    SDP_CHECK(read_int(h, errw, &herr));
    if (herr & 1) return fail(h, SDPLRP_ERR_ARG, "preprocess: coordinate outside 1..n");

    SDP_CHECK(dev_alloc(h, &h->ent_row, Ec)); SDP_CHECK(dev_alloc(h, &h->ent_col, Ec));
    SDP_CHECK(dev_alloc(h, &h->ent_one, Ec)); SDP_CHECK(dev_alloc(h, &h->ent_two, Ec));
    SDP_CHECK(dev_alloc(h, &h->ent_slot, Ec));
    SDP_CHECK(dev_alloc(h, &h->matptr, nA + 1)); SDP_CHECK(dev_alloc(h, &h->mat_gid, nA));
    unsigned long long *keyT = tmp.get<unsigned long long>(h, Ec, &rc);
    unsigned long long *UT = tmp.get<unsigned long long>(h, Ec, &rc);
    if (rc) return rc;
    if (nnz > 0) {
        k_compact<<<GS, TPB, 0, st>>>(nnz, dI, dJ, dV, flag, tpos, h->ent_row, h->ent_col, h->ent_one, h->ent_two, keyT);
        KLAUNCH(h);
    }
    k_matptr<<<grid_for(nA + 1, TPB, GS), TPB, 0, st>>>(nA, nnz, Ec, dOff, tpos, h->matptr, dG, h->mat_gid);
    KLAUNCH(h);

    // ---- the two sparse() calls: sort + unique (src/preprocess.jl:90,93) ----
    const int end_bit = 32 + bits_for(n);
    i64 nnzT = 0, nnzF = 0;
    SDP_CHECK(sort_unique(h, keyT, keyS, Ec, end_bit, UT, &nnzT));
    SDP_CHECK(sort_unique(h, keyF, keyS, nnz, end_bit, UF, &nnzF));
    h->nnzT = nnzT; h->nnzF = nnzF;

    SDP_CHECK(dev_alloc(h, &h->triu_colptr, n + 1)); SDP_CHECK(dev_alloc(h, &h->triu_rowval, nnzT));
    SDP_CHECK(dev_alloc(h, &h->ref_full_ptr, n + 1 + 8)); SDP_CHECK(dev_alloc(h, &h->ref_full_idx, nnzF + 8));  // slack: gather.cu copies 16-byte aligned spans
    SDP_CHECK(dev_alloc(h, &h->mapped, nnzF)); SDP_CHECK(dev_alloc(h, &h->S, nnzF + 8));
    SDP_CHECK(dev_alloc(h, &h->triuS_static, nnzT));
    k_colptr<<<grid_for(n + 1, TPB, GS), TPB, 0, st>>>(n, nnzT, UT, h->triu_colptr); KLAUNCH(h);
    k_colptr<<<grid_for(n + 1, TPB, GS), TPB, 0, st>>>(n, nnzF, UF, h->ref_full_ptr); KLAUNCH(h);
    if (nnzT > 0) { k_low32<<<GS, TPB, 0, st>>>(nnzT, UT, h->triu_rowval); KLAUNCH(h); }
    if (nnzF > 0) { k_low32<<<GS, TPB, 0, st>>>(nnzF, UF, h->ref_full_idx); KLAUNCH(h); }

    // ---- index maps ----------------------------------------------------------
    if (Ec > 0) { k_nzind<<<GS, TPB, 0, st>>>(Ec, h->ent_row, h->ent_col, h->triu_colptr, h->triu_rowval, h->ent_slot); KLAUNCH(h); }
    if (nnzF > 0) { k_mapped<<<GS, TPB, 0, st>>>(nnzF, UF, h->triu_colptr, h->triu_rowval, h->mapped, errw); KLAUNCH(h); }
    SDP_CHECK(read_int(h, errw, &herr));
    CUDA_TRY(h, cudaMemsetAsync(h->S, 0, (size_t)std::max<i64>(nnzF, 1) * sizeof(double), st));
    const bool asym = (herr & 2) != 0;

    // ---- internal vertex order: descending degree of the aggregated pattern -------
    // Hub rows become a contiguous prefix of every n x r factor (L2-resident gather
    // targets) and the row classes become ranges.  "auto" relabels only skewed patterns
    // (max degree >= 8x the mean): regular / banded patterns keep their natural locality.
    h->relabeled = false;
    h->full_ptr = h->ref_full_ptr; h->full_idx = h->ref_full_idx;
    if (nnzF > 0 && h->relabel_mode != 0) {
        unsigned *dkey = tmp.get<unsigned>(h, n, &rc), *dkey2 = tmp.get<unsigned>(h, n, &rc);
        int *dval = tmp.get<int>(h, n, &rc);
        if (rc) return rc;
        SDP_CHECK(dev_alloc(h, &h->iperm, n)); SDP_CHECK(dev_alloc(h, &h->perm, n));
        k_deg_key<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, h->ref_full_ptr, dkey, dval); KLAUNCH(h);
        h->launches += 4;
        SDP_CHECK(with_cub_temp(h, [&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, dkey, dkey2, dval, h->iperm, (int)n, 0, bits_for(n + 2), st);
        }));
        bool want = h->relabel_mode == 1;
        if (h->relabel_mode < 0) {
            unsigned k0 = 0;
            CUDA_TRY(h, cudaMemcpyAsync(&k0, dkey2, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(h, cudaStreamSynchronize(st));
            const double maxdeg = (double)(n - (i64)k0), mean = (double)nnzF / (double)n;
            want = maxdeg >= 8.0 * mean;
        }
        if (want) {
            h->row_starts.assign((size_t)h->world + 1, 0);
            h->dealt = false;
            if (h->world > 1) {
                int *dealt = tmp.get<int>(h, n, &rc);
                if (rc) return rc;
                const int P = h->world;
                const i64 B = (n + P - 1) / P;
                const int rem = (int)(n % P);
                const i64 lastT = n - (i64)(P - 1) * B;   // rows of the last rank when all others hold exactly B
                h->equal_blocks = lastT >= 1;
                h->block_rows = B;
                k_deal_rows<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, P, B, lastT, rem, h->equal_blocks, h->iperm, dealt); KLAUNCH(h);
                CUDA_TRY(h, cudaMemcpyAsync(h->iperm, dealt, (size_t)n * sizeof(int), cudaMemcpyDeviceToDevice, st));
                for (int q = 0; q < P; q++)
                    h->row_starts[(size_t)q + 1] = h->equal_blocks ? std::min<i64>(n, (i64)(q + 1) * B)
                                                                     : h->row_starts[(size_t)q] + (n - q + P - 1) / P;
                h->dealt = true;
            }
            k_invert_perm<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, h->iperm, h->perm); KLAUNCH(h);
            unsigned long long *ikey = tmp.get<unsigned long long>(h, nnzF, &rc);
            int *ipay = tmp.get<int>(h, nnzF, &rc);
            if (rc) return rc;
            SDP_CHECK(dev_alloc(h, &h->i2r, nnzF)); SDP_CHECK(dev_alloc(h, &h->r2i, nnzF));
            k_internal_keys<<<GS, TPB, 0, st>>>(nnzF, UF, h->perm, ikey, ipay); KLAUNCH(h);
            h->launches += 8;
            // keyF (the unsorted input keys) is dead by now: reuse it as the sorted-key output
            SDP_CHECK(with_cub_temp(h, [&](void *t, size_t &b) {
                return cub::DeviceRadixSort::SortPairs(t, b, ikey, keyF, ipay, h->i2r, (int)nnzF, 0, end_bit, st);
            }));
            k_scatter_inverse<<<GS, TPB, 0, st>>>(nnzF, h->i2r, h->r2i); KLAUNCH(h);
            h->full_ptr = nullptr; h->full_idx = nullptr;
            SDP_CHECK(dev_alloc(h, &h->full_ptr, n + 1 + 8)); SDP_CHECK(dev_alloc(h, &h->full_idx, nnzF + 8));
            k_colptr<<<grid_for(n + 1, TPB, GS), TPB, 0, st>>>(n, nnzF, keyF, h->full_ptr); KLAUNCH(h);
            k_low32<<<GS, TPB, 0, st>>>(nnzF, keyF, h->full_idx); KLAUNCH(h);
            h->relabeled = true;
        } else {
            dev_free(&h->iperm); dev_free(&h->perm);
        }
    }

    // ---- the constraint passes index factor rows: entry coordinates in internal labels
    if (h->relabeled && Ec > 0) {
        k_apply_perm<<<GS, TPB, 0, st>>>(Ec, h->perm, h->ent_row); KLAUNCH(h);
        k_apply_perm<<<GS, TPB, 0, st>>>(Ec, h->perm, h->ent_col); KLAUNCH(h);
    }

    // ---- single-diagonal-entry constraints as per-row lists + the internal constraint order --------
    // Constraints that are one diagonal entry (Diag(X) = 1 ...) are numbered first, in internal row order, so
    // that constraint p of row i sits at rowc_ptr[i] <= p < rowc_ptr[i+1] and every m-vector (lambda, y,
    // residuals, A_RD, A_DD) streams together with the factor rows; all other constraints follow in their
    // original order; the objective keeps slot m.  Invisible at the ABI (perm.cu converts m-vectors).
    h->n_sd = 0;
    SDP_CHECK(dev_alloc(h, &h->rowc_ptr, n + 1));
    SDP_CHECK(dev_alloc(h, &h->sd_flag, nA));
    SDP_CHECK(dev_alloc(h, &h->cperm, m + 1));
    CUDA_TRY(h, cudaMemsetAsync(h->rowc_ptr, 0, (size_t)(n + 1) * sizeof(int), st));
    {
        int *assigned = tmp.get<int>(h, m + 1, &rc), *unassigned = tmp.get<int>(h, m + 1, &rc), *crank = tmp.get<int>(h, m + 1, &rc);
        if (rc) return rc;
        CUDA_TRY(h, cudaMemsetAsync(assigned, 0, (size_t)(m + 1) * sizeof(int), st));
        if (nA > 0) {
            unsigned *skey = tmp.get<unsigned>(h, nA, &rc), *skey2 = tmp.get<unsigned>(h, nA, &rc);
            int *sval = tmp.get<int>(h, nA, &rc), *sval2 = tmp.get<int>(h, nA, &rc);
            if (rc) return rc;
            k_sd_keys<<<grid_for(nA, TPB, GS), TPB, 0, st>>>(nA, n, h->obj_mat, h->matptr, h->ent_row, h->ent_col, skey, sval, h->sd_flag);
            KLAUNCH(h);
            h->launches += 4;
            SDP_CHECK(with_cub_temp(h, [&](void *t, size_t &b) {
                return cub::DeviceRadixSort::SortPairs(t, b, skey, skey2, sval, sval2, (int)nA, 0, bits_for(n + 2), st);
            }));
            k_lower_bound_u32<<<grid_for(n + 1, TPB, GS), TPB, 0, st>>>(n, nA, skey2, h->rowc_ptr); KLAUNCH(h);
            int nsd = 0;
            SDP_CHECK(read_int(h, h->rowc_ptr + n, &nsd));
            h->n_sd = nsd;
            SDP_CHECK(dev_alloc(h, &h->rowc_val, nsd));
            if (nsd > 0) {
                k_sd_vals<<<grid_for(nsd, TPB, GS), TPB, 0, st>>>(nsd, sval2, h->matptr, h->ent_two, h->rowc_val); KLAUNCH(h);
                k_cperm_sd<<<grid_for(nsd, TPB, GS), TPB, 0, st>>>(nsd, sval2, h->mat_gid, h->cperm, assigned); KLAUNCH(h);
            }
        }
        k_not<<<grid_for(m + 1, TPB, GS), TPB, 0, st>>>(m + 1, assigned, unassigned); KLAUNCH(h);
        SDP_CHECK(exclusive_scan(h, unassigned, crank, m + 1));
        k_cperm_rest<<<grid_for(m + 1, TPB, GS), TPB, 0, st>>>(m, h->n_sd, assigned, crank, h->cperm); KLAUNCH(h);
        if (nA > 0) { k_apply_perm<<<grid_for(nA, TPB, GS), TPB, 0, st>>>(nA, h->cperm, h->mat_gid); KLAUNCH(h); }  // mat_gid -> internal slots
        CUDA_TRY(h, cudaStreamSynchronize(st));
    }

    // ---- long matrices -> chunk lists (constraint passes) --------------------
    h->n_long = 0; h->n_chunks = 0;
    if (nA > 0) {
        int *lflag = tmp.get<int>(h, nA + 1, &rc), *lpos = tmp.get<int>(h, nA + 1, &rc);
        if (rc) return rc;
        CUDA_TRY(h, cudaMemsetAsync(lflag, 0, (size_t)(nA + 1) * sizeof(int), st));
        k_len_flag<<<grid_for(nA, TPB, GS), TPB, 0, st>>>(nA, h->matptr, kLongMatThreshold, lflag); KLAUNCH(h);
        SDP_CHECK(exclusive_scan(h, lflag, lpos, nA + 1));
        int nl = 0;
        SDP_CHECK(read_int(h, lpos + nA, &nl));
        h->n_long = nl;
        if (nl > 0) {
            SDP_CHECK(dev_alloc(h, &h->long_mat, nl)); SDP_CHECK(dev_alloc(h, &h->long_chunk_ptr, nl + 1));
            int *ccnt = tmp.get<int>(h, nl + 1, &rc);
            if (rc) return rc;
            CUDA_TRY(h, cudaMemsetAsync(ccnt, 0, (size_t)(nl + 1) * sizeof(int), st));
            k_compact_ids<<<grid_for(nA, TPB, GS), TPB, 0, st>>>(nA, lflag, lpos, h->long_mat); KLAUNCH(h);
            k_chunk_counts<<<grid_for(nl, TPB, GS), TPB, 0, st>>>(nl, h->long_mat, h->matptr, kChunkEntries, ccnt); KLAUNCH(h);
            SDP_CHECK(exclusive_scan(h, ccnt, h->long_chunk_ptr, nl + 1));
            int nc = 0;
            SDP_CHECK(read_int(h, h->long_chunk_ptr + nl, &nc));
            h->n_chunks = nc;
            SDP_CHECK(dev_alloc(h, &h->chunk_mat, nc)); SDP_CHECK(dev_alloc(h, &h->chunk_part, (i64)nc * 2));
            k_chunk_mat<<<grid_for(nc, TPB, GS), TPB, 0, st>>>(nc, nl, h->long_chunk_ptr, h->chunk_mat); KLAUNCH(h);
        }
    }

    // ---- S assembly layout: static objective part + dynamic slots -----------
    h->n_dyn = 0;
    if (Ec > 0) {
        int *ent_mat = tmp.get<int>(h, Ec, &rc), *iota = tmp.get<int>(h, Ec, &rc);
        int *sorted_slot = tmp.get<int>(h, Ec, &rc), *sorted_t = tmp.get<int>(h, Ec, &rc);
        int *slot_ptr = tmp.get<int>(h, nnzT + 1, &rc);
        int *dcnt = tmp.get<int>(h, nnzT + 1, &rc), *dflag = tmp.get<int>(h, nnzT + 1, &rc);
        int *dindex = tmp.get<int>(h, nnzT + 1, &rc), *doff = tmp.get<int>(h, nnzT + 1, &rc);
        if (rc) return rc;
        k_ent_mat<<<GS, TPB, 0, st>>>(Ec, nA, h->matptr, ent_mat); KLAUNCH(h);
        k_iota<<<GS, TPB, 0, st>>>(Ec, iota); KLAUNCH(h);
        h->launches += 4;
        SDP_CHECK(with_cub_temp(h, [&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, reinterpret_cast<const unsigned *>(h->ent_slot),
                                                   reinterpret_cast<unsigned *>(sorted_slot), iota, sorted_t, (int)Ec, 0,
                                                   bits_for(nnzT + 1), st);
        }));
        k_slot_ptr<<<grid_for(nnzT + 1, TPB, GS), TPB, 0, st>>>(nnzT, Ec, sorted_slot, slot_ptr); KLAUNCH(h);
        CUDA_TRY(h, cudaMemsetAsync(dcnt, 0, (size_t)(nnzT + 1) * sizeof(int), st));
        CUDA_TRY(h, cudaMemsetAsync(dflag, 0, (size_t)(nnzT + 1) * sizeof(int), st));
        k_slot_classify<<<GS, TPB, 0, st>>>(nnzT, slot_ptr, sorted_t, ent_mat, h->ent_one, h->obj_mat, h->triuS_static, dcnt, dflag);
        KLAUNCH(h);
        SDP_CHECK(exclusive_scan(h, dflag, dindex, nnzT + 1));
        SDP_CHECK(exclusive_scan(h, dcnt, doff, nnzT + 1));
        int nd = 0, ndc = 0;
        SDP_CHECK(read_int(h, dindex + nnzT, &nd));
        SDP_CHECK(read_int(h, doff + nnzT, &ndc));
        h->n_dyn = nd;
        SDP_CHECK(dev_alloc(h, &h->dyn_slot, nd)); SDP_CHECK(dev_alloc(h, &h->dyn_ptr, nd + 1)); SDP_CHECK(dev_alloc(h, &h->dyn_nsd_end, nd));
        SDP_CHECK(dev_alloc(h, &h->dyn_gid, ndc)); SDP_CHECK(dev_alloc(h, &h->dyn_val, ndc));
        SDP_CHECK(dev_alloc(h, &h->dyn_pos_a, nd)); SDP_CHECK(dev_alloc(h, &h->dyn_pos_b, nd));
        if (nd > 0) {
            k_dyn_fill<<<GS, TPB, 0, st>>>(nnzT, slot_ptr, sorted_t, ent_mat, h->ent_one, h->mat_gid, h->obj_mat, dflag,
                                           dindex, doff, h->triu_rowval, UT, h->relabeled ? h->perm : nullptr, h->full_ptr, h->full_idx, h->sd_flag,
                                           h->dyn_slot, h->dyn_ptr, h->dyn_nsd_end, h->dyn_gid, h->dyn_val, h->dyn_pos_a, h->dyn_pos_b);
            KLAUNCH(h);
        }
        h->n_dyn_nsd = (i64)ndc - h->n_sd;  // contributors that are not single-diagonal-entry constraints (each of those has exactly one)
        CUDA_TRY(h, cudaMemcpyAsync(h->dyn_ptr + nd, &ndc, sizeof(int), cudaMemcpyHostToDevice, st));
        CUDA_TRY(h, cudaStreamSynchronize(st));
    }

    // ---- objective values on the full pattern + the dynamic pattern as CSR -------
    SDP_CHECK(dev_alloc(h, &h->Cfull, nnzF + 8));
    SDP_CHECK(dev_alloc(h, &h->dynS, h->n_dyn));
    SDP_CHECK(dev_alloc(h, &h->dynrow_ptr, n + 1));
    SDP_CHECK(dev_alloc(h, &h->dyn_diag, n));
    k_fill_int<<<grid_for(n, TPB, GS), TPB, 0, st>>>(n, -1, h->dyn_diag); KLAUNCH(h);
    h->n_dynF = 0;
    if (nnzF > 0) {
        k_cfull<<<GS, TPB, 0, st>>>(nnzF, h->mapped, h->i2r, h->triuS_static, h->Cfull); KLAUNCH(h);
        if (h->obj_mat >= 0) SDP_CHECK(detect_value_free(h, tmp));
        int *fflag = tmp.get<int>(h, nnzF + 1, &rc), *fpos = tmp.get<int>(h, nnzF + 1, &rc), *fsrc = tmp.get<int>(h, nnzF + 1, &rc);
        if (rc) return rc;
        CUDA_TRY(h, cudaMemsetAsync(fflag, 0, (size_t)(nnzF + 1) * sizeof(int), st));
        if (h->n_dyn > 0) { k_dyn_mark<<<GS, TPB, 0, st>>>(h->n_dyn, h->dyn_pos_a, h->dyn_pos_b, h->full_idx, h->dyn_ptr, h->dyn_nsd_end, fflag, fsrc, h->dyn_diag); KLAUNCH(h); }
        SDP_CHECK(exclusive_scan(h, fflag, fpos, nnzF + 1));
        int ndf = 0;
        SDP_CHECK(read_int(h, fpos + nnzF, &ndf));
        h->n_dynF = ndf;
        SDP_CHECK(dev_alloc(h, &h->dynrow_col, ndf)); SDP_CHECK(dev_alloc(h, &h->dynrow_src, ndf));
        if (ndf > 0) { k_dyn_rows<<<GS, TPB, 0, st>>>(nnzF, fflag, fpos, fsrc, h->full_idx, h->dynrow_col, h->dynrow_src); KLAUNCH(h); }
        k_gather_ptr<<<grid_for(n + 1, TPB, GS), TPB, 0, st>>>(n, h->full_ptr, fpos, h->dynrow_ptr); KLAUNCH(h);
    } else {
        CUDA_TRY(h, cudaMemsetAsync(h->dynrow_ptr, 0, (size_t)(n + 1) * sizeof(int), st));
        SDP_CHECK(dev_alloc(h, &h->dynrow_col, 0)); SDP_CHECK(dev_alloc(h, &h->dynrow_src, 0));
    }

    // ---- row bins of both patterns (sparse x dense kernels) -----------------------
    SDP_CHECK(build_classes(h, tmp, n, h->full_ptr, h->full_cls));
    SDP_CHECK(build_classes(h, tmp, n, h->dynrow_ptr, h->dyn_cls));
    // rows of the third class (> kRowWarpMax nonzeros) cut into chunks of kRowWarpMax for the register kernels
    SDP_CHECK(tile_build(h, tmp, n, h->full_ptr, h->full_long, kRowWarpMax));
    SDP_CHECK(tile_build(h, tmp, n, h->dynrow_ptr, h->dyn_long, kRowWarpMax));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    CUDA_TRY(h, cudaGetLastError());
    h->preprocessed = true;
    h->S_static_valid = false;
    h->row_lo = 0; h->row_hi = n;
    if (asym) {
        h->err = "preprocess: a lower-triangular entry has no mirrored upper entry (maps exported with 0 there)";
        return SDPLRP_ERR_ASYMMETRIC;
    }
    return SDPLRP_OK;
}

int32_t pre_export(sdplrp_handle *h, int64_t *triu_colptr, int64_t *triu_rowval, int64_t *matptr, int64_t *nzind,
                   double *one, double *two, int64_t *full_colptr, int64_t *full_rowval, int64_t *mapped) {
    cudaStream_t st = h->stream;
    const i64 n = h->n, nA = h->nA, nnzT = h->nnzT, nnzF = h->nnzF, Ec = h->Ec;
    i64 maxlen = std::max(std::max(n + 1, nA + 1), std::max(std::max(nnzT, nnzF), Ec));
    int64_t *buf = nullptr;
    CUDA_TRY(h, cudaMalloc((void **)&buf, (size_t)std::max<i64>(maxlen, 1) * sizeof(int64_t)));
    struct Item { const int *src; int64_t *dst; i64 len; };
    Item items[] = {{h->triu_colptr, triu_colptr, n + 1}, {h->triu_rowval, triu_rowval, nnzT}, {h->matptr, matptr, nA + 1},
                    {h->ent_slot, nzind, Ec}, {h->ref_full_ptr, full_colptr, n + 1}, {h->ref_full_idx, full_rowval, nnzF},
                    {h->mapped, mapped, nnzF}};
    int32_t rc = SDPLRP_OK;
    for (const Item &it : items) {
        if (!it.dst || it.len <= 0) continue;
        k_export_i32<<<grid_for(it.len, TPB, 8 * kNumSM), TPB, 0, st>>>(it.len, it.src, buf);
        KLAUNCH(h);
        cudaError_t e = cudaMemcpyAsync(it.dst, buf, (size_t)it.len * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { h->err = std::string("pattern_export: ") + cudaGetErrorString(e); rc = SDPLRP_ERR_CUDA; break; }
    }
    cudaFree(buf);
    if (rc) return rc;
    if (one && Ec > 0) CUDA_TRY(h, cudaMemcpy(one, h->ent_one, (size_t)Ec * 8, cudaMemcpyDeviceToHost));
    if (two && Ec > 0) CUDA_TRY(h, cudaMemcpy(two, h->ent_two, (size_t)Ec * 8, cudaMemcpyDeviceToHost));
    return SDPLRP_OK;
}
