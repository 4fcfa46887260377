// rounding.cu -- hyperplane (Goemans-Williamson) rounding of the factor R into +-1 vectors, best of K candidates.
//
// Candidates go in batches of kRoundB = 64, one bit per candidate in a 64-bit word per vertex (internal order):
//   sign pass   k_round_sign: every owned row of R is read once, its 64 dots <R_i, g_k> are formed against the batch's
//               hyperplanes (in shared memory) and bit k of word_i is set when <R_i, g_k> >= 0.  The per-candidate counts
//               of set bits are fused in through the deterministic grid reduction.  2*64*r flops per 8r bytes of R.
//   eval pass   k_round_eval: over the nonzeros of the owned rows of the full pattern, t = w_i ^ w_j, and C_ij is added to
//               every candidate whose bit of t is set (x_i x_j = -1 there).  obj_k = sum(C) - 2 * that sum.
// Several GPUs: the words are all-gathered by row block after the sign pass, every rank evaluates its own rows of the
// replicated full pattern, and the 2K partial sums (set bits, eval sums) are all-reduced once at the end.
// Nothing outside the rounding buffers (h->rnd) and the reduction scratch is written.
#include <math.h>
#include <algorithm>
#include <vector>
#include "common.cuh"

namespace {
constexpr int kRoundB = 64;        // candidates per batch = bits of a word
constexpr int kSignTPB = 128;
constexpr int kSignCols = 32;      // columns of the batch's hyperplanes held in shared memory at a time
constexpr int kEvalTPB = 128;
constexpr int kEvalChunk = 32;     // nonzeros per thread chunk of the evaluation pass
typedef unsigned long long Word;

// words[i] bit k = (<R_i, g_k> >= 0) for the owned rows; cnt[k] = number of set bits over them (k < 64)
__global__ void __launch_bounds__(kSignTPB) k_round_sign(i64 row_lo, i64 nrows, int r, const double *__restrict__ R,
                                                          const double *__restrict__ G, int nb, Word *__restrict__ words,
                                                          double *partials, unsigned *ticket, double *cnt_out) {
    __shared__ double Gs[kSignCols][kRoundB];
    const int lane = threadIdx.x & 31;
    unsigned cnt[2] = {0u, 0u};  // candidates lane and lane + 32 of this warp
    const bool single = r <= kSignCols;
    auto load_cols = [&](int c0) {
        const int nc = min(kSignCols, r - c0);
        for (int e = threadIdx.x; e < kSignCols * kRoundB; e += blockDim.x) {
            const int c = e / kRoundB, k = e - c * kRoundB;
            Gs[c][k] = (c < nc && k < nb) ? G[(size_t)k * r + c0 + c] : 0.0;
        }
    };
    if (single) { load_cols(0); __syncthreads(); }
    for (i64 base = (i64)blockIdx.x * blockDim.x; base < nrows; base += (i64)gridDim.x * blockDim.x) {
        const i64 i = base + threadIdx.x;
        const bool valid = i < nrows;
        const double *Ri = R + (size_t)(row_lo + (valid ? i : 0)) * r;
        double acc[kRoundB];
#pragma unroll
        for (int k = 0; k < kRoundB; k++) acc[k] = 0.0;
        for (int c0 = 0; c0 < r; c0 += kSignCols) {
            if (!single) { __syncthreads(); load_cols(c0); __syncthreads(); }
            const int nc = min(kSignCols, r - c0);
            if (valid) {
                for (int c = 0; c < nc; c++) {
                    const double x = Ri[c0 + c];
#pragma unroll
                    for (int k = 0; k < kRoundB; k++) acc[k] = fma(x, Gs[c][k], acc[k]);
                }
            }
        }
        Word w = 0ull;
#pragma unroll
        for (int k = 0; k < kRoundB; k++) w |= (Word)(acc[k] >= 0.0) << k;
        if (!valid) w = 0ull;
        else words[row_lo + i] = w;
#pragma unroll
        for (int k = 0; k < kRoundB; k++) {
            const unsigned c = __popc(__ballot_sync(0xffffffffu, (w >> k) & 1ull));
            if (lane == (k & 31)) cnt[k >> 5] += c;
        }
    }
    double v[kRoundB];
#pragma unroll
    for (int k = 0; k < kRoundB; k++) v[k] = lane == (k & 31) ? (double)cnt[k >> 5] : 0.0;
    grid_sum_finalize<kRoundB>(v, partials, ticket, [&](double (&s)[kRoundB]) {
#pragma unroll
        for (int k = 0; k < kRoundB; k++) if (k < nb) cnt_out[k] = s[k];
    });
}

// first owned row of every chunk of kEvalChunk nonzeros (chunk c starts at nonzero e_lo + c * kEvalChunk)
__global__ void k_round_chunk_rows(i64 row_lo, i64 row_hi, i64 e_lo, const int *__restrict__ ptr, int *__restrict__ chunk_row) {
    for (i64 i = row_lo + blockIdx.x * (i64)blockDim.x + threadIdx.x; i < row_hi; i += (i64)gridDim.x * blockDim.x) {
        const i64 a = ptr[i] - e_lo, b = ptr[i + 1] - e_lo;
        for (i64 c = (a + kEvalChunk - 1) / kEvalChunk; c * kEvalChunk < b; c++) chunk_row[c] = (int)i;
    }
}

// sums[k] = sum of C_ij over the owned nonzeros with bit k of (w_i ^ w_j) set.  Per-thread register accumulators for the
// 64 candidates: the candidate loop is unrolled into predicated adds, and a nonzero costs one gathered word, not a
// shared-memory broadcast per candidate.  The chunk -> thread map is fixed, so the sums are bit-reproducible.
__global__ void __launch_bounds__(kEvalTPB) k_round_eval(i64 e_lo, i64 e_hi, i64 nchunks, const int *__restrict__ ptr,
                                                          const int *__restrict__ idx, const double *__restrict__ val,
                                                          const int *__restrict__ chunk_row, const Word *__restrict__ words, int nb,
                                                          double *partials, unsigned *ticket, double *sums_out) {
    double acc[kRoundB];
#pragma unroll
    for (int k = 0; k < kRoundB; k++) acc[k] = 0.0;
    for (i64 c = blockIdx.x * (i64)blockDim.x + threadIdx.x; c < nchunks; c += (i64)gridDim.x * blockDim.x) {
        const i64 e0 = e_lo + c * kEvalChunk, e1 = min(e0 + kEvalChunk, e_hi);
        i64 row = chunk_row[c];
        i64 rend = ptr[row + 1];
        Word wi = words[row];
        // one nonzero of look-ahead: its column word is in flight while the current one is accumulated
        int j = idx[e0];
        double v = val[e0];
        Word wj = words[j];
        for (i64 e = e0; e < e1; e++) {
            int jn = 0;
            double vn = 0.0;
            Word wn = 0ull;
            if (e + 1 < e1) { jn = idx[e + 1]; vn = val[e + 1]; wn = words[jn]; }
            while (e >= rend) { row++; rend = ptr[row + 1]; wi = words[row]; }
            const Word t = wi ^ wj;
            const unsigned lo = (unsigned)t, hi = (unsigned)(t >> 32);
#pragma unroll
            for (int k = 0; k < 32; k++) {
                if (lo & (1u << k)) acc[k] += v;
                if (hi & (1u << k)) acc[32 + k] += v;
            }
            j = jn; v = vn; wj = wn;
        }
    }
    grid_sum_finalize<kRoundB>(acc, partials, ticket, [&](double (&s)[kRoundB]) {
#pragma unroll
        for (int k = 0; k < kRoundB; k++) if (k < nb) sums_out[k] = s[k];
    });
}

__global__ void __launch_bounds__(256) k_round_csum(i64 len, const double *__restrict__ val, double *partials, unsigned *ticket,
                                                    double *out) {
    double acc[1] = {0.0};
    for (i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x; e < len; e += (i64)gridDim.x * blockDim.x) acc[0] += val[e];
    grid_sum_finalize<1>(acc, partials, ticket, [&](double (&s)[1]) { out[0] = s[0]; });
}

// x[i] = +1 / -1 from bit b of word i (every row: the words are complete on every rank)
__global__ void k_round_expand(i64 n, const Word *__restrict__ words, int b, double *__restrict__ x) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x)
        x[i] = ((words[i] >> b) & 1ull) ? 1.0 : -1.0;
}

unsigned long long mix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// standard normal keyed by (seed, candidate, column) (counter-based hash + Box-Muller): independent of K, of the vertex
// order and of the number of GPUs
double hyperplane_normal(unsigned long long seed, i64 k, i64 c) {
    const unsigned long long base = mix64(seed ^ mix64(0xA0761D6478BD642Full * (unsigned long long)(k + 1)));
    const unsigned long long a = mix64(base ^ (2ull * (unsigned long long)c));
    const unsigned long long b = mix64(base ^ (2ull * (unsigned long long)c + 1ull));
    const double u1 = ((double)(a >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    const double u2 = (double)(b >> 11) * (1.0 / 9007199254740992.0);
    return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
}

int32_t ensure(sdplrp_handle *h, double **p, i64 *cap, i64 len) {
    if (*cap >= len) return SDPLRP_OK;
    SDP_CHECK(dev_alloc(h, p, len));
    *cap = len;
    return SDPLRP_OK;
}

// the problem-sized buffers: words (n), x scratch (n), chunk -> row map of the owned nonzeros (first use after preprocessing)
int32_t ensure_problem_buffers(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    if (s.words) return SDPLRP_OK;
    SDP_CHECK(dev_alloc(h, &s.words, h->n));
    SDP_CHECK(dev_alloc(h, &s.x, h->n));
    int e[2] = {0, 0};
    CUDA_TRY(h, cudaMemcpyAsync(&e[0], h->full_ptr + h->row_lo, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(&e[1], h->full_ptr + h->row_hi, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    s.e_lo = e[0]; s.e_hi = e[1];
    s.nchunks = (s.e_hi - s.e_lo + kEvalChunk - 1) / kEvalChunk;
    SDP_CHECK(dev_alloc(h, &s.chunk_row, s.nchunks));
    if (h->row_hi > h->row_lo) {
        k_round_chunk_rows<<<grid_for(h->row_hi - h->row_lo, 256, kRedBlocks * 4), 256, 0, h->stream>>>(h->row_lo, h->row_hi, s.e_lo,
                                                                                                     h->full_ptr, s.chunk_row);
        KLAUNCH(h);
        CUDA_TRY(h, cudaGetLastError());
    }
    return SDPLRP_OK;
}

int32_t sign_pass(sdplrp_handle *h, const double *dG, int nb, double *cnt_out) {
    const i64 nrows = h->row_hi - h->row_lo;
    k_round_sign<<<grid_for(std::max<i64>(nrows, 1), kSignTPB, 2 * kRedBlocks), kSignTPB, 0, h->stream>>>(
        h->row_lo, nrows, h->r, h->R, dG, nb, h->rnd.words, h->partials, h->ticket, cnt_out);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}
}  // namespace

void round_free(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    if (s.words) { cudaFree(s.words); s.words = nullptr; }
    dev_free(&s.x); dev_free(&s.chunk_row); dev_free(&s.G); dev_free(&s.sums);
    s.G_len = s.sums_len = 0;
    s.e_lo = s.e_hi = s.nchunks = 0;
}

extern "C" int32_t sdplrp_round_hyperplane(sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, double *G_out, double *obj,
                                           double *sum, int64_t *best, double *best_x) {
    if (!h) return SDPLRP_ERR_ARG;
    if (!h->preprocessed) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_preprocess first");
    if (h->r <= 0) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_set_rank first");
    if (K < 1 || !obj || !best) return fail(h, SDPLRP_ERR_ARG, "round_hyperplane: K >= 1 and the obj / best outputs are required");
    for (const LowRank &L : h->lr)
        if (L.gid == h->m) return fail(h, SDPLRP_ERR_ARG, "round_hyperplane: the objective has a low-rank part");
    if (h->obj_mat < 0) return fail(h, SDPLRP_ERR_ARG, "round_hyperplane: needs a sparse objective");
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int r = h->r;
    const i64 n = h->n;

    // hyperplanes on the host: the caller's, or the counter-based normals
    std::vector<double> Gh;
    if (!G) {
        Gh.resize((size_t)K * r);
        for (i64 k = 0; k < K; k++)
            for (int c = 0; c < r; c++) Gh[(size_t)k * r + c] = hyperplane_normal(seed, k, c);
        G = Gh.data();
    }
    if (h->world > 1) {   // SPMD: every rank must round with the same K and the same hyperplanes
        unsigned long long cs = mix64((unsigned long long)K);
        const unsigned long long *bits = reinterpret_cast<const unsigned long long *>(G);
        for (i64 e = 0; e < K * r; e++) cs = mix64(cs ^ bits[e]);
        SDP_CHECK(comm_check_same(h, cs, "hyperplanes (K, seed, G)"));
    }

    RoundingState &s = h->rnd;
    SDP_CHECK(ensure_problem_buffers(h));
    SDP_CHECK(ensure(h, &s.G, &s.G_len, K * r));
    SDP_CHECK(ensure(h, &s.sums, &s.sums_len, 2 * K + 1));
    CUDA_TRY(h, cudaMemcpyAsync(s.G, G, (size_t)(K * r) * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    double *cnt = s.sums, *esum = s.sums + K, *csum = s.sums + 2 * K;
    k_round_csum<<<kRedBlocks, 256, 0, h->stream>>>(h->nnzF, h->Cfull, h->partials, h->ticket, csum);   // replicated: same bits everywhere
    KLAUNCH(h);
    const i64 nbatch = (K + kRoundB - 1) / kRoundB;
    for (i64 bt = 0; bt < nbatch; bt++) {
        const int nb = (int)std::min<i64>(kRoundB, K - bt * kRoundB);
        const double *dG = s.G + (size_t)(bt * kRoundB) * r;
        SDP_CHECK(sign_pass(h, dG, nb, cnt + bt * kRoundB));
        SDP_CHECK(comm_gather_rowbytes(h, s.words, sizeof(Word)));
        if (s.nchunks > 0) {
            k_round_eval<<<grid_for(s.nchunks, kEvalTPB, 2 * kRedBlocks), kEvalTPB, 0, h->stream>>>(
                s.e_lo, s.e_hi, s.nchunks, h->full_ptr, h->full_idx, h->Cfull, s.chunk_row, s.words, nb, h->partials, h->ticket,
                esum + bt * kRoundB);
            KLAUNCH(h);
        } else {
            CUDA_TRY(h, cudaMemsetAsync(esum + bt * kRoundB, 0, (size_t)nb * sizeof(double), h->stream));
        }
        CUDA_TRY(h, cudaGetLastError());
    }
    SDP_CHECK(comm_reduce_ptr(h, s.sums, (int)(2 * K)));
    std::vector<double> hs((size_t)(2 * K + 1));
    CUDA_TRY(h, cudaMemcpyAsync(hs.data(), s.sums, hs.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));

    const double sumC = hs[(size_t)(2 * K)];
    i64 kb = 0;
    for (i64 k = 0; k < K; k++) {
        obj[k] = sumC - 2.0 * hs[(size_t)(K + k)];
        if (sum) sum[k] = 2.0 * hs[(size_t)k] - (double)n;
        if (obj[k] < obj[kb]) kb = k;
    }
    *best = kb + 1;
    if (G_out) std::copy(G, G + (size_t)(K * r), G_out);
    if (best_x) {
        const i64 bt = kb / kRoundB;
        if (bt != nbatch - 1) {   // the words of that batch were overwritten: the same kernel on the same data gives the same bits
            const int nb = (int)std::min<i64>(kRoundB, K - bt * kRoundB);
            SDP_CHECK(sign_pass(h, s.G + (size_t)(bt * kRoundB) * r, nb, cnt + bt * kRoundB));
            SDP_CHECK(comm_gather_rowbytes(h, s.words, sizeof(Word)));
        }
        k_round_expand<<<grid_for(n, 256, kRedBlocks * 4), 256, 0, h->stream>>>(n, s.words, (int)(kb - bt * kRoundB), s.x);
        KLAUNCH(h);
        CUDA_TRY(h, cudaGetLastError());
        SDP_CHECK(perm_download(h, s.x, best_x, 1, true));
    }
    return SDPLRP_OK;
}
