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
//
// One-flip local search (sdplrp_round_local_search) runs on the same words between two evaluation passes.  Round t:
//   want pass   k_ls_want (+ k_ls_want_seg / k_ls_want_combine for long rows): for every owned row flagged dirty,
//               h_ik = sum_{j != i, C_ij != 0} C_ij x_jk for the 64 candidates, and bit k of want_i = (x_ik h_ik > 0).
//               A row that is not dirty keeps its want word: it depends only on x_i and the x_j of its neighbours.
//   flip pass   k_ls_flip (+ k_ls_flip_seg): flip_i = want_i & ~OR{want_j : j a neighbour with a higher priority}, and the
//               per-candidate counts of wanting vertices.  The flipped vertices of a candidate are pairwise non-adjacent,
//               so their gains add up and the objective falls by 4 sum |h_ik| every round.
//   apply pass  k_ls_apply (+ k_ls_apply_seg): word_i ^= flip_i on every row, per-candidate flip counts over the owned
//               rows, and a flipped row marks itself and its neighbours dirty (identical byte stores).
// Rows with more than kLsLong nonzeros are cut into segments of kLsSeg nonzeros, one CTA each; the want sums of a long row
// are combined over its segments in a fixed order.
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
constexpr int kLsTPB = 128;
constexpr int kLsLong = 128;       // local search: rows with more nonzeros than this go to the segment kernels
constexpr int kLsSeg = 4096;       // nonzeros per segment (one CTA) of a long row
typedef unsigned long long Word;

__host__ __device__ inline unsigned long long mix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// cnt[k >> 5] of lane (k & 31) += number of lanes of the warp with bit k of w set (all 32 lanes call it)
__device__ __forceinline__ void ballot_counts(Word w, int lane, unsigned (&cnt)[2]) {
#pragma unroll
    for (int k = 0; k < kRoundB; k++) {
        const unsigned c = __popc(__ballot_sync(0xffffffffu, (w >> k) & 1ull));
        if (lane == (k & 31)) cnt[k >> 5] += c;
    }
}

// the ballot counts of a thread as the 64 per-thread values of a grid reduction
__device__ __forceinline__ void counts_to_values(const unsigned (&cnt)[2], int lane, double (&v)[kRoundB]) {
#pragma unroll
    for (int k = 0; k < kRoundB; k++) v[k] = lane == (k & 31) ? (double)cnt[k >> 5] : 0.0;
}

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
        ballot_counts(w, lane, cnt);
    }
    double v[kRoundB];
    counts_to_values(cnt, lane, v);
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

// ---- one-flip local search --------------------------------------------------------------------------------------------
// priority of the vertex with internal label i in a round: mix64(ref ^ salt), ref = its input label (iperm[i]),
// salt = mix64(0xD1B54A32D192ED03 * (t + 1)).  No candidate index enters it: candidate k's descent does not depend on K.
__device__ __forceinline__ Word ls_key(const int *__restrict__ iperm, i64 i, Word salt, Word &ref) {
    ref = iperm ? (Word)iperm[i] : (Word)i;
    return mix64(ref ^ salt);
}

__device__ __forceinline__ bool ls_beats(Word kj, Word rj, Word ki, Word ri) { return kj > ki || (kj == ki && rj < ri); }

// acc[k] += x_jk * v, x_jk = +1 where bit k of wj is set
__device__ __forceinline__ void ls_accumulate(Word wj, double v, double (&acc)[kRoundB]) {
    const unsigned lo = (unsigned)wj, hi = (unsigned)(wj >> 32);
#pragma unroll
    for (int k = 0; k < 32; k++) {
        acc[k] += (lo & (1u << k)) ? v : -v;
        acc[32 + k] += (hi & (1u << k)) ? v : -v;
    }
}

// bit k set iff x_ik * h_ik > 0 (strictly), restricted to the candidates of the batch
__device__ __forceinline__ Word ls_want_word(Word wi, const double (&h)[kRoundB], Word mask) {
    Word w = 0ull;
#pragma unroll
    for (int k = 0; k < kRoundB; k++) w |= (Word)(((wi >> k) & 1ull) ? h[k] > 0.0 : h[k] < 0.0) << k;
    return w & mask;
}

// want pass, rows with at most kLsLong nonzeros: one thread per dirty owned row, 64 register sums in pattern order
__global__ void __launch_bounds__(kLsTPB) k_ls_want(i64 row_lo, i64 row_hi, const int *__restrict__ ptr, const int *__restrict__ idx,
                                                   const double *__restrict__ val, const Word *__restrict__ words, Word mask,
                                                   unsigned char *__restrict__ dirty, Word *__restrict__ want) {
    for (i64 i = row_lo + blockIdx.x * (i64)blockDim.x + threadIdx.x; i < row_hi; i += (i64)gridDim.x * blockDim.x) {
        if (!dirty[i]) continue;
        const int a = ptr[i], b = ptr[i + 1];
        if (b - a > kLsLong) continue;
        dirty[i] = 0;
        double acc[kRoundB];
#pragma unroll
        for (int k = 0; k < kRoundB; k++) acc[k] = 0.0;
        for (int e = a; e < b; e++) {
            const int j = idx[e];
            const double v = val[e];
            if (j == i || v == 0.0) continue;
            ls_accumulate(words[j], v, acc);
        }
        want[i] = ls_want_word(words[i], acc, mask);
    }
}

// want pass, long rows: one CTA per segment of a dirty owned row; part[s][k] = the segment's sums (fixed-order CTA sum)
__global__ void __launch_bounds__(kLsTPB) k_ls_want_seg(i64 s_lo, i64 s_hi, const int *__restrict__ seg_row, const int *__restrict__ seg_start,
                                                       const int *__restrict__ ptr, const int *__restrict__ idx,
                                                       const double *__restrict__ val, const Word *__restrict__ words,
                                                       const unsigned char *__restrict__ dirty, double *__restrict__ part) {
    for (i64 s = s_lo + blockIdx.x; s < s_hi; s += gridDim.x) {
        const int i = seg_row[s];
        if (!dirty[i]) continue;   // the same for the whole CTA
        const int e0 = seg_start[s], e1 = min(e0 + kLsSeg, ptr[i + 1]);
        double acc[kRoundB];
#pragma unroll
        for (int k = 0; k < kRoundB; k++) acc[k] = 0.0;
        for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            const int j = idx[e];
            const double v = val[e];
            if (j == i || v == 0.0) continue;
            ls_accumulate(words[j], v, acc);
        }
        block_sum<kRoundB>(acc);
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < kRoundB; k++) part[(size_t)s * kRoundB + k] = acc[k];
        }
    }
}

// want pass, long rows: the segment sums of every dirty owned long row added in segment order
__global__ void k_ls_want_combine(i64 l_lo, i64 l_hi, const int *__restrict__ long_rows, const int *__restrict__ long_sptr,
                                  const double *__restrict__ part, const Word *__restrict__ words, Word mask,
                                  unsigned char *__restrict__ dirty, Word *__restrict__ want) {
    for (i64 L = l_lo + blockIdx.x * (i64)blockDim.x + threadIdx.x; L < l_hi; L += (i64)gridDim.x * blockDim.x) {
        const int i = long_rows[L];
        if (!dirty[i]) continue;
        dirty[i] = 0;
        double acc[kRoundB];
#pragma unroll
        for (int k = 0; k < kRoundB; k++) acc[k] = 0.0;
        for (int s = long_sptr[L]; s < long_sptr[L + 1]; s++) {
#pragma unroll
            for (int k = 0; k < kRoundB; k++) acc[k] += part[(size_t)s * kRoundB + k];
        }
        want[i] = ls_want_word(words[i], acc, mask);
    }
}

// flip pass: flip_i = want_i & ~OR{want_j : j a neighbour that beats i} over the owned rows (long rows: want_i here, their
// blocked bits are cleared by k_ls_flip_seg), and cnt[k] = number of owned rows with bit k of want set
__global__ void __launch_bounds__(kLsTPB) k_ls_flip(i64 row_lo, i64 nrows, const int *__restrict__ ptr, const int *__restrict__ idx,
                                                   const double *__restrict__ val, const int *__restrict__ iperm, Word salt,
                                                   const Word *__restrict__ want, Word *__restrict__ flip, int nb,
                                                   double *partials, unsigned *ticket, double *cnt_out) {
    const int lane = threadIdx.x & 31;
    unsigned cnt[2] = {0u, 0u};
    for (i64 base = (i64)blockIdx.x * blockDim.x; base < nrows; base += (i64)gridDim.x * blockDim.x) {
        const bool valid = base + threadIdx.x < nrows;
        const i64 i = row_lo + base + threadIdx.x;
        const Word wi = valid ? want[i] : 0ull;
        if (__any_sync(0xffffffffu, wi != 0ull)) ballot_counts(wi, lane, cnt);
        if (!valid) continue;
        Word m = wi;
        const int a = ptr[i], b = ptr[i + 1];
        if (m != 0ull && b - a <= kLsLong) {
            Word ri, rj;
            const Word ki = ls_key(iperm, i, salt, ri);
            for (int e = a; e < b && m != 0ull; e++) {
                const int j = idx[e];
                const Word wj = want[j] & m;
                if (wj == 0ull || j == i || val[e] == 0.0) continue;
                const Word kj = ls_key(iperm, j, salt, rj);
                if (ls_beats(kj, rj, ki, ri)) m &= ~wj;
            }
        }
        flip[i] = m;
    }
    double v[kRoundB];
    counts_to_values(cnt, lane, v);
    grid_sum_finalize<kRoundB>(v, partials, ticket, [&](double (&s)[kRoundB]) {
#pragma unroll
        for (int k = 0; k < kRoundB; k++) if (k < nb) cnt_out[k] = s[k];
    });
}

// flip pass, long rows: one CTA per segment of an owned long row that wants to flip; clears the bits a beating neighbour
// of the segment also wants (atomic AND: the result does not depend on the order)
__global__ void __launch_bounds__(kLsTPB) k_ls_flip_seg(i64 s_lo, i64 s_hi, const int *__restrict__ seg_row, const int *__restrict__ seg_start,
                                                       const int *__restrict__ ptr, const int *__restrict__ idx,
                                                       const double *__restrict__ val, const int *__restrict__ iperm, Word salt,
                                                       const Word *__restrict__ want, Word *__restrict__ flip) {
    for (i64 s = s_lo + blockIdx.x; s < s_hi; s += gridDim.x) {
        const int i = seg_row[s];
        const Word wi = want[i];
        if (wi == 0ull) continue;
        Word ri, rj, blocked = 0ull;
        const Word ki = ls_key(iperm, i, salt, ri);
        const int e0 = seg_start[s], e1 = min(e0 + kLsSeg, ptr[i + 1]);
        for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            const int j = idx[e];
            const Word wj = want[j] & wi;
            if (wj == 0ull || j == i || val[e] == 0.0) continue;
            const Word kj = ls_key(iperm, j, salt, rj);
            if (ls_beats(kj, rj, ki, ri)) blocked |= wj;
        }
        if (blocked) atomicAnd(&flip[i], ~blocked);
    }
}

// apply pass, every row (the words are replicated): word_i ^= flip_i; a flipped row marks itself and, when it has at most
// kLsLong nonzeros, its neighbours dirty.  flips[k] += the number of owned rows with bit k of flip set.
__global__ void __launch_bounds__(kLsTPB) k_ls_apply(i64 n, i64 row_lo, i64 row_hi, const int *__restrict__ ptr,
                                                    const int *__restrict__ idx, const double *__restrict__ val,
                                                    const Word *__restrict__ flip, Word *__restrict__ words,
                                                    unsigned char *__restrict__ dirty, int nb, double *partials, unsigned *ticket,
                                                    double *flips_acc) {
    const int lane = threadIdx.x & 31;
    unsigned cnt[2] = {0u, 0u};
    for (i64 base = (i64)blockIdx.x * blockDim.x; base < n; base += (i64)gridDim.x * blockDim.x) {
        const i64 i = base + threadIdx.x;
        const Word f = i < n ? flip[i] : 0ull;
        const Word fo = (i >= row_lo && i < row_hi) ? f : 0ull;
        if (__any_sync(0xffffffffu, fo != 0ull)) ballot_counts(fo, lane, cnt);
        if (f == 0ull) continue;
        words[i] ^= f;
        dirty[i] = 1;
        const int a = ptr[i], b = ptr[i + 1];
        if (b - a > kLsLong) continue;
        for (int e = a; e < b; e++) {
            const int j = idx[e];
            if (j != i && val[e] != 0.0) dirty[j] = 1;
        }
    }
    double v[kRoundB];
    counts_to_values(cnt, lane, v);
    grid_sum_finalize<kRoundB>(v, partials, ticket, [&](double (&s)[kRoundB]) {
#pragma unroll
        for (int k = 0; k < kRoundB; k++) if (k < nb) flips_acc[k] += s[k];
    });
}

// apply pass, long rows: one CTA per segment of a flipped row marks the segment's neighbours dirty
__global__ void __launch_bounds__(kLsTPB) k_ls_apply_seg(i64 nseg, const int *__restrict__ seg_row, const int *__restrict__ seg_start,
                                                        const int *__restrict__ ptr, const int *__restrict__ idx,
                                                        const double *__restrict__ val, const Word *__restrict__ flip,
                                                        unsigned char *__restrict__ dirty) {
    for (i64 s = blockIdx.x; s < nseg; s += gridDim.x) {
        const int i = seg_row[s];
        if (flip[i] == 0ull) continue;
        const int e0 = seg_start[s], e1 = min(e0 + kLsSeg, ptr[i + 1]);
        for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            const int j = idx[e];
            if (j != i && val[e] != 0.0) dirty[j] = 1;
        }
    }
}

// cnt[k] = number of owned rows with bit k of the word set (sum(x_k) after the search)
__global__ void __launch_bounds__(kLsTPB) k_ls_count(i64 row_lo, i64 nrows, const Word *__restrict__ words, int nb, double *partials,
                                                    unsigned *ticket, double *cnt_out) {
    const int lane = threadIdx.x & 31;
    unsigned cnt[2] = {0u, 0u};
    for (i64 base = (i64)blockIdx.x * blockDim.x; base < nrows; base += (i64)gridDim.x * blockDim.x) {
        const bool valid = base + threadIdx.x < nrows;
        ballot_counts(valid ? words[row_lo + base + threadIdx.x] : 0ull, lane, cnt);
    }
    double v[kRoundB];
    counts_to_values(cnt, lane, v);
    grid_sum_finalize<kRoundB>(v, partials, ticket, [&](double (&s)[kRoundB]) {
#pragma unroll
        for (int k = 0; k < kRoundB; k++) if (k < nb) cnt_out[k] = s[k];
    });
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

int32_t eval_pass(sdplrp_handle *h, int nb, double *sums_out) {
    RoundingState &s = h->rnd;
    if (s.nchunks > 0) {
        k_round_eval<<<grid_for(s.nchunks, kEvalTPB, 2 * kRedBlocks), kEvalTPB, 0, h->stream>>>(
            s.e_lo, s.e_hi, s.nchunks, h->full_ptr, h->full_idx, h->Cfull, s.chunk_row, s.words, nb, h->partials, h->ticket, sums_out);
        KLAUNCH(h);
    } else {
        CUDA_TRY(h, cudaMemsetAsync(sums_out, 0, (size_t)nb * sizeof(double), h->stream));
    }
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

template <typename T>
int32_t upload(sdplrp_handle *h, T **dst, const std::vector<T> &src) {
    SDP_CHECK(dev_alloc(h, dst, (i64)src.size()));
    if (!src.empty()) CUDA_TRY(h, cudaMemcpyAsync(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    return SDPLRP_OK;
}

// local-search buffers (first use after preprocessing): want / flip / best words and dirty flags (n each), and the segments
// of the rows of the full pattern with more than kLsLong nonzeros (all rows: the apply pass covers every row on every rank)
int32_t ensure_search_buffers(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    if (s.want) return SDPLRP_OK;
    const i64 n = h->n;
    std::vector<int> ptr((size_t)n + 1), long_rows, long_sptr(1, 0), seg_row, seg_start;
    CUDA_TRY(h, cudaMemcpyAsync(ptr.data(), h->full_ptr, ptr.size() * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (i64 i = 0; i < n; i++) {
        const int a = ptr[(size_t)i], b = ptr[(size_t)i + 1];
        if (b - a <= kLsLong) continue;
        long_rows.push_back((int)i);
        for (int e = a; e < b; e += kLsSeg) { seg_row.push_back((int)i); seg_start.push_back(e); }
        long_sptr.push_back((int)seg_row.size());
    }
    s.n_seg = (i64)seg_row.size();
    s.l_lo = std::lower_bound(long_rows.begin(), long_rows.end(), (int)h->row_lo) - long_rows.begin();
    s.l_hi = std::lower_bound(long_rows.begin(), long_rows.end(), (int)h->row_hi) - long_rows.begin();
    s.s_lo = long_sptr[(size_t)s.l_lo];
    s.s_hi = long_sptr[(size_t)s.l_hi];
    SDP_CHECK(upload(h, &s.long_rows, long_rows));
    SDP_CHECK(upload(h, &s.long_sptr, long_sptr));
    SDP_CHECK(upload(h, &s.seg_row, seg_row));
    SDP_CHECK(upload(h, &s.seg_start, seg_start));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    SDP_CHECK(dev_alloc(h, &s.seg_part, s.n_seg * kRoundB));
    SDP_CHECK(dev_alloc(h, &s.flip, n));
    SDP_CHECK(dev_alloc(h, &s.best_words, n));
    SDP_CHECK(dev_alloc(h, &s.dirty, n));
    SDP_CHECK(dev_alloc(h, &s.want, n));
    return SDPLRP_OK;
}

// one-flip descent of the batch's nb candidates on the words (complete on every rank).  wcnt: 64 doubles of scratch;
// flips_acc[k] += the flips of candidate k on the owned rows; rounds[k] = the last round that flipped candidate k, 0 if none,
// -1 when it still wanted to flip after max_rounds rounds.  *applied: some round flipped something.
int32_t local_search(sdplrp_handle *h, int nb, i64 max_rounds, double *wcnt, double *flips_acc, int64_t *rounds, bool *applied) {
    RoundingState &s = h->rnd;
    const i64 n = h->n, nrows = h->row_hi - h->row_lo;
    const Word mask = nb == kRoundB ? ~0ull : (1ull << nb) - 1ull;
    const int *iperm = h->relabeled ? h->iperm : nullptr;
    std::vector<double> wc((size_t)nb);
    std::fill(rounds, rounds + nb, (int64_t)0);
    *applied = false;
    CUDA_TRY(h, cudaMemsetAsync(s.dirty, 1, (size_t)n, h->stream));
    for (i64 t = 0;; t++) {
        const Word salt = mix64(0xD1B54A32D192ED03ull * (Word)(t + 1));
        if (nrows > 0) {
            k_ls_want<<<grid_for(nrows, kLsTPB, 8 * kNumSM), kLsTPB, 0, h->stream>>>(h->row_lo, h->row_hi, h->full_ptr, h->full_idx,
                                                                                       h->Cfull, s.words, mask, s.dirty, s.want);
            KLAUNCH(h);
        }
        if (s.s_hi > s.s_lo) {
            k_ls_want_seg<<<grid_for(s.s_hi - s.s_lo, 1, 8 * kNumSM), kLsTPB, 0, h->stream>>>(
                s.s_lo, s.s_hi, s.seg_row, s.seg_start, h->full_ptr, h->full_idx, h->Cfull, s.words, s.dirty, s.seg_part);
            KLAUNCH(h);
            k_ls_want_combine<<<grid_for(s.l_hi - s.l_lo, 128, 4 * kNumSM), 128, 0, h->stream>>>(
                s.l_lo, s.l_hi, s.long_rows, s.long_sptr, s.seg_part, s.words, mask, s.dirty, s.want);
            KLAUNCH(h);
        }
        SDP_CHECK(comm_gather_rowbytes(h, s.want, sizeof(Word)));
        k_ls_flip<<<grid_for(std::max<i64>(nrows, 1), kLsTPB, 2 * kRedBlocks), kLsTPB, 0, h->stream>>>(
            h->row_lo, nrows, h->full_ptr, h->full_idx, h->Cfull, iperm, salt, s.want, s.flip, nb, h->partials, h->ticket, wcnt);
        KLAUNCH(h);
        if (s.s_hi > s.s_lo) {
            k_ls_flip_seg<<<grid_for(s.s_hi - s.s_lo, 1, 8 * kNumSM), kLsTPB, 0, h->stream>>>(
                s.s_lo, s.s_hi, s.seg_row, s.seg_start, h->full_ptr, h->full_idx, h->Cfull, iperm, salt, s.want, s.flip);
            KLAUNCH(h);
        }
        CUDA_TRY(h, cudaGetLastError());
        SDP_CHECK(comm_reduce_ptr(h, wcnt, nb));
        CUDA_TRY(h, cudaMemcpyAsync(wc.data(), wcnt, (size_t)nb * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        if (std::none_of(wc.begin(), wc.end(), [](double c) { return c > 0.0; })) break;
        if (t == max_rounds) {
            for (int k = 0; k < nb; k++) if (wc[(size_t)k] > 0.0) rounds[k] = -1;
            break;
        }
        SDP_CHECK(comm_gather_rowbytes(h, s.flip, sizeof(Word)));
        k_ls_apply<<<grid_for(n, kLsTPB, 2 * kRedBlocks), kLsTPB, 0, h->stream>>>(n, h->row_lo, h->row_hi, h->full_ptr, h->full_idx, h->Cfull,
                                                                                   s.flip, s.words, s.dirty, nb, h->partials, h->ticket,
                                                                                   flips_acc);
        KLAUNCH(h);
        if (s.n_seg > 0) {
            k_ls_apply_seg<<<grid_for(s.n_seg, 1, 8 * kNumSM), kLsTPB, 0, h->stream>>>(s.n_seg, s.seg_row, s.seg_start, h->full_ptr,
                                                                                         h->full_idx, h->Cfull, s.flip, s.dirty);
            KLAUNCH(h);
        }
        CUDA_TRY(h, cudaGetLastError());
        for (int k = 0; k < nb; k++) if (wc[(size_t)k] > 0.0) rounds[k] = t + 1;
        *applied = true;
    }
    return SDPLRP_OK;
}

// per batch of 64 candidates, a block of sums: set bits, final eval sums, first eval sums (before the search), flips
constexpr int kSumBlock = 4 * kRoundB;

// K candidates in batches of 64: sign pass, all-gather of the words, evaluation pass and, when `search`, the one-flip
// descent and a second evaluation pass.  sdplrp_round_hyperplane is the case without search.
int32_t round_batches(sdplrp_handle *h, const char *name, int64_t K, const double *G, uint64_t seed, bool search, int64_t max_rounds,
                      double *G_out, double *obj_round, double *obj, double *sum, int64_t *flips, int64_t *rounds, int64_t *best,
                      double *best_x) {
    if (!h->preprocessed) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_preprocess first");
    if (h->r <= 0) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_set_rank first");
    if (K < 1 || !obj || !best) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": K >= 1 and the obj / best outputs are required");
    if (max_rounds < 0) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": max_rounds >= 0 is required");
    for (const LowRank &L : h->lr)
        if (L.gid == h->m) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": the objective has a low-rank part");
    if (h->obj_mat < 0) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": needs a sparse objective");
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
    if (h->world > 1) {   // SPMD: every rank must round with the same K, the same hyperplanes and the same search
        unsigned long long cs = mix64((unsigned long long)K);
        if (search) cs = mix64(cs ^ (unsigned long long)(max_rounds + 1));
        const unsigned long long *bits = reinterpret_cast<const unsigned long long *>(G);
        for (i64 e = 0; e < K * r; e++) cs = mix64(cs ^ bits[e]);
        SDP_CHECK(comm_check_same(h, cs, "hyperplanes (K, seed, G) or max_rounds"));
    }

    RoundingState &s = h->rnd;
    SDP_CHECK(ensure_problem_buffers(h));
    if (search) SDP_CHECK(ensure_search_buffers(h));
    const i64 nbatch = (K + kRoundB - 1) / kRoundB;
    const i64 csum_at = nbatch * kSumBlock, sums_len = csum_at + 1 + kRoundB;   // + sum of C, + want counts of a round
    SDP_CHECK(ensure(h, &s.G, &s.G_len, K * r));
    SDP_CHECK(ensure(h, &s.sums, &s.sums_len, sums_len));
    CUDA_TRY(h, cudaMemcpyAsync(s.G, G, (size_t)(K * r) * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(s.sums, 0, (size_t)sums_len * sizeof(double), h->stream));
    double *csum = s.sums + csum_at, *wcnt = csum + 1;
    k_round_csum<<<kRedBlocks, 256, 0, h->stream>>>(h->nnzF, h->Cfull, h->partials, h->ticket, csum);   // replicated: same bits everywhere
    KLAUNCH(h);
    double sumC = 0.0;
    if (search) {
        CUDA_TRY(h, cudaMemcpyAsync(&sumC, csum, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    std::vector<double> blk_h(kSumBlock);
    std::vector<int64_t> rounds_h(search ? (size_t)K : 0);
    i64 kb = -1;
    double best_obj = 0.0;
    for (i64 bt = 0; bt < nbatch; bt++) {
        const int nb = (int)std::min<i64>(kRoundB, K - bt * kRoundB);
        const double *dG = s.G + (size_t)(bt * kRoundB) * r;
        double *blk = s.sums + bt * kSumBlock, *cnt = blk, *esum = blk + kRoundB, *esum0 = blk + 2 * kRoundB, *fl = blk + 3 * kRoundB;
        SDP_CHECK(sign_pass(h, dG, nb, cnt));
        SDP_CHECK(comm_gather_rowbytes(h, s.words, sizeof(Word)));
        if (!search) {
            SDP_CHECK(eval_pass(h, nb, esum));
            continue;
        }
        SDP_CHECK(eval_pass(h, nb, esum0));
        bool applied = false;
        SDP_CHECK(local_search(h, nb, max_rounds, wcnt, fl, rounds_h.data() + bt * kRoundB, &applied));
        if (applied) {
            SDP_CHECK(eval_pass(h, nb, esum));
            k_ls_count<<<grid_for(std::max<i64>(h->row_hi - h->row_lo, 1), kLsTPB, 2 * kRedBlocks), kLsTPB, 0, h->stream>>>(
                h->row_lo, h->row_hi - h->row_lo, s.words, nb, h->partials, h->ticket, cnt);
            KLAUNCH(h);
            CUDA_TRY(h, cudaGetLastError());
        } else {
            CUDA_TRY(h, cudaMemcpyAsync(esum, esum0, (size_t)nb * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        }
        // the best candidate so far needs this batch's final words: keep them before the next batch overwrites them
        SDP_CHECK(comm_reduce_ptr(h, blk, kSumBlock));
        CUDA_TRY(h, cudaMemcpyAsync(blk_h.data(), blk, kSumBlock * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        bool improved = false;
        for (int k = 0; k < nb; k++) {
            const double o = sumC - 2.0 * blk_h[(size_t)(kRoundB + k)];
            if (kb < 0 || o < best_obj) { kb = bt * kRoundB + k; best_obj = o; improved = true; }
        }
        if (improved && best_x)
            CUDA_TRY(h, cudaMemcpyAsync(s.best_words, s.words, (size_t)n * sizeof(Word), cudaMemcpyDeviceToDevice, h->stream));
    }
    if (!search) SDP_CHECK(comm_reduce_ptr(h, s.sums, (int)csum_at));
    std::vector<double> hs((size_t)(csum_at + 1));
    CUDA_TRY(h, cudaMemcpyAsync(hs.data(), s.sums, hs.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));

    sumC = hs[(size_t)csum_at];
    kb = 0;
    for (i64 k = 0; k < K; k++) {
        const double *blk = hs.data() + (k / kRoundB) * kSumBlock;
        const i64 kk = k % kRoundB;
        obj[k] = sumC - 2.0 * blk[kRoundB + kk];
        if (obj_round) obj_round[k] = search ? sumC - 2.0 * blk[2 * kRoundB + kk] : obj[k];
        if (sum) sum[k] = 2.0 * blk[kk] - (double)n;
        if (flips) flips[k] = (int64_t)blk[3 * kRoundB + kk];
        if (rounds) rounds[k] = search ? rounds_h[(size_t)k] : 0;
        if (obj[k] < obj[kb]) kb = k;
    }
    *best = kb + 1;
    if (G_out) std::copy(G, G + (size_t)(K * r), G_out);
    if (best_x) {
        const i64 bt = kb / kRoundB;
        const Word *bw = s.words;
        if (search) {
            bw = s.best_words;
        } else if (bt != nbatch - 1) {   // the words of that batch were overwritten: the same kernel on the same data gives the same bits
            const int nb = (int)std::min<i64>(kRoundB, K - bt * kRoundB);
            SDP_CHECK(sign_pass(h, s.G + (size_t)(bt * kRoundB) * r, nb, s.sums + bt * kSumBlock));
            SDP_CHECK(comm_gather_rowbytes(h, s.words, sizeof(Word)));
        }
        k_round_expand<<<grid_for(n, 256, kRedBlocks * 4), 256, 0, h->stream>>>(n, bw, (int)(kb - bt * kRoundB), s.x);
        KLAUNCH(h);
        CUDA_TRY(h, cudaGetLastError());
        SDP_CHECK(perm_download(h, s.x, best_x, 1, true));
    }
    return SDPLRP_OK;
}
}  // namespace

void round_free(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    if (s.words) { cudaFree(s.words); s.words = nullptr; }
    dev_free(&s.x); dev_free(&s.chunk_row); dev_free(&s.G); dev_free(&s.sums);
    dev_free(&s.want); dev_free(&s.flip); dev_free(&s.best_words); dev_free(&s.dirty);
    dev_free(&s.long_rows); dev_free(&s.long_sptr); dev_free(&s.seg_row); dev_free(&s.seg_start); dev_free(&s.seg_part);
    s.G_len = s.sums_len = 0;
    s.e_lo = s.e_hi = s.nchunks = 0;
    s.n_seg = s.l_lo = s.l_hi = s.s_lo = s.s_hi = 0;
}

extern "C" int32_t sdplrp_round_hyperplane(sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, double *G_out, double *obj,
                                           double *sum, int64_t *best, double *best_x) {
    if (!h) return SDPLRP_ERR_ARG;
    return round_batches(h, "round_hyperplane", K, G, seed, false, 0, G_out, nullptr, obj, sum, nullptr, nullptr, best, best_x);
}

extern "C" int32_t sdplrp_round_local_search(sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, int64_t max_rounds,
                                             double *G_out, double *obj_round, double *obj, double *sum, int64_t *flips,
                                             int64_t *rounds, int64_t *best, double *best_x) {
    if (!h) return SDPLRP_ERR_ARG;
    return round_batches(h, "round_local_search", K, G, seed, max_rounds > 0 || rounds != nullptr, max_rounds, G_out, obj_round, obj,
                         sum, flips, rounds, best, best_x);
}
