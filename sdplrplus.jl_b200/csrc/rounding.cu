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
//   want pass   k_nbr_short / k_nbr_seg / k_nbr_combine<LsWant>: for every owned row flagged dirty,
//               h_ik = sum_{j != i, C_ij != 0} C_ij x_jk for the 64 candidates, and bit k of want_i = (x_ik h_ik > 0).
//   flip pass   k_ls_flip (+ k_ls_flip_seg): flip_i = want_i & ~OR{want_j : j a neighbour with a higher priority}, and the
//               per-candidate counts of wanting vertices.  The flipped vertices of a candidate are pairwise non-adjacent,
//               so their gains add up and the objective falls by 4 sum |h_ik| every round.
//   apply pass  k_ls_apply (+ k_ls_apply_seg): word_i ^= flip_i on every row, per-candidate flip counts over the owned
//               rows, and a flipped row marks itself and its neighbours dirty (identical byte stores).
// Rows with more than kLsLong nonzeros are cut into segments of kLsSeg nonzeros, one CTA each; the want and delta sums of a
// long row are combined over its segments in a fixed order.
//
// Sweep rounding (sdplrp_round_sweep) goes in batches of kSweepB = 16 candidates, one 128-byte row of projections per vertex:
// projection pass (k_round_sign<16, true>) -> per candidate a stable radix sort of (key, input id) -> delta pass
// (k_nbr_*<SwDelta>, the move deltas along each order) -> three-phase tile scan and selection (k_sw_tile_sums, k_sw_tile_scan, k_sw_scan,
// k_sw_select) -> words of the chosen prefixes (k_sw_words) -> evaluation pass.  DESIGN.md §3f.
// Nothing outside the rounding buffers (h->rnd) and the reduction scratch is written.
#include <limits.h>
#include <math.h>
#include <string.h>
#include <algorithm>
#include <cmath>
#include <cub/cub.cuh>
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
constexpr int kSweepB = 16;        // sweep rounding: candidates per batch (a vertex's projections are one 128-byte row)
constexpr int kSwTPB = 256;        // sweep scan: threads per tile
constexpr int kSwItems = 16;       // consecutive sweep positions per thread
constexpr int kSwTile = kSwTPB * kSwItems;
constexpr int kSwSel = 5;          // per candidate: f(t), t (-1: none feasible), W(S_t), boundary projection, boundary input id
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

// the ballot counts of every thread summed over the grid (fixed order) into out[k] for k < nb, stored or, when `add`, added
__device__ __forceinline__ void counts_finalize(const unsigned (&cnt)[2], int lane, int nb, double *partials, unsigned *ticket,
                                                double *out, bool add) {
    double v[kRoundB];
#pragma unroll
    for (int k = 0; k < kRoundB; k++) v[k] = lane == (k & 31) ? (double)cnt[k >> 5] : 0.0;
    grid_sum_finalize<kRoundB>(v, partials, ticket, [&](double (&s)[kRoundB]) {
#pragma unroll
        for (int k = 0; k < kRoundB; k++) if (k < nb) out[k] = add ? out[k] + s[k] : s[k];
    });
}

// words[i] bit k = (<R_i, g_k> >= 0) for the owned rows; cnt[k] = number of set bits over them (k < 64).
// PROJ (sweep rounding, NB = kSweepB): proj[i * NB + k] = <R_i, g_k> (-0.0 stored as +0.0, 0 for k >= nb) instead of the
// bits, no counts.  The per-candidate FMA chain is the same in both forms, so proj >= 0 is bit for bit the sign bit.
template <int NB, bool PROJ>
__global__ void __launch_bounds__(kSignTPB) k_round_sign(i64 row_lo, i64 nrows, int r, const double *__restrict__ R,
                                                          const double *__restrict__ G, int nb, Word *__restrict__ words,
                                                          double *__restrict__ proj, double *partials, unsigned *ticket,
                                                          double *cnt_out) {
    __shared__ double Gs[kSignCols][NB];
    const int lane = threadIdx.x & 31;
    unsigned cnt[2] = {0u, 0u};  // candidates lane and lane + 32 of this warp
    const bool single = r <= kSignCols;
    auto load_cols = [&](int c0) {
        const int nc = min(kSignCols, r - c0);
        for (int e = threadIdx.x; e < kSignCols * NB; e += blockDim.x) {
            const int c = e / NB, k = e - c * NB;
            Gs[c][k] = (c < nc && k < nb) ? G[(size_t)k * r + c0 + c] : 0.0;
        }
    };
    if (single) { load_cols(0); __syncthreads(); }
    for (i64 base = (i64)blockIdx.x * blockDim.x; base < nrows; base += (i64)gridDim.x * blockDim.x) {
        const i64 i = base + threadIdx.x;
        const bool valid = i < nrows;
        const double *Ri = R + (size_t)(row_lo + (valid ? i : 0)) * r;
        double acc[NB];
#pragma unroll
        for (int k = 0; k < NB; k++) acc[k] = 0.0;
        for (int c0 = 0; c0 < r; c0 += kSignCols) {
            if (!single) { __syncthreads(); load_cols(c0); __syncthreads(); }
            const int nc = min(kSignCols, r - c0);
            if (valid) {
                for (int c = 0; c < nc; c++) {
                    const double x = Ri[c0 + c];
#pragma unroll
                    for (int k = 0; k < NB; k++) acc[k] = fma(x, Gs[c][k], acc[k]);
                }
            }
        }
        if constexpr (PROJ) {
            if (valid) {
                double2 *Pi = reinterpret_cast<double2 *>(proj + (size_t)(row_lo + i) * NB);
#pragma unroll
                for (int k = 0; k < NB; k += 2) Pi[k / 2] = make_double2(acc[k] + 0.0, acc[k + 1] + 0.0);
            }
        } else {
            Word w = 0ull;
#pragma unroll
            for (int k = 0; k < NB; k++) w |= (Word)(acc[k] >= 0.0) << k;
            if (!valid) w = 0ull;
            else words[row_lo + i] = w;
            ballot_counts(w, lane, cnt);
        }
    }
    if constexpr (!PROJ) counts_finalize(cnt, lane, nb, partials, ticket, cnt_out, false);
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

// nonzero e (column j) of row i is a neighbour in the sums and dirty marks: off the diagonal, with a nonzero value (read only
// off the diagonal)
template <class I>
__device__ __forceinline__ bool is_neighbour(int j, I i, const double *__restrict__ val, int e) {
    return j != i && val[e] != 0.0;
}

// segment s of long row i: nonzeros [e0, e1), at most kLsSeg of them
__device__ __forceinline__ void seg_range(const int *__restrict__ seg_start, const int *__restrict__ ptr, i64 s, int i, int &e0,
                                          int &e1) {
    e0 = seg_start[s];
    e1 = min(e0 + kLsSeg, ptr[i + 1]);
}

// ---- neighbour sums: acc_i[k] = sum over the neighbours j of row i of a term of (j, C_ij), for the want and delta passes --
// Op supplies NB (sums per row), Row row(i) (per-row state), gather(j) (what the term reads of neighbour j),
// add(row, gather(j), C_ij, acc), finish(i, acc) (writes row i's output) and kSegMinCTAs (resident CTAs per SM the
// segment kernel is compiled for, 0: no bound).  With a gate (the local search's dirty flags), only the rows whose flag is
// set are summed, and the flag is cleared when the row's output is written.  Rows with at most kLsLong nonzeros: one
// thread per row, pattern order.  Long rows: one CTA per segment, thread-strided and block_sum into
// part[s][k], then the segments of each row added in segment order.

// want pass of the local search: h_ik = sum C_ij x_jk for the 64 candidates, on the dirty rows, and bit k of want_i =
// (x_ik h_ik > 0).  A row that is not dirty keeps its want word: it depends only on x_i and the x_j of its neighbours.
struct LsWant {
    static constexpr int NB = kRoundB;
    static constexpr int kSegMinCTAs = 0;
    struct Row {};
    const Word *words;
    Word mask;
    Word *want;
    __device__ Row row(i64) const { return {}; }
    __device__ Word gather(int j) const { return __ldg(words + j); }   // issued with idx / val, ahead of the neighbour test
    __device__ void add(const Row &, Word wj, double v, double (&acc)[NB]) const { ls_accumulate(wj, v, acc); }
    __device__ void finish(i64 i, const double (&acc)[NB]) const { want[i] = ls_want_word(__ldg(words + i), acc, mask); }
};

template <class Op>
__global__ void __launch_bounds__(kLsTPB) k_nbr_short(i64 row_lo, i64 row_hi, const int *__restrict__ ptr, const int *__restrict__ idx,
                                                     const double *__restrict__ val, const Op op, unsigned char *__restrict__ gate) {
    for (i64 i = row_lo + blockIdx.x * (i64)blockDim.x + threadIdx.x; i < row_hi; i += (i64)gridDim.x * blockDim.x) {
        if (gate && !gate[i]) continue;
        const int a = ptr[i], b = ptr[i + 1];
        if (b - a > kLsLong) continue;
        if (gate) gate[i] = 0;
        const typename Op::Row row = op.row(i);
        double acc[Op::NB];
#pragma unroll
        for (int k = 0; k < Op::NB; k++) acc[k] = 0.0;
        for (int e = a; e < b; e++) {
            const int j = idx[e];
            const double v = val[e];
            const auto x = op.gather(j);
            if (is_neighbour(j, i, val, e)) op.add(row, x, v, acc);
        }
        op.finish(i, acc);
    }
}

template <class Op>
__global__ void __launch_bounds__(kLsTPB, Op::kSegMinCTAs) k_nbr_seg(i64 s_lo, i64 s_hi, const int *__restrict__ seg_row,
                                                                     const int *__restrict__ seg_start,
                                                   const int *__restrict__ ptr, const int *__restrict__ idx,
                                                   const double *__restrict__ val, const Op op, const unsigned char *__restrict__ gate,
                                                   double *__restrict__ part) {
    for (i64 s = s_lo + blockIdx.x; s < s_hi; s += gridDim.x) {
        const int i = seg_row[s];
        if (gate && !gate[i]) continue;   // the same for the whole CTA
        int e0, e1;
        seg_range(seg_start, ptr, s, i, e0, e1);
        const typename Op::Row row = op.row(i);
        double acc[Op::NB];
#pragma unroll
        for (int k = 0; k < Op::NB; k++) acc[k] = 0.0;
        for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            const int j = idx[e];
            const double v = val[e];
            const auto x = op.gather(j);
            if (is_neighbour(j, i, val, e)) op.add(row, x, v, acc);
        }
        block_sum<Op::NB>(acc);
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < Op::NB; k++) part[(size_t)s * Op::NB + k] = acc[k];
        }
    }
}

template <class Op>
__global__ void k_nbr_combine(i64 l_lo, i64 l_hi, const int *__restrict__ long_rows, const int *__restrict__ long_sptr,
                              const double *__restrict__ part, const Op op, unsigned char *__restrict__ gate) {
    for (i64 L = l_lo + blockIdx.x * (i64)blockDim.x + threadIdx.x; L < l_hi; L += (i64)gridDim.x * blockDim.x) {
        const int i = long_rows[L];
        if (gate && !gate[i]) continue;
        if (gate) gate[i] = 0;
        double acc[Op::NB];
#pragma unroll
        for (int k = 0; k < Op::NB; k++) acc[k] = 0.0;
        for (int s = long_sptr[L]; s < long_sptr[L + 1]; s++) {
#pragma unroll
            for (int k = 0; k < Op::NB; k++) acc[k] += part[(size_t)s * Op::NB + k];
        }
        op.finish(i, acc);
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
                if (wj == 0ull || !is_neighbour(j, i, val, e)) continue;
                const Word kj = ls_key(iperm, j, salt, rj);
                if (ls_beats(kj, rj, ki, ri)) m &= ~wj;
            }
        }
        flip[i] = m;
    }
    counts_finalize(cnt, lane, nb, partials, ticket, cnt_out, false);
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
        int e0, e1;
        seg_range(seg_start, ptr, s, i, e0, e1);
        for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            const int j = idx[e];
            const Word wj = want[j] & wi;
            if (wj == 0ull || !is_neighbour(j, i, val, e)) continue;
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
            if (is_neighbour(j, i, val, e)) dirty[j] = 1;
        }
    }
    counts_finalize(cnt, lane, nb, partials, ticket, flips_acc, true);
}

// apply pass, long rows: one CTA per segment of a flipped row marks the segment's neighbours dirty
__global__ void __launch_bounds__(kLsTPB) k_ls_apply_seg(i64 nseg, const int *__restrict__ seg_row, const int *__restrict__ seg_start,
                                                        const int *__restrict__ ptr, const int *__restrict__ idx,
                                                        const double *__restrict__ val, const Word *__restrict__ flip,
                                                        unsigned char *__restrict__ dirty) {
    for (i64 s = blockIdx.x; s < nseg; s += gridDim.x) {
        const int i = seg_row[s];
        if (flip[i] == 0ull) continue;
        int e0, e1;
        seg_range(seg_start, ptr, s, i, e0, e1);
        for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            const int j = idx[e];
            if (is_neighbour(j, i, val, e)) dirty[j] = 1;
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
    counts_finalize(cnt, lane, nb, partials, ticket, cnt_out, false);
}

// ---- sweep rounding --------------------------------------------------------------------------------------------------
// Candidate k orders the vertices by (p_ik, input id) ascending; S_t = the first t of them.  Vertex j comes after v in that
// order iff (p_jk, ref_j) > (p_vk, ref_v); the input ids are read only where projections are equal.
__device__ __forceinline__ int sw_ref(const int *__restrict__ iperm, i64 i) { return iperm ? iperm[i] : (int)i; }

__device__ __forceinline__ void sw_load_row(const double *__restrict__ P, i64 i, double (&p)[kSweepB]) {
    const double2 *row = reinterpret_cast<const double2 *>(P + (size_t)i * kSweepB);
#pragma unroll
    for (int k = 0; k < kSweepB; k += 2) { const double2 t = __ldg(row + k / 2); p[k] = t.x; p[k + 1] = t.y; }
}

// acc[k] += C_vj when j comes after v in candidate k's order, -= C_vj when before (k < nb: mask = low nb bits)
__device__ __forceinline__ void sw_accumulate(const double *__restrict__ P, const int *__restrict__ iperm, int j, double v,
                                              const double (&pv)[kSweepB], int rv, unsigned mask, double (&acc)[kSweepB]) {
    double pj[kSweepB];
    sw_load_row(P, j, pj);
    unsigned gt = 0u, eq = 0u;
#pragma unroll
    for (int k = 0; k < kSweepB; k++) { gt |= (unsigned)(pj[k] > pv[k]) << k; eq |= (unsigned)(pj[k] == pv[k]) << k; }
    eq &= mask;
    if (eq && sw_ref(iperm, j) > rv) gt |= eq;
#pragma unroll
    for (int k = 0; k < kSweepB; k++) acc[k] += ((gt >> k) & 1u) ? v : -v;
}

// sort input of candidate k in input vertex order: keys[u] = order-preserving bits of p_{perm(u)k}, vals[u] = perm(u)
__global__ void k_sw_keys(i64 n, int k, const double *__restrict__ P, const int *__restrict__ perm, Word *__restrict__ keys,
                          int *__restrict__ vals) {
    for (i64 u = blockIdx.x * (i64)blockDim.x + threadIdx.x; u < n; u += (i64)gridDim.x * blockDim.x) {
        const int i = perm ? perm[u] : (int)u;
        const Word b = (Word)__double_as_longlong(P[(size_t)i * kSweepB + k]);
        keys[u] = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
        vals[u] = i;
    }
}

// delta pass of the sweep: delta[v][k] = -4 (sum_after C_vj - sum_before C_vj) along candidate k's order, on every row
struct SwDelta {
    static constexpr int NB = kSweepB;
    static constexpr int kSegMinCTAs = 5;   // at most 96 registers: the 128-byte row gathers of hub rows want the occupancy
    struct Row {
        double p[kSweepB];
        int ref;
    };
    const double *P;
    const int *iperm;
    unsigned mask;
    double *delta;
    __device__ Row row(i64 i) const {
        Row r;
        sw_load_row(P, i, r.p);
        r.ref = sw_ref(iperm, i);
        return r;
    }
    __device__ int gather(int j) const { return j; }   // the row of P is read in add, after the neighbour test
    __device__ void add(const Row &r, int j, double v, double (&acc)[NB]) const { sw_accumulate(P, iperm, j, v, r.p, r.ref, mask, acc); }
    __device__ void finish(i64 i, const double (&acc)[NB]) const {
        double2 *out = reinterpret_cast<double2 *>(delta + (size_t)i * kSweepB);
#pragma unroll
        for (int k = 0; k < kSweepB; k += 2) out[k / 2] = make_double2(-4.0 * acc[k], -4.0 * acc[k + 1]);
    }
};

// exclusive prefix of (a, b) over the threads of the CTA in thread order (shuffle scans: the same bits every run)
__device__ __forceinline__ void sw_block_exscan(double &a, double &b) {
    __shared__ double ws[2][32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    double ia = a, ib = b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += ta; ib += tb; }
    }
    double ea = __shfl_up_sync(0xffffffffu, ia, 1), eb = __shfl_up_sync(0xffffffffu, ib, 1);
    if (lane == 0) { ea = 0.0; eb = 0.0; }
    __syncthreads();   // ws reused across calls
    if (lane == 31) { ws[0][wid] = ia; ws[1][wid] = ib; }
    __syncthreads();
    if (wid == 0) {
        double xa = lane < nw ? ws[0][lane] : 0.0, xb = lane < nw ? ws[1][lane] : 0.0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double ta = __shfl_up_sync(0xffffffffu, xa, o), tb = __shfl_up_sync(0xffffffffu, xb, o);
            if (lane >= o) { xa += ta; xb += tb; }
        }
        double pa = __shfl_up_sync(0xffffffffu, xa, 1), pb = __shfl_up_sync(0xffffffffu, xb, 1);
        if (lane == 0) { pa = 0.0; pb = 0.0; }
        if (lane < nw) { ws[0][lane] = pa; ws[1][lane] = pb; }
    }
    __syncthreads();
    a = ws[0][wid] + ea;
    b = ws[1][wid] + eb;
}

// (f, t, W) minimum over the CTA: smallest f, ties to the smallest t (t = INT64_MAX: none).  Exact comparisons only, so the
// result does not depend on the order.  Valid in thread 0.
__device__ __forceinline__ bool sw_better(double f, long long t, double bf, long long bt) { return f < bf || (f == bf && t < bt); }

__device__ __forceinline__ void sw_block_argmin(double &f, long long &t, double &w) {
    __shared__ double sf[32], sw[32];
    __shared__ long long st[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double of = __shfl_xor_sync(0xffffffffu, f, o), ow = __shfl_xor_sync(0xffffffffu, w, o);
        const long long ot = __shfl_xor_sync(0xffffffffu, t, o);
        if (sw_better(of, ot, f, t)) { f = of; t = ot; w = ow; }
    }
    __syncthreads();
    if (lane == 0) { sf[wid] = f; st[wid] = t; sw[wid] = w; }
    __syncthreads();
    if (wid == 0) {
        f = lane < nw ? sf[lane] : INFINITY;
        t = lane < nw ? st[lane] : LLONG_MAX;
        w = lane < nw ? sw[lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double of = __shfl_xor_sync(0xffffffffu, f, o), ow = __shfl_xor_sync(0xffffffffu, w, o);
            const long long ot = __shfl_xor_sync(0xffffffffu, t, o);
            if (sw_better(of, ot, f, t)) { f = of; t = ot; w = ow; }
        }
    }
}

// scan phase 1, grid (tiles, candidates): tsum[k][tile] = the tile's sums of delta and w along candidate k's order
__global__ void __launch_bounds__(kSwTPB) k_sw_tile_sums(i64 n, i64 ntiles, const int *__restrict__ order, const double *__restrict__ delta,
                                                        const double *__restrict__ w, double *__restrict__ tsum_d,
                                                        double *__restrict__ tsum_w) {
    const int k = blockIdx.y;
    const int *ord = order + (size_t)k * n;
    const i64 base = (i64)blockIdx.x * kSwTile;
    double v[2] = {0.0, 0.0};
    for (int q = 0; q < kSwItems; q++) {
        const i64 s = base + q * kSwTPB + threadIdx.x;
        if (s < n) {
            const int u = ord[s];
            v[0] += delta[(size_t)u * kSweepB + k];
            v[1] += w ? w[u] : 1.0;
        }
    }
    block_sum<2>(v);
    if (threadIdx.x == 0) { tsum_d[(size_t)k * ntiles + blockIdx.x] = v[0]; tsum_w[(size_t)k * ntiles + blockIdx.x] = v[1]; }
}

// scan phase 2, one CTA per candidate: the tile sums replaced by their exclusive prefix, in tile order
__global__ void __launch_bounds__(kSwTPB) k_sw_tile_scan(i64 ntiles, double *__restrict__ tsum_d, double *__restrict__ tsum_w) {
    double *d = tsum_d + (size_t)blockIdx.x * ntiles, *w = tsum_w + (size_t)blockIdx.x * ntiles;
    __shared__ double carry[2];
    if (threadIdx.x == 0) { carry[0] = 0.0; carry[1] = 0.0; }
    __syncthreads();
    for (i64 t0 = 0; t0 < ntiles; t0 += kSwTPB) {
        const i64 t = t0 + threadIdx.x;
        const double a0 = t < ntiles ? d[t] : 0.0, b0 = t < ntiles ? w[t] : 0.0;
        double a = a0, b = b0;
        sw_block_exscan(a, b);
        const double ca = carry[0], cb = carry[1];
        if (t < ntiles) { d[t] = ca + a; w[t] = cb + b; }
        __syncthreads();
        if (threadIdx.x == kSwTPB - 1) { carry[0] = ca + (a + a0); carry[1] = cb + (b + b0); }
        __syncthreads();
    }
}

// scan phase 3, grid (tiles, candidates): the tile rescanned from its offset.  Position s adds delta / w of vertex
// order[s]: f(s + 1) = sum(C) + prefix, W(S_{s+1}) = prefix of w.  The feasible minimum of the tile (ties to the smallest t)
// goes to tbest; prof (candidate 0 only, may be NULL) receives f(0..n).
__global__ void __launch_bounds__(kSwTPB) k_sw_scan(i64 n, i64 ntiles, const int *__restrict__ order, const double *__restrict__ delta,
                                                   const double *__restrict__ w, const double *__restrict__ toff_d,
                                                   const double *__restrict__ toff_w, const double *__restrict__ csum, double wlo,
                                                   double whi, double *__restrict__ prof, double *__restrict__ tbest) {
    __shared__ int ids[kSwTile];
    const int k = blockIdx.y;
    const int *ord = order + (size_t)k * n;
    const i64 base = (i64)blockIdx.x * kSwTile;
    for (int q = 0; q < kSwItems; q++) {
        const i64 s = base + q * kSwTPB + threadIdx.x;
        ids[q * kSwTPB + threadIdx.x] = s < n ? ord[s] : -1;
    }
    __syncthreads();
    double dl[kSwItems], wl[kSwItems], a = 0.0, b = 0.0;
#pragma unroll
    for (int q = 0; q < kSwItems; q++) {
        const int u = ids[threadIdx.x * kSwItems + q];
        dl[q] = u >= 0 ? delta[(size_t)u * kSweepB + k] : 0.0;
        wl[q] = u >= 0 ? (w ? w[u] : 1.0) : 0.0;
        a += dl[q];
        b += wl[q];
    }
    sw_block_exscan(a, b);
    const size_t tk = (size_t)k * ntiles + blockIdx.x;
    double pd = toff_d[tk] + a, pw = toff_w[tk] + b;
    const double c = *csum;
    double bf = INFINITY, bw = 0.0;
    long long bt = LLONG_MAX;
    if (blockIdx.x == 0 && threadIdx.x == 0) {   // t = 0: S empty
        if (prof) prof[0] = c;
        if (wlo <= 0.0 && 0.0 <= whi) { bf = c; bt = 0; }
    }
#pragma unroll
    for (int q = 0; q < kSwItems; q++) {
        const i64 s = base + (i64)threadIdx.x * kSwItems + q;
        if (s < n) {
            pd += dl[q];
            pw += wl[q];
            const double f = c + pd;
            if (prof) prof[s + 1] = f;
            if (wlo <= pw && pw <= whi && f < bf) { bf = f; bt = s + 1; bw = pw; }
        }
    }
    sw_block_argmin(bf, bt, bw);
    if (threadIdx.x == 0) {
        double *o = tbest + tk * 3;
        o[0] = bf; o[1] = (double)bt; o[2] = bw;
    }
}

// selection, one CTA per candidate: the minimum over the tiles, and the boundary vertex b = order[t] whose (p, input id)
// starts the +1 side (t = n: none, every x = -1; no feasible t: every x = +1, the candidate is reported infeasible)
__global__ void __launch_bounds__(kSwTPB) k_sw_select(i64 n, i64 ntiles, const double *__restrict__ tbest, const int *__restrict__ order,
                                                     const double *__restrict__ P, const int *__restrict__ iperm,
                                                     double *__restrict__ sel) {
    const int k = blockIdx.x;
    double bf = INFINITY, bw = 0.0;
    long long bt = LLONG_MAX;
    for (i64 tile = threadIdx.x; tile < ntiles; tile += blockDim.x) {
        const double *o = tbest + ((size_t)k * ntiles + tile) * 3;
        const long long t = o[1] >= 9.0e18 ? LLONG_MAX : (long long)o[1];
        if (sw_better(o[0], t, bf, bt)) { bf = o[0]; bt = t; bw = o[2]; }
    }
    sw_block_argmin(bf, bt, bw);
    if (threadIdx.x == 0) {
        double *o = sel + (size_t)k * kSwSel;
        const bool none = bt == LLONG_MAX;
        o[0] = bf;
        o[1] = none ? -1.0 : (double)bt;
        o[2] = bw;
        if (none) { o[3] = -INFINITY; o[4] = -1.0; }
        else if (bt == n) { o[3] = INFINITY; o[4] = 0.0; }
        else { const int u = order[(size_t)k * n + bt]; o[3] = P[(size_t)u * kSweepB + k]; o[4] = (double)sw_ref(iperm, u); }
    }
}

// words of the owned rows: bit k set (x = +1) iff (p_ik, input id) >= the boundary of candidate k
__global__ void k_sw_words(i64 row_lo, i64 row_hi, const double *__restrict__ P, const int *__restrict__ iperm,
                           const double *__restrict__ sel, int nb, Word *__restrict__ words) {
    __shared__ double bp[kSweepB], bi[kSweepB];
    if (threadIdx.x < kSweepB) {
        bp[threadIdx.x] = threadIdx.x < nb ? sel[threadIdx.x * kSwSel + 3] : INFINITY;
        bi[threadIdx.x] = threadIdx.x < nb ? sel[threadIdx.x * kSwSel + 4] : 0.0;
    }
    __syncthreads();
    for (i64 i = row_lo + blockIdx.x * (i64)blockDim.x + threadIdx.x; i < row_hi; i += (i64)gridDim.x * blockDim.x) {
        double p[kSweepB];
        sw_load_row(P, i, p);
        const double ri = (double)sw_ref(iperm, i);
        Word w = 0ull;
#pragma unroll
        for (int k = 0; k < kSweepB; k++) w |= (Word)(p[k] > bp[k] || (p[k] == bp[k] && ri >= bi[k])) << k;
        words[i] = w;
    }
}

// out[s] = 1-based input id of the vertex at sweep position s
__global__ void k_sw_order_out(i64 n, const int *__restrict__ order, const int *__restrict__ iperm, int64_t *__restrict__ out) {
    for (i64 s = blockIdx.x * (i64)blockDim.x + threadIdx.x; s < n; s += (i64)gridDim.x * blockDim.x)
        out[s] = (int64_t)sw_ref(iperm, order[s]) + 1;
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
    k_round_sign<kRoundB, false><<<grid_for(std::max<i64>(nrows, 1), kSignTPB, 2 * kRedBlocks), kSignTPB, 0, h->stream>>>(
        h->row_lo, nrows, h->r, h->R, dG, nb, h->rnd.words, nullptr, h->partials, h->ticket, cnt_out);
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

// the segments of the rows of the full pattern with more than kLsLong nonzeros (all rows: the apply pass of the local search
// covers every row on every rank), and their partial sums (first use after preprocessing)
int32_t ensure_segments(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    if (s.seg_part) return SDPLRP_OK;
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
    return SDPLRP_OK;
}

// the neighbour sums of op over the owned rows (kernels above), gated by `gate` unless it is NULL; the long rows' segment
// sums go through seg_part
template <class Op>
int32_t neighbour_sums(sdplrp_handle *h, const Op &op, unsigned char *gate) {
    RoundingState &s = h->rnd;
    const i64 nrows = h->row_hi - h->row_lo;
    if (nrows > 0) {
        k_nbr_short<Op><<<grid_for(nrows, kLsTPB, 8 * kNumSM), kLsTPB, 0, h->stream>>>(h->row_lo, h->row_hi, h->full_ptr, h->full_idx,
                                                                                        h->Cfull, op, gate);
        KLAUNCH(h);
    }
    if (s.s_hi > s.s_lo) {
        k_nbr_seg<Op><<<grid_for(s.s_hi - s.s_lo, 1, 8 * kNumSM), kLsTPB, 0, h->stream>>>(
            s.s_lo, s.s_hi, s.seg_row, s.seg_start, h->full_ptr, h->full_idx, h->Cfull, op, gate, s.seg_part);
        KLAUNCH(h);
        k_nbr_combine<Op><<<grid_for(s.l_hi - s.l_lo, 128, 4 * kNumSM), 128, 0, h->stream>>>(s.l_lo, s.l_hi, s.long_rows, s.long_sptr,
                                                                                             s.seg_part, op, gate);
        KLAUNCH(h);
    }
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

// local-search buffers (first use after preprocessing): the segments, want / flip / best words and dirty flags (n each)
int32_t ensure_search_buffers(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    if (s.want) return SDPLRP_OK;
    const i64 n = h->n;
    SDP_CHECK(ensure_segments(h));
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
        SDP_CHECK(neighbour_sums(h, LsWant{s.words, mask, s.want}, s.dirty));
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

// the checks every rounding entry point makes before it touches the device
int32_t rounding_check(sdplrp_handle *h, const char *name, int64_t K, const void *obj, const void *best) {
    if (!h->preprocessed) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_preprocess first");
    if (h->r <= 0) return fail(h, SDPLRP_ERR_STATE, "call sdplrp_set_rank first");
    if (K < 1 || !obj || !best) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": K >= 1 and the obj / best outputs are required");
    return SDPLRP_OK;
}

int32_t objective_check(sdplrp_handle *h, const char *name) {
    for (const LowRank &L : h->lr)
        if (L.gid == h->m) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": the objective has a low-rank part");
    if (h->obj_mat < 0) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": needs a sparse objective");
    return SDPLRP_OK;
}

// hyperplanes on the host: the caller's G, or the counter-based normals (kept in Gh)
const double *hyperplanes(const sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, std::vector<double> &Gh) {
    if (G) return G;
    const int r = h->r;
    Gh.resize((size_t)K * r);
    for (i64 k = 0; k < K; k++)
        for (int c = 0; c < r; c++) Gh[(size_t)k * r + c] = hyperplane_normal(seed, k, c);
    return Gh.data();
}

Word double_bits(double x) {
    Word b;
    memcpy(&b, &x, sizeof b);
    return b;
}

// The device half of every rounding call, after its argument checks.  G becomes the hyperplanes (the caller's, or the
// seeded normals kept in Gh).  Several GPUs: every rank must round the same call, so a checksum of K ^ salt, the
// hyperplanes, `extra` and the bits of tail[0..ntail) is compared across ranks ("what" names them in the error).  Then the
// problem buffers, G on the device, sums_len zeroed sums and the sum of C at sums[csum_at] (replicated: same bits everywhere).
int32_t round_setup(sdplrp_handle *h, int64_t K, const double *&G, uint64_t seed, std::vector<double> &Gh, Word salt,
                    std::initializer_list<Word> extra, const double *tail, i64 ntail, const char *what, i64 sums_len, i64 csum_at) {
    CUDA_TRY(h, cudaSetDevice(h->device));
    const i64 len = K * h->r;
    G = hyperplanes(h, K, G, seed, Gh);
    if (h->world > 1) {
        Word cs = mix64((Word)K ^ salt);
        for (i64 e = 0; e < len; e++) cs = mix64(cs ^ double_bits(G[e]));
        for (Word x : extra) cs = mix64(cs ^ x);
        for (i64 e = 0; e < ntail; e++) cs = mix64(cs ^ double_bits(tail[e]));
        SDP_CHECK(comm_check_same(h, cs, what));
    }
    RoundingState &s = h->rnd;
    SDP_CHECK(ensure_problem_buffers(h));
    SDP_CHECK(ensure(h, &s.G, &s.G_len, len));
    SDP_CHECK(ensure(h, &s.sums, &s.sums_len, sums_len));
    CUDA_TRY(h, cudaMemcpyAsync(s.G, G, (size_t)len * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(s.sums, 0, (size_t)sums_len * sizeof(double), h->stream));
    k_round_csum<<<kRedBlocks, 256, 0, h->stream>>>(h->nnzF, h->Cfull, h->partials, h->ticket, s.sums + csum_at);
    KLAUNCH(h);
    return SDPLRP_OK;
}

// best_x (input order) = +1 / -1 from bit b of the words
int32_t download_signs(sdplrp_handle *h, const Word *words, int b, double *best_x) {
    k_round_expand<<<grid_for(h->n, 256, kRedBlocks * 4), 256, 0, h->stream>>>(h->n, words, b, h->rnd.x);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    return perm_download(h, h->rnd.x, best_x, 1, true);
}

// K candidates in batches of 64: sign pass, all-gather of the words, evaluation pass and, when `search`, the one-flip
// descent and a second evaluation pass.  sdplrp_round_hyperplane is the case without search.
int32_t round_batches(sdplrp_handle *h, const char *name, int64_t K, const double *G, uint64_t seed, bool search, int64_t max_rounds,
                      double *G_out, double *obj_round, double *obj, double *sum, int64_t *flips, int64_t *rounds, int64_t *best,
                      double *best_x) {
    SDP_CHECK(rounding_check(h, name, K, obj, best));
    if (max_rounds < 0) return fail(h, SDPLRP_ERR_ARG, std::string(name) + ": max_rounds >= 0 is required");
    SDP_CHECK(objective_check(h, name));
    const int r = h->r;
    const i64 n = h->n;
    const i64 nbatch = (K + kRoundB - 1) / kRoundB;
    const i64 csum_at = nbatch * kSumBlock, sums_len = csum_at + 1 + kRoundB;   // + sum of C, + want counts of a round
    std::vector<double> Gh;
    SDP_CHECK(round_setup(h, K, G, seed, Gh, 0, {search ? (Word)(max_rounds + 1) : 0}, nullptr, 0,
                          "hyperplanes (K, seed, G) or max_rounds", sums_len, csum_at));
    RoundingState &s = h->rnd;
    if (search) SDP_CHECK(ensure_search_buffers(h));
    double *csum = s.sums + csum_at, *wcnt = csum + 1;
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
        SDP_CHECK(download_signs(h, bw, (int)(kb - bt * kRoundB), best_x));
    }
    return SDPLRP_OK;
}

// sweep buffers (first use after preprocessing)
int32_t ensure_sweep_buffers(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    SDP_CHECK(ensure_segments(h));
    if (s.sw_P) return SDPLRP_OK;
    const i64 n = h->n;
    if (n > 0x7fffffffLL) return fail(h, SDPLRP_ERR_ARG, "round_sweep: more than 2^31 - 1 vertices");
    s.sw_ntiles = (n + kSwTile - 1) / kSwTile;
    SDP_CHECK(dev_alloc(h, &s.sw_P, n * kSweepB));
    SDP_CHECK(dev_alloc(h, &s.sw_delta, n * kSweepB));
    SDP_CHECK(dev_alloc(h, &s.sw_order, n * kSweepB));
    SDP_CHECK(dev_alloc(h, &s.sw_keys, 2 * n));
    SDP_CHECK(dev_alloc(h, &s.sw_vals, n));
    SDP_CHECK(dev_alloc(h, &s.sw_tiles, s.sw_ntiles * kSweepB * 5));
    size_t bytes = 0;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(nullptr, bytes, s.sw_keys, s.sw_keys + n, s.sw_vals, s.sw_order, (int)n, 0, 64,
                                                h->stream));
    SDP_CHECK(dev_alloc(h, &s.sw_cub, (i64)bytes));
    s.sw_cub_bytes = bytes;
    return SDPLRP_OK;
}

// one batch of nb <= 16 sweep candidates (hyperplanes dG): projection, sorts, delta pass, scan and selection (sel: nb x kSwSel),
// then, when `words`, the words of the chosen vectors and, when esum != NULL, the evaluation pass.  prof (nb = 1): f(0..n).
int32_t sweep_batch(sdplrp_handle *h, const double *dG, int nb, const double *w, double wlo, double whi, const double *csum,
                    double *sel, double *prof, bool words, double *esum) {
    RoundingState &s = h->rnd;
    const i64 n = h->n, nrows = h->row_hi - h->row_lo, nt = s.sw_ntiles;
    const int *iperm = h->relabeled ? h->iperm : nullptr, *perm = h->relabeled ? h->perm : nullptr;
    const unsigned mask = (1u << nb) - 1u;
    // 1. projections of the owned rows, all-gathered
    k_round_sign<kSweepB, true><<<grid_for(std::max<i64>(nrows, 1), kSignTPB, 2 * kRedBlocks), kSignTPB, 0, h->stream>>>(
        h->row_lo, nrows, h->r, h->R, dG, nb, nullptr, s.sw_P, nullptr, nullptr, nullptr);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    SDP_CHECK(comm_gather_rowbytes(h, s.sw_P, kSweepB * sizeof(double)));
    // 2. one stable radix sort per candidate of (key, input id): every rank sorts the whole vector
    for (int k = 0; k < nb; k++) {
        k_sw_keys<<<grid_for(n, 256, kRedBlocks * 4), 256, 0, h->stream>>>(n, k, s.sw_P, perm, s.sw_keys, s.sw_vals);
        KLAUNCH(h);
        size_t bytes = s.sw_cub_bytes;
        CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(s.sw_cub, bytes, s.sw_keys, s.sw_keys + n, s.sw_vals, s.sw_order + (size_t)k * n,
                                                    (int)n, 0, 64, h->stream));
        h->launches += 4;
    }
    // 3. deltas of the owned rows, all-gathered
    SDP_CHECK(neighbour_sums(h, SwDelta{s.sw_P, iperm, mask, s.sw_delta}, nullptr));
    SDP_CHECK(comm_gather_rowbytes(h, s.sw_delta, kSweepB * sizeof(double)));
    // 4. three-phase scan and selection
    double *tsum_d = s.sw_tiles, *tsum_w = tsum_d + nt * kSweepB, *tbest = tsum_w + nt * kSweepB;
    k_sw_tile_sums<<<dim3((unsigned)nt, nb), kSwTPB, 0, h->stream>>>(n, nt, s.sw_order, s.sw_delta, w, tsum_d, tsum_w);
    KLAUNCH(h);
    k_sw_tile_scan<<<nb, kSwTPB, 0, h->stream>>>(nt, tsum_d, tsum_w);
    KLAUNCH(h);
    k_sw_scan<<<dim3((unsigned)nt, nb), kSwTPB, 0, h->stream>>>(n, nt, s.sw_order, s.sw_delta, w, tsum_d, tsum_w, csum, wlo, whi, prof,
                                                               tbest);
    KLAUNCH(h);
    k_sw_select<<<nb, kSwTPB, 0, h->stream>>>(n, nt, tbest, s.sw_order, s.sw_P, iperm, sel);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    if (!words) return SDPLRP_OK;
    // 5. the chosen vectors as words, and their exact objective by the evaluation pass
    if (nrows > 0) {
        k_sw_words<<<grid_for(nrows, 256, kRedBlocks * 4), 256, 0, h->stream>>>(h->row_lo, h->row_hi, s.sw_P, iperm, sel, nb, s.words);
        KLAUNCH(h);
        CUDA_TRY(h, cudaGetLastError());
    }
    SDP_CHECK(comm_gather_rowbytes(h, s.words, sizeof(Word)));
    if (esum) SDP_CHECK(eval_pass(h, nb, esum));
    return SDPLRP_OK;
}

int32_t round_sweep(sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, const double *w, double wlo, double whi,
                    double *G_out, double *obj, double *sum, double *wS, int64_t *thresh, int64_t *best, double *best_x,
                    double *best_profile, int64_t *best_order) {
    const char *name = "round_sweep";
    SDP_CHECK(rounding_check(h, name, K, obj, best));
    SDP_CHECK(objective_check(h, name));
    if (std::isnan(wlo) || std::isnan(whi) || wlo > whi)
        return fail(h, SDPLRP_ERR_ARG, "round_sweep: the window needs wlo <= whi (no NaN)");
    const i64 n = h->n;
    const int r = h->r;
    if (w)
        for (i64 i = 0; i < n; i++)
            if (!(w[i] >= 0.0) || !std::isfinite(w[i]))
                return fail(h, SDPLRP_ERR_ARG, "round_sweep: vertex weight " + std::to_string(i) + " is negative or not finite");
    // sums: per batch 16 evaluation sums (all-reduced), then per batch + 1 (the recomputed best) 16 x kSwSel selections, sum of C
    const i64 nbatch = (K + kSweepB - 1) / kSweepB;
    const i64 sel_at = nbatch * kSweepB, csum_at = sel_at + (nbatch + 1) * kSweepB * kSwSel, sums_len = csum_at + 1;
    std::vector<double> Gh;
    SDP_CHECK(round_setup(h, K, G, seed, Gh, 0x5357454550ull, {double_bits(wlo), double_bits(whi), w ? 1ull : 2ull}, w, w ? n : 0,
                          "hyperplanes (K, seed, G), weights or window", sums_len, csum_at));
    RoundingState &s = h->rnd;
    SDP_CHECK(ensure_sweep_buffers(h));
    double *csum = s.sums + csum_at;
    const double *wd = nullptr;
    if (w) {
        if (!s.sw_w) SDP_CHECK(dev_alloc(h, &s.sw_w, n));
        SDP_CHECK(perm_upload(h, s.sw_w, w, 1, true));
        wd = s.sw_w;
    }
    for (i64 bt = 0; bt < nbatch; bt++) {
        const int nb = (int)std::min<i64>(kSweepB, K - bt * kSweepB);
        SDP_CHECK(sweep_batch(h, s.G + (size_t)(bt * kSweepB) * r, nb, wd, wlo, whi, csum, s.sums + sel_at + bt * kSweepB * kSwSel,
                              nullptr, true, s.sums + bt * kSweepB));
    }
    SDP_CHECK(comm_reduce_ptr(h, s.sums, (int)sel_at));
    std::vector<double> hs((size_t)sums_len);
    CUDA_TRY(h, cudaMemcpyAsync(hs.data(), s.sums, hs.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));

    const double sumC = hs[(size_t)csum_at];
    i64 kb = -1;
    for (i64 k = 0; k < K; k++) {
        const double *sl = hs.data() + sel_at + k * kSwSel;
        const i64 t = (i64)sl[1];
        const bool ok = t >= 0;
        obj[k] = ok ? sumC - 2.0 * hs[(size_t)k] : INFINITY;
        if (sum) sum[k] = ok ? (double)(n - 2 * t) : NAN;
        if (wS) wS[k] = ok ? sl[2] : NAN;
        if (thresh) thresh[k] = t;
        if (ok && (kb < 0 || obj[k] < obj[kb])) kb = k;
    }
    if (kb < 0) return fail(h, SDPLRP_ERR_ARG, "round_sweep: no threshold of any candidate satisfies the weight window");
    *best = kb + 1;
    if (G_out) std::copy(G, G + (size_t)(K * r), G_out);
    if (best_x || best_profile || best_order) {
        // the best candidate alone (same FMA chain, sort, deltas and tiles: the same order, profile and vector)
        if (best_profile) {
            if (!s.sw_prof) SDP_CHECK(dev_alloc(h, &s.sw_prof, n + 1));
        }
        SDP_CHECK(sweep_batch(h, s.G + (size_t)kb * r, 1, wd, wlo, whi, csum, s.sums + sel_at + nbatch * kSweepB * kSwSel,
                              best_profile ? s.sw_prof : nullptr, best_x != nullptr, nullptr));
        if (best_x) SDP_CHECK(download_signs(h, s.words, 0, best_x));
        if (best_profile) {
            CUDA_TRY(h, cudaMemcpyAsync(best_profile, s.sw_prof, (size_t)(n + 1) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        }
        if (best_order) {
            int64_t *ord = reinterpret_cast<int64_t *>(s.sw_keys);   // the sort is done: its key buffer holds the download
            k_sw_order_out<<<grid_for(n, 256, kRedBlocks * 4), 256, 0, h->stream>>>(n, s.sw_order, h->relabeled ? h->iperm : nullptr, ord);
            KLAUNCH(h);
            CUDA_TRY(h, cudaGetLastError());
            CUDA_TRY(h, cudaMemcpyAsync(best_order, ord, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
        }
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return SDPLRP_OK;
}
}  // namespace

void round_free(sdplrp_handle *h) {
    RoundingState &s = h->rnd;
    dev_free(&s.words); dev_free(&s.x); dev_free(&s.chunk_row); dev_free(&s.G); dev_free(&s.sums);
    dev_free(&s.want); dev_free(&s.flip); dev_free(&s.best_words); dev_free(&s.dirty);
    dev_free(&s.long_rows); dev_free(&s.long_sptr); dev_free(&s.seg_row); dev_free(&s.seg_start); dev_free(&s.seg_part);
    s.G_len = s.sums_len = 0;
    s.e_lo = s.e_hi = s.nchunks = 0;
    s.n_seg = s.l_lo = s.l_hi = s.s_lo = s.s_hi = 0;
    dev_free(&s.sw_P); dev_free(&s.sw_delta); dev_free(&s.sw_order); dev_free(&s.sw_keys); dev_free(&s.sw_vals); dev_free(&s.sw_cub);
    dev_free(&s.sw_tiles); dev_free(&s.sw_w); dev_free(&s.sw_prof);
    s.sw_cub_bytes = 0;
    s.sw_ntiles = 0;
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

extern "C" int32_t sdplrp_round_sweep(sdplrp_handle *h, int64_t K, const double *G, uint64_t seed, const double *w, double wlo,
                                      double whi, double *G_out, double *obj, double *sum, double *wS, int64_t *thresh, int64_t *best,
                                      double *best_x, double *best_profile, int64_t *best_order) {
    if (!h) return SDPLRP_ERR_ARG;
    return round_sweep(h, K, G, seed, w, wlo, whi, G_out, obj, sum, wS, thresh, best, best_x, best_profile, best_order);
}
