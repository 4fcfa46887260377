// gradient.cu -- y formation, assembly of S = C - sum (lambda_i - sigma v_i) A_i
// on the aggregated pattern, the sparse x dense-factor products, and the S*x
// product used by Lanczos.
//
// Reference: src/coreop.jl:205-317 (At_preprocess_sparse!, copy2y_lambda_sub_pvio!,
// At_preprocess!, At! left/right, g!) and src/structs.jl:90-145 (BDB' mul!).
//
// Design (not a translation)
//  * S is split as  S(y) = y_obj * C  +  S_dyn(y):  the objective's values are
//    static (Cfull, resident in HBM), only the "dynamic" slots that some
//    constraint touches are re-evaluated per iteration through a deterministic
//    slot->contributors gather (no atomics).  Constraints that are a single diagonal
//    entry never enter that gather: they are applied from per-row lists.
//  * The hot loop never multiplies by the full S.  It keeps CR = C*R by the
//    recurrence CR += alpha*CD (the same device the reference uses for the
//    residual vector, src/linesearch.jl:118) where CD = C*D is the ONE gather
//    pass per inner iteration; that pass also yields <C,DD'> = <D,CD> and
//    <C,RD'+DR'> = 2<D,CR> for the exact line search, and the gradient becomes
//    G = 2*(y_obj*CR + S_dyn*R): a streaming pass plus, only for constraints with
//    off-diagonal entries, a gather over the off-diagonal dynamic pattern.  CR is
//    rebuilt from scratch by every f! (major iteration), which bounds the drift.
//  * k_step_grad fuses the whole tail of an iteration (step, residual recurrence,
//    y, gradient, both norms) into one pass over the rows (sdplrp_step_g).
//  * Sparse x dense kernels walk the symmetric pattern (internal hub-first labels)
//    as CSR with rows binned by length: <= kRowGroupMax nonzeros -> one lane group
//    of exactly r/2 lanes per row (6 rows per warp at r = 10), fully predicated
//    blocks of 8 nonzeros; <= kRowWarpMax -> one warp per row (lane groups split the
//    nonzeros, 4 independent 128-bit gathers in flight per lane); longer rows are cut
//    into kRowWarpMax-nonzero chunks, one warp each, combined per row in chunk order.
//    Lanes own 128-bit slices of the r-vector; accumulators stay in registers; every
//    reduction has a fixed order.  L2 policies: pattern streams evict_first, gathers
//    of the hub prefix evict_last.
//  * The seam-level operators At!(Y,X) / At!(y,x) still use the full S (tests,
//    Lanczos); S is materialised from Cfull + dynamic slots on demand.
#include <algorithm>
#include "common.cuh"

namespace {

constexpr int TPB = 256;

// L2 eviction policies: the pattern streams (idx, val) and cold gathers are evict_first, gathers of the hub prefix
// (internal rows < hot_rows, preprocess.cu) evict_last, so that the hubs stay L2-resident across the pass
__device__ __forceinline__ unsigned long long pol_evict_last() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ unsigned long long pol_evict_first() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ int ldg_i32_hint(const int *p, unsigned long long pol) {
    int v;
    asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ double ldg_f64_hint(const double *p, unsigned long long pol) {
    double v;
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ double2 ldg_f64x2_hint(const double *p, unsigned long long pol) {
    double2 v;
    asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
}

// y_i = -min(ub_i, lambda_i - sigma*raw_i), y_{m+1} = 1   (src/coreop.jl:229-236)
__global__ void k_form_y(i64 m, double sigma, const double *__restrict__ lambda, const double *__restrict__ ub,
                         const double *__restrict__ raw, double *__restrict__ y) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i <= m; i += (i64)gridDim.x * blockDim.x) {
        if (i == m) { y[i] = 1.0; continue; }
        y[i] = -fmin(ub[i], lambda[i] - sigma * raw[i]);
    }
}

// static part: S[k] = y_obj * Cfull[k]
__global__ void k_S_static(i64 nnzF, double yobj, const double *__restrict__ cfull, double *__restrict__ S) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < nnzF; k += (i64)gridDim.x * blockDim.x) S[k] = yobj * cfull[k];
}

// dynamic slots: constraints first (in matrix order), objective last -- the
// accumulation order of the reference's CSC mat-vec (src/coreop.jl:221).
// MODE 0: write the total into S at both mirrored positions
// MODE 1: write the total into triu_out[slot]
// MODE 2: write only the constraint part into dyn_out[d]   (S_dyn of the hot loop)
template <int MODE>
__global__ void k_S_dynamic(i64 nd, double yobj, const int *__restrict__ dyn_slot, const int *__restrict__ dyn_ptr,
                            const int *__restrict__ dyn_nsd_end, const int *__restrict__ dyn_gid, const double *__restrict__ dyn_val,
                            const int *__restrict__ pos_a, const int *__restrict__ pos_b, const double *__restrict__ st,
                            const double *__restrict__ y, double *__restrict__ out) {
    for (i64 d = blockIdx.x * (i64)blockDim.x + threadIdx.x; d < nd; d += (i64)gridDim.x * blockDim.x) {
        double s = 0.0;
        // MODE 2 leaves out the single-diagonal-entry constraints (listed last): the hot loop applies them per row
        const int jend = (MODE == 2) ? dyn_nsd_end[d] : dyn_ptr[d + 1];
        for (int j = dyn_ptr[d]; j < jend; j++) s += dyn_val[j] * y[dyn_gid[j]];
        if (MODE == 2) { out[d] = s; continue; }
        const int t = dyn_slot[d];
        s += yobj * st[t];
        if (MODE == 1) {
            out[t] = s;
        } else {
            out[pos_a[d]] = s;
            const int pb = pos_b[d];
            if (pb >= 0) out[pb] = s;
        }
    }
}

__global__ void k_scale_copy(i64 len, double a, const double *__restrict__ x, double *__restrict__ y) {
    for (i64 k = blockIdx.x * (i64)blockDim.x + threadIdx.x; k < len; k += (i64)gridDim.x * blockDim.x) y[k] = a * x[k];
}

// ---- sparse x dense-factor kernels ------------------------------------------
template <int VEC>
struct Acc;
template <>
struct Acc<1> {
    double v;
    __device__ __forceinline__ void zero() { v = 0.0; }
    __device__ __forceinline__ void fma(double s, const double *p) { v += s * __ldg(p); }
    __device__ __forceinline__ void fma_hint(double s, const double *p, unsigned long long pol) { v += s * ldg_f64_hint(p, pol); }
    __device__ __forceinline__ void shfl_add(int o) { v += __shfl_xor_sync(0xffffffffu, v, o); }
    __device__ __forceinline__ void add_from_lane(const Acc &o, int src) { v += __shfl_sync(0xffffffffu, o.v, src & 31); }
    __device__ __forceinline__ void scale_add(double sc, double a, const double *p) { v = sc * (v + a * __ldg(p)); }
    __device__ __forceinline__ void accumulate_onto(double sc, const double *p) { v = p[0] + sc * v; }
    __device__ __forceinline__ void fma_reg(double s, const Acc &o) { v += s * o.v; }
    __device__ __forceinline__ void add_mem(const double *p) { v += p[0]; }
    __device__ __forceinline__ void scale(double sc) { v *= sc; }
    __device__ __forceinline__ double dot_ld(const double *p) const { return v * __ldg(p); }
    __device__ __forceinline__ double norm2() const { return v * v; }
    __device__ __forceinline__ void store(double *p) const { *p = v; }
    __device__ __forceinline__ void ld(const double *p) { v = __ldg(p); }
    __device__ __forceinline__ void ld_hint(const double *p, unsigned long long pol) { v = ldg_f64_hint(p, pol); }
    __device__ __forceinline__ double dot_reg(const Acc &o) const { return v * o.v; }
    __device__ __forceinline__ void add_reg_first(const Acc &o) { v = o.v + 1.0 * v; }   // accumulate_onto(1.0, .) on a preloaded value
};
template <>
struct Acc<2> {
    double2 v;
    __device__ __forceinline__ void zero() { v.x = v.y = 0.0; }
    __device__ __forceinline__ void fma(double s, const double *p) {
        const double2 x = ldg2(p);
        v.x += s * x.x; v.y += s * x.y;
    }
    __device__ __forceinline__ void fma_hint(double s, const double *p, unsigned long long pol) {
        const double2 x = ldg_f64x2_hint(p, pol);
        v.x += s * x.x; v.y += s * x.y;
    }
    __device__ __forceinline__ void shfl_add(int o) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
        v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
    }
    __device__ __forceinline__ void add_from_lane(const Acc &o, int src) {
        v.x += __shfl_sync(0xffffffffu, o.v.x, src & 31);
        v.y += __shfl_sync(0xffffffffu, o.v.y, src & 31);
    }
    __device__ __forceinline__ void scale_add(double sc, double a, const double *p) {
        const double2 x = ldg2(p);
        v.x = sc * (v.x + a * x.x); v.y = sc * (v.y + a * x.y);
    }
    __device__ __forceinline__ void scale(double sc) { v.x *= sc; v.y *= sc; }
    __device__ __forceinline__ void accumulate_onto(double sc, const double *p) {
        const double2 x = *reinterpret_cast<const double2 *>(p);
        v.x = x.x + sc * v.x; v.y = x.y + sc * v.y;
    }
    __device__ __forceinline__ void fma_reg(double s, const Acc &o) { v.x += s * o.v.x; v.y += s * o.v.y; }
    __device__ __forceinline__ void add_mem(const double *p) {
        const double2 x = *reinterpret_cast<const double2 *>(p);
        v.x += x.x; v.y += x.y;
    }
    __device__ __forceinline__ double dot_ld(const double *p) const {
        const double2 x = ldg2(p);
        return v.x * x.x + v.y * x.y;
    }
    __device__ __forceinline__ double norm2() const { return v.x * v.x + v.y * v.y; }
    __device__ __forceinline__ void store(double *p) const { *reinterpret_cast<double2 *>(p) = v; }
    __device__ __forceinline__ void ld(const double *p) { v = ldg2(p); }
    __device__ __forceinline__ void ld_hint(const double *p, unsigned long long pol) { v = ldg_f64x2_hint(p, pol); }
    __device__ __forceinline__ double dot_reg(const Acc &o) const { return v.x * o.v.x + v.y * o.v.y; }
    __device__ __forceinline__ void add_reg_first(const Acc &o) { v.x = o.v.x + 1.0 * v.x; v.y = o.v.y + 1.0 * v.y; }
};

// EPI 0: Y_i = scale * acc                                   (seam-level At!)
// EPI 1: Y_i = scale * (acc + yobj*ADD_i); sum0 += |Y_i|^2    (gradient)
// EPI 2: Y_i = acc; sum0 += <X_i, acc>; sum1 += <X_i, Z_i>    (CD = C*D with the line-search dots; CR = C*R with obj)
// EPI 3: Y_i += scale * acc
// EPI 4: Y_i += acc, then the sums of EPI 2 on the total     (second phase of the two-phase pass)
struct RowArgs {
    const int *rows;   // compacted row list of this class, nullptr = identity over [0, n_rows)
    i64 n_rows;
    const int *ptr, *idx;
    const int *beg_arr, *end_arr;  // row i covers [beg_arr[i], end_arr[i]); nullptr = ptr[i] / ptr[i+1] (two-phase pass: hub | tail columns)
    const double *val;
    const int *src;    // IND: value = val[src[k]]
    const double *X;
    double *Y;
    int r, G;
    int Gw;            // lanes per group of the warp-per-row kernels (= pieces per row when <= 16, else G)
    int G0;            // lanes per row of the class-0 kernel (= pieces per row: no idle lanes, no shuffles there)
    int hot_rows;      // gathers of columns < hot_rows are L2 evict_last
    double scale, yobj;
    const double *ADD, *Z;
    double *partials;
    unsigned *ticket;
    double *out;       // EPI != 0: out[0], out[1]
    i64 own_lo, own_hi;
    // long rows (> kRowWarpMax nonzeros) are cut into chunks: one warp per chunk, partial sums in `scratch`
    const int *chunk_start, *chunk_end, *chunk_row;
    const int *long_rows, *long_cptr;
    double *scratch;
    // VF (value-free rows, uniform off-diagonal C = vf_scale = +-2^k): the nonzeros contribute X_j unscaled, the diagonal
    // contributes (C_ii / vf_scale) * X_i, and the row total is scaled once -- the same bits as the valued sum
    const double *vf_diag;
    double vf_scale;
};

template <int VEC, int MAXU, int EPI, bool VF = false>
__device__ __forceinline__ void row_epilogue(const RowArgs &a, i64 i, Acc<VEC> (&acc)[MAXU], int lg, int nv, double &s0, double &s1,
                                             int G) {
#pragma unroll
    for (int u = 0; u < MAXU; u++) {
        const int c = lg + u * G;
        if (c < nv) {
            const size_t off = (size_t)i * a.r + c * VEC;
            if (VF) acc[u].scale(a.vf_scale);   // exact: a power of two
            if (EPI == 0) {
                acc[u].scale(a.scale);
            } else if (EPI == 3) {
                acc[u].accumulate_onto(a.scale, a.Y + off);  // Y_i + scale*acc
            } else if (EPI == 4) {
                acc[u].accumulate_onto(1.0, a.Y + off);      // hub part (phase one) + tail part
                s0 += acc[u].dot_ld(a.X + off);
                if (a.Z) {
                    Acc<VEC> t;
                    t.zero(); t.fma(1.0, a.X + off);
                    s1 += t.dot_ld(a.Z + off);
                }
            } else if (EPI == 1) {
                if (a.ADD) acc[u].scale_add(a.scale, a.yobj, a.ADD + off); else acc[u].scale(a.scale);
                s0 += acc[u].norm2();
            } else {
                s0 += acc[u].dot_ld(a.X + off);
                if (a.Z) {
                    Acc<VEC> t;
                    t.zero(); t.fma(1.0, a.X + off);
                    s1 += t.dot_ld(a.Z + off);
                }
            }
            acc[u].store(a.Y + off);
        }
    }
}

template <int EPI>
__device__ __forceinline__ void finish_sums(const RowArgs &a, double s0, double s1) {
    if (EPI == 0 || EPI == 3) return;
    double v[2] = {s0, s1};
    double *out = a.out;
    grid_sum_finalize<2>(v, a.partials, a.ticket, [&](double (&s)[2]) { out[0] = s[0]; out[1] = s[1]; });
}

#define VAL_AT(k) (IND ? __ldg(a.val + __ldg(a.src + (k))) : __ldg(a.val + (k)))

// Register budget handed to ptxas for the DEFAULT row kernels: the second __launch_bounds__ argument (minimum resident CTAs
// per SM).  Without it ptxas aims at 48-64 registers and splits the gathers of a block into dependent batches (1 + 2 + 5 in
// k_rows_group, 2 + 2 in k_rows_warp: profiles/r1_gather_size_sweep.md); with 3 (80 registers) it can keep them together.
// 0 = no second argument = the configuration every measurement of round 1 was taken with.  A/B: scripts/r2_launch_bounds.sh
// (make EXTRA="-DSDPLRP_LB_GROUP=3 -DSDPLRP_LB_WARP=3").
#ifndef SDPLRP_LB_GROUP
#define SDPLRP_LB_GROUP 0
#endif
#ifndef SDPLRP_LB_WARP
#define SDPLRP_LB_WARP 0
#endif
#if SDPLRP_LB_GROUP > 0
#define LB_GROUP __launch_bounds__(TPB, SDPLRP_LB_GROUP)
#else
#define LB_GROUP __launch_bounds__(TPB)
#endif
#if SDPLRP_LB_WARP > 0
#define LB_WARP __launch_bounds__(TPB, SDPLRP_LB_WARP)
#else
#define LB_WARP __launch_bounds__(TPB)
#endif

// class 0: one group of G0 lanes per row (G0 = pieces per row when that fits a warp: 6 rows per warp at r = 10);
// the row's nonzeros are taken NB at a time, fully predicated, so a row of <= NB nonzeros costs one round trip
// ptr -> idx/val -> gathers with NB independent 128-bit gathers in flight per lane
// VF: the rows carry no values (RowArgs::vf_diag): every nonzero weighs 1 except the diagonal
// (VF, one unit per row: at most 64 registers, 4 CTAs per SM as the valued kernel; ptxas would otherwise take 66 and drop to 3)
template <int VEC, int MAXU, bool IND, int EPI, int NB, bool VF>
__global__ void __launch_bounds__(TPB, VF && MAXU == 1 ? 4 : SDPLRP_LB_GROUP) k_rows_group(RowArgs a) {
    const int nv = a.r / VEC;
    const int G = a.G0;
    const int gpb = TPB / G;                       // groups per CTA (lanes beyond gpb*G idle)
    const int gib = threadIdx.x / G;
    const int lg = threadIdx.x - gib * G;
    const bool lane_ok = gib < gpb;
    const i64 group = (i64)blockIdx.x * gpb + gib;
    const i64 n_groups = (i64)gridDim.x * gpb;
    const unsigned long long p_hot = pol_evict_last(), p_str = pol_evict_first();
    double s0 = 0.0, s1 = 0.0;
    if (lane_ok)
    for (i64 q = group; q < a.n_rows; q += n_groups) {
        const i64 i = a.rows ? a.rows[q] : q;
        if (i < a.own_lo || i >= a.own_hi) continue;
        const int beg = a.beg_arr ? a.beg_arr[i] : a.ptr[i], end = a.end_arr ? a.end_arr[i] : a.ptr[i + 1];
        const double dii = VF ? a.vf_diag[i] : 0.0;
        Acc<VEC> acc[MAXU];
#pragma unroll
        for (int u = 0; u < MAXU; u++) acc[u].zero();
        for (int k0 = beg; k0 < end; k0 += NB) {
            int cc[NB];
            double vv[NB];
#pragma unroll
            for (int j = 0; j < NB; j++) {
                const bool ok = k0 + j < end;
                cc[j] = ok ? ldg_i32_hint(a.idx + k0 + j, p_str) : 0;
                if (VF) vv[j] = ok ? (cc[j] == (int)i ? dii : 1.0) : 0.0;
                else vv[j] = ok ? (IND ? __ldg(a.val + ldg_i32_hint(a.src + k0 + j, p_str)) : ldg_f64_hint(a.val + k0 + j, p_str)) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < MAXU; u++) {
                const int c = lg + u * G;
                if (c < nv) {
                    if (VF) {   // every gather of the block issued before the first use (vv = 0 past the row's end)
                        Acc<VEC> x[NB];
#pragma unroll
                        for (int j = 0; j < NB; j++) {
                            x[j].zero();
                            if (k0 + j < end) x[j].ld_hint(a.X + (size_t)cc[j] * a.r + c * VEC, cc[j] < a.hot_rows ? p_hot : p_str);
                        }
#pragma unroll
                        for (int j = 0; j < NB; j++) acc[u].fma_reg(vv[j], x[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < NB; j++)
                            if (k0 + j < end) acc[u].fma_hint(vv[j], a.X + (size_t)cc[j] * a.r + c * VEC, cc[j] < a.hot_rows ? p_hot : p_str);
                    }
                }
            }
        }
        row_epilogue<VEC, MAXU, EPI, VF>(a, i, acc, lg, nv, s0, s1, G);
    }
    finish_sums<EPI>(a, s0, s1);
}

// class 1: one warp per row; the 32/G lane groups take 4 nonzeros each per step.
// CHUNK: the work items are the kRowWarpMax-nonzero chunks of the long rows (class 2) and the warp leaves its partial
// sums in a.scratch (combined per row, in chunk order, by k_rows_combine) -- a hub row of 30 k nonzeros is spread over
// 60 warps instead of serialising one CTA, which is what lets the pass scale when the rows are divided among GPUs.
template <int VEC, int MAXU, bool IND, int EPI, bool CHUNK, bool VF>
__global__ void LB_WARP k_rows_warp(RowArgs a) {
    const int nv = a.r / VEC;
    const int lane = threadIdx.x & 31;
    // lane groups of Gw lanes split the nonzeros of the row.  Gw = the number of 16-byte pieces of a factor row when that is
    // <= 16 (5 at r = 10: six groups, 24 gathers in flight per warp step, lanes 30-31 idle) -- with the next power of two
    // (8) three lanes of every group idled: 16 gathers per step.  Wider rows keep power-of-two groups with several units.
    const int Gw = a.Gw, ng = 32 / Gw;
    const int grp = lane / Gw, lg = lane - grp * Gw;
    const bool lane_ok = grp < ng;
    const i64 warp = (i64)blockIdx.x * (TPB / 32) + (threadIdx.x >> 5);
    const i64 n_warps = (i64)gridDim.x * (TPB / 32);
    const unsigned long long p_hot = pol_evict_last(), p_str = pol_evict_first();
    double s0 = 0.0, s1 = 0.0;
    for (i64 q = warp; q < a.n_rows; q += n_warps) {  // warp-uniform
        const i64 i = CHUNK ? a.chunk_row[q] : (a.rows ? a.rows[q] : q);
        if (i < a.own_lo || i >= a.own_hi) continue;
        const int beg = CHUNK ? a.chunk_start[q] : (a.beg_arr ? a.beg_arr[i] : a.ptr[i]);
        const int end = CHUNK ? a.chunk_end[q] : (a.end_arr ? a.end_arr[i] : a.ptr[i + 1]);
        const double dii = VF ? a.vf_diag[i] : 0.0;
        Acc<VEC> acc[MAXU];
#pragma unroll
        for (int u = 0; u < MAXU; u++) acc[u].zero();
        for (int k0 = beg + grp * 4; lane_ok && k0 < end; k0 += ng * 4) {
            int cc[4];
            double vv[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const bool ok = k0 + j < end;
                cc[j] = ok ? ldg_i32_hint(a.idx + k0 + j, p_str) : 0;
                if (VF) vv[j] = ok ? (cc[j] == (int)i ? dii : 1.0) : 0.0;
                else vv[j] = ok ? (IND ? __ldg(a.val + ldg_i32_hint(a.src + k0 + j, p_str)) : ldg_f64_hint(a.val + k0 + j, p_str)) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < MAXU; u++) {
                const int c = lg + u * Gw;
                if (c < nv) {
                    if (VF) {   // every gather of the block issued before the first use (vv = 0 past the row's end)
                        Acc<VEC> x[4];
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            x[j].zero();
                            if (k0 + j < end) x[j].ld_hint(a.X + (size_t)cc[j] * a.r + c * VEC, cc[j] < a.hot_rows ? p_hot : p_str);
                        }
#pragma unroll
                        for (int j = 0; j < 4; j++) acc[u].fma_reg(vv[j], x[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; j++)
                            if (k0 + j < end) acc[u].fma_hint(vv[j], a.X + (size_t)cc[j] * a.r + c * VEC, cc[j] < a.hot_rows ? p_hot : p_str);
                    }
                }
            }
        }
        // sum the lane groups: xor offsets Gw, 2Gw, ... < 32 for power-of-two groups; otherwise group 0 adds the groups
        // 1, 2, ... in that order (every lane takes part in the shuffles, only group 0's totals are used)
        if ((Gw & (Gw - 1)) == 0) {
#pragma unroll
            for (int u = 0; u < MAXU; u++)
                for (int o = Gw; o < 32; o <<= 1) acc[u].shfl_add(o);
        } else {
#pragma unroll
            for (int u = 0; u < MAXU; u++) {
                const Acc<VEC> own = acc[u];
                for (int o = 1; o < ng; o++) acc[u].add_from_lane(own, (((lane_ok ? grp : 0) + o) % ng) * Gw + lg);
            }
        }
        if (grp == 0) {
            if (CHUNK) {
#pragma unroll
                for (int u = 0; u < MAXU; u++) {
                    const int c = lg + u * Gw;
                    if (c < nv) acc[u].store(a.scratch + (size_t)q * a.r + c * VEC);
                }
            } else {
                row_epilogue<VEC, MAXU, EPI, VF>(a, i, acc, lg, nv, s0, s1, Gw);
            }
        }
    }
    if (!CHUNK) finish_sums<EPI>(a, s0, s1);
}

// class 2, second step: per long row the chunk partials are added in chunk order, then the row epilogue
template <int VEC, int MAXU, int EPI, bool VF>
__global__ void __launch_bounds__(TPB) k_rows_combine(RowArgs a) {
    const int nv = a.r / VEC;
    const int lg = threadIdx.x & (a.G - 1);
    const i64 group = ((i64)blockIdx.x * TPB + threadIdx.x) / a.G;
    const i64 n_groups = (i64)gridDim.x * TPB / a.G;
    double s0 = 0.0, s1 = 0.0;
    for (i64 q = group; q < a.n_rows; q += n_groups) {
        const i64 i = a.long_rows[q];
        if (i < a.own_lo || i >= a.own_hi) continue;
        Acc<VEC> acc[MAXU];
#pragma unroll
        for (int u = 0; u < MAXU; u++) acc[u].zero();
        for (int c = a.long_cptr[q]; c < a.long_cptr[q + 1]; c++) {
#pragma unroll
            for (int u = 0; u < MAXU; u++) {
                const int p = lg + u * a.G;
                if (p < nv) acc[u].add_mem(a.scratch + (size_t)c * a.r + p * VEC);
            }
        }
        row_epilogue<VEC, MAXU, EPI, VF>(a, i, acc, lg, nv, s0, s1, a.G);
    }
    finish_sums<EPI>(a, s0, s1);
}

// Y[j,:] += scale*coeff * sum_k XB[:,k] D[k] B[j,k]     (src/structs.jl:135-145)
__global__ void k_lr_apply(i64 lo, i64 hi, int r, int s, i64 n, const double *__restrict__ XB, const double *__restrict__ Dg,
                           const double *__restrict__ B, const double *__restrict__ y, int gid, double scale,
                           double *__restrict__ Y) {
    const double coeff = scale * y[gid];
    for (i64 e = lo * r + blockIdx.x * (i64)blockDim.x + threadIdx.x; e < hi * r; e += (i64)gridDim.x * blockDim.x) {
        const i64 j = e / r;
        const int i = (int)(e - j * r);
        double t = 0.0;
        for (int k = 0; k < s; k++) t += XB[k * r + i] * Dg[k] * __ldg(&B[j + k * n]);
        Y[e] += coeff * t;
    }
}

// ---- SpMV (seam-level At!(y, aux, x)): y = S*x, 8 lanes per row -----------------
constexpr int SPMV_L = 8;
__global__ void __launch_bounds__(TPB) k_spmv(i64 n, const int *__restrict__ ptr, const int *__restrict__ idx,
                                              const double *__restrict__ S, const double *__restrict__ x,
                                              double *__restrict__ y) {
    const int lg = threadIdx.x & (SPMV_L - 1);
    const i64 warp_global = (i64)blockIdx.x * (TPB / 32) + (threadIdx.x >> 5);
    const i64 n_warps = (i64)gridDim.x * (TPB / 32);
    const int g_in_warp = (threadIdx.x & 31) / SPMV_L;
    constexpr int gpw = 32 / SPMV_L;
    for (i64 base = warp_global * gpw; base < n; base += n_warps * gpw) {
        const i64 i = base + g_in_warp;
        double t = 0.0;
        if (i < n)
            for (int k = ptr[i] + lg; k < ptr[i + 1]; k += SPMV_L) t += __ldg(S + k) * __ldg(x + __ldg(idx + k));
#pragma unroll
        for (int o = SPMV_L >> 1; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (i < n && lg == 0) y[i] = t;
    }
}

__global__ void __launch_bounds__(TPB) k_lr_dot(i64 n, const double *__restrict__ B, const double *__restrict__ x,
                                                double *__restrict__ partials, unsigned *__restrict__ ticket,
                                                double *__restrict__ out) {
    double acc[1] = {0.0};
    for (i64 j = blockIdx.x * (i64)blockDim.x + threadIdx.x; j < n; j += (i64)gridDim.x * blockDim.x) acc[0] += B[j] * x[j];
    grid_sum_finalize<1>(acc, partials, ticket, [&](double (&sv)[1]) { out[0] = sv[0]; });
}
__global__ void k_lr_axpy_vec(i64 n, const double *__restrict__ B, const double *__restrict__ dot, const double *__restrict__ Dg,
                              int k, const double *__restrict__ yv, int gid, double *__restrict__ out) {
    const double t = dot[0] * Dg[k] * yv[gid];
    for (i64 j = blockIdx.x * (i64)blockDim.x + threadIdx.x; j < n; j += (i64)gridDim.x * blockDim.x) out[j] += B[j] * t;
}

// objective slots of the line-search vectors from the fused sums of CD = C*D
__global__ void k_obj_slots(int ncls, const double *__restrict__ sums /* ncls x 2 */, double *a_rd_m, double *a_dd_m) {
    double s0 = 0.0, s1 = 0.0;
    for (int c = 0; c < ncls; c++) { s0 += sums[2 * c]; s1 += sums[2 * c + 1]; }
    if (a_dd_m) *a_dd_m = s0;        // <C, DD'> = <D, CD>
    if (a_rd_m) *a_rd_m = 2.0 * s1;  // <C, RD'+DR'> = 2 <D, CR>
}
__global__ void k_sum_slots(int ncls, const double *__restrict__ sums, int stride, double *out) {
    double s = 0.0;
    for (int c = 0; c < ncls; c++) s += sums[stride * c];
    *out = s;
}

// the hot-loop gradient without its gathered parts:  G_i = 2*(y_obj*CR_i + d_i*R_i),  d_i = S_dyn(i,i)  (src/coreop.jl:305-317
// with S = y_obj*C + S_dyn and C*R kept by recurrence); ||G||_F^2 fused.  Pure streaming: 3N bytes.
template <int VEC>
__global__ void __launch_bounds__(TPB) k_grad_diag(i64 lo, i64 hi, int r, double yobj, const double *__restrict__ CR,
                                                   const double *__restrict__ R, const int *__restrict__ rowc_ptr,
                                                   const double *__restrict__ rowc_val, const double *__restrict__ y,
                                                   const int *__restrict__ dyn_diag,
                                                   const double *__restrict__ dynS, double *__restrict__ G, double *partials,
                                                   unsigned *ticket, double *out) {
    const int nv = r / VEC;
    const i64 total = (hi - lo) * nv;
    double acc[1] = {0.0};
    for (i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x; e < total; e += (i64)gridDim.x * blockDim.x) {
        const i64 i = lo + e / nv;
        const int c = (int)(e - (i - lo) * nv);
        double d = 0.0;
        for (int p = rowc_ptr[i]; p < rowc_ptr[i + 1]; p++) d += rowc_val[p] * y[p];  // single-diagonal-entry constraints of row i
        if (dynS) {
            const int dd = dyn_diag[i];
            if (dd >= 0) d += dynS[dd];
        }
        const size_t off = (size_t)i * r + c * VEC;
        Acc<VEC> g;
        g.zero();
        g.fma(d, R + off);
        if (CR) g.scale_add(2.0, yobj, CR + off); else g.scale(2.0);
        acc[0] += g.norm2();
        g.store(G + off);
    }
    grid_sum_finalize<1>(acc, partials, ticket, [&](double (&s)[1]) { out[0] = s[0]; });
}

// The whole tail of an inner iteration for the rows and their per-row (single-diagonal-entry) constraints in ONE
// streaming pass (src/linesearch.jl:118-124, src/sdplr.jl:219, src/coreop.jl:229-236, 305-317, src/sdplr.jl:224-234):
//   R_i += a*D_i ;  CR_i += a*CD_i ;
//   for the constraints p of row i:  raw_p += a*(a*A_DD_p + A_RD_p) ;  y_p = -min(ub_p, lambda_p - sigma*raw_p)
//   G_i = 2*(y_obj*CR_i + (sum_p val_p*y_p + S_dyn(i,i))*R_i) ;  ||G||^2 and ||max(raw,lb)||^2 fused.
// 7N + ~9 doubles per constraint instead of the 9N + 3 m-vector passes of step / y / gradient / norm kernels.
// raw is double-buffered (raw_in -> raw_out): every piece-thread of a row re-derives y_p from raw_in, only piece 0 writes.
#ifndef SDPLRP_LB_TAIL   // as SDPLRP_LB_GROUP, for the fused tail: its seven m-vector loads per constraint are issued in four dependent batches at 40 registers
#define SDPLRP_LB_TAIL 0
#endif
#if SDPLRP_LB_TAIL > 0
#define LB_TAIL __launch_bounds__(TPB, SDPLRP_LB_TAIL)
#else
#define LB_TAIL __launch_bounds__(TPB)
#endif
template <int VEC>
__global__ void LB_TAIL k_step_grad(i64 lo, i64 hi, int r, double a, double sigma, double yobj,
                                                   const double *__restrict__ D, double *__restrict__ R,
                                                   const double *__restrict__ CD, double *__restrict__ CR,
                                                   const int *__restrict__ rowc_ptr, const double *__restrict__ rowc_val,
                                                   const double *__restrict__ lambda, const double *__restrict__ ub,
                                                   const double *__restrict__ lb, const double *__restrict__ raw_in,
                                                   double *__restrict__ raw_out, const double *__restrict__ q1v,
                                                   const double *__restrict__ q2v, double *__restrict__ y,
                                                   const int *__restrict__ dyn_diag, const double *__restrict__ dynS,
                                                   double *__restrict__ G, const double *__restrict__ pn2_rest,
                                                   double *partials, unsigned *ticket, double *gn2_out, double *pn2_out) {
    const int nv = r / VEC;
    const i64 total = (hi - lo) * nv;
    double acc[2] = {0.0, 0.0};
    for (i64 e = blockIdx.x * (i64)blockDim.x + threadIdx.x; e < total; e += (i64)gridDim.x * blockDim.x) {
        const i64 i = lo + e / nv;
        const int c = (int)(e - (i - lo) * nv);
        const size_t off = (size_t)i * r + c * VEC;
        // independent row loads first (in flight while the constraint chain below resolves)
        Acc<VEC> rr, cr;
        rr.zero(); cr.zero();
        rr.fma(1.0, R + off); rr.fma(a, D + off);           // R_i + a*D_i
        if (CR) { cr.fma(1.0, CR + off); cr.fma(a, CD + off); }
        double d = 0.0;
        for (int p = rowc_ptr[i]; p < rowc_ptr[i + 1]; p++) {
            const double v = raw_in[p] + a * (a * q2v[p] + q1v[p]);
            const double yp = -fmin(ub[p], lambda[p] - sigma * v);
            d += rowc_val[p] * yp;
            if (c == 0) {
                raw_out[p] = v;
                y[p] = yp;
                const double w = fmax(v, lb[p]);
                acc[1] += w * w;
            }
        }
        if (dynS) {
            const int dd = dyn_diag[i];
            if (dd >= 0) d += dynS[dd];
        }
        rr.store(R + off);
        if (CR) cr.store(CR + off);
        Acc<VEC> g;
        g.zero();
        g.fma_reg(d, rr);
        if (CR) g.fma_reg(yobj, cr);
        g.scale(2.0);
        acc[0] += g.norm2();
        g.store(G + off);
    }
    grid_sum_finalize<2>(acc, partials, ticket, [&](double (&s)[2]) { gn2_out[0] = s[0]; pn2_out[0] = s[1] + pn2_rest[0]; });
}

}  // namespace

// leading (hub) rows of a gathered factor whose gathers carry the L2 evict_last policy (hub-first internal order)
i64 tile_hot_rows(const sdplrp_handle *h) {
    if (h->hot_rows >= 0) return std::min<i64>(h->hot_rows, h->n);
    if (!h->relabeled) return 0;
    if (h->dealt) return h->n;  // multi-GPU deal: hubs are spread over the rank blocks; one policy for every gather, streams evict_first
    return std::min<i64>(h->n, (i64)(48.0 * 1024 * 1024) / (8 * (i64)std::max(1, h->r)));   // ~48 MB of leading factor rows
}

namespace {

int pick_group(int nv) {
    int G = 1;
    while (G < nv && G < 32) G <<= 1;
    return G;
}

struct Csr {
    const int *ptr, *idx;
    const double *val;
    const int *src;
    const RowClasses *cls;
};

// long_empty: the long rows (class 2) take the warp-per-row kernel over an EMPTY range (second phase of the two-phase pass:
// their nonzeros were all handled, chunked, in the first phase; only the epilogue is left)
// side streams of the row classes: everything enqueued on the main stream so far happens before them / they before what follows
static int32_t classes_fork(sdplrp_handle *h) {
    if (!h->class_streams[0]) return SDPLRP_OK;
    CUDA_TRY(h, cudaEventRecord(h->ev_fork, h->stream));
    for (int c = 0; c < 2; c++) CUDA_TRY(h, cudaStreamWaitEvent(h->class_streams[c], h->ev_fork, 0));
    h->fork_open = true;
    return SDPLRP_OK;
}
static int32_t classes_join(sdplrp_handle *h) {
    if (!h->class_streams[0]) return SDPLRP_OK;
    for (int c = 0; c < 2; c++) {
        CUDA_TRY(h, cudaEventRecord(h->ev_join[c], h->class_streams[c]));
        CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_join[c], 0));
    }
    h->fork_open = false;
    return SDPLRP_OK;
}

template <int VEC, int MAXU, bool IND, int EPI, bool VF>
int32_t launch_classes(sdplrp_handle *h, RowArgs a, const RowClasses &cls, const TileLayout &longs, double *sums /* 3 x 2 or null */,
                       bool long_empty = false, int class_mask = 7) {
    const int gpb = TPB / a.G;
    const int gpb0 = TPB / a.G0;
    const int spmm_cap = 16 * kNumSM;   // grid cap of the grid-stride row kernels (measured on C5: 8 / 16 / 32 CTAs per SM -> 4.07 / 3.98 / 3.98 ms)
    // The three row classes are independent (disjoint rows, their own sums, their own reduction scratch): the medium and the
    // long rows run on side streams next to the short rows.  On one GPU each kernel fills the machine anyway; with the rows
    // divided among 8 GPUs the medium / long kernels are a few hundred CTAs each and would otherwise run one after the other
    // at a fraction of the occupancy this latency-bound pass needs.
    const bool fork = h->class_streams[0] != nullptr;
    const bool own_fork = fork && !h->fork_open;   // a caller that issues several launches of one pass forks / joins around them
    if (own_fork) SDP_CHECK(classes_fork(h));
    for (int c = 0; c < 3; c++) {
        if (!(class_mask & (1 << c))) continue;   // this class belongs to another launch of the pass
        cudaStream_t st = (fork && c > 0) ? h->class_streams[c - 1] : h->stream;
        if (sums) a.out = sums + 2 * c;
        a.partials = h->partials + (size_t)c * 16384;   // <= spmm_cap CTAs x 2 sums per class
        a.ticket = h->ticket + c;
        a.rows = cls.list[c];
        a.n_rows = cls.cnt[c];
        if (a.n_rows <= 0) {
            if (sums) CUDA_TRY(h, cudaMemsetAsync(sums + 2 * c, 0, 2 * sizeof(double), st));
            continue;
        }
        if (c == 0) {
            if (h->spmm_unroll >= 8) k_rows_group<VEC, MAXU, IND, EPI, 8, VF><<<grid_for(a.n_rows, gpb0, spmm_cap), TPB, 0, st>>>(a);
            else k_rows_group<VEC, MAXU, IND, EPI, 4, VF><<<grid_for(a.n_rows, gpb0, spmm_cap), TPB, 0, st>>>(a);
        } else if (c == 1) {
            k_rows_warp<VEC, MAXU, IND, EPI, false, VF><<<grid_for(a.n_rows, TPB / 32, spmm_cap), TPB, 0, st>>>(a);
        } else if (long_empty) {
            RowArgs b = a;
            b.beg_arr = a.ptr + 1; b.end_arr = a.ptr + 1;
            k_rows_warp<VEC, MAXU, IND, EPI, false, VF><<<grid_for(b.n_rows, TPB / 32, spmm_cap), TPB, 0, st>>>(b);
        } else {
            // long rows: one warp per chunk, then the per-row combination with the epilogue
            const i64 need = longs.n_chunks * (i64)a.r;
            if (h->tile_scratch_len < need) {
                if (fork) CUDA_TRY(h, cudaDeviceSynchronize());   // (re)allocation under concurrent streams: rare, first call per rank
                SDP_CHECK(dev_alloc(h, &h->tile_scratch, need));
                h->tile_scratch_len = need;
            }
            RowArgs b = a;
            b.chunk_start = longs.chunk_start; b.chunk_end = longs.chunk_end; b.chunk_row = longs.chunk_row;
            b.long_rows = longs.long_rows; b.long_cptr = longs.long_cptr; b.scratch = h->tile_scratch;
            b.n_rows = longs.n_chunks;
            k_rows_warp<VEC, MAXU, IND, EPI, true, VF><<<grid_for(b.n_rows, TPB / 32, spmm_cap), TPB, 0, st>>>(b);
            KLAUNCH(h);
            b.n_rows = longs.n_long;
            k_rows_combine<VEC, MAXU, EPI, VF><<<grid_for(b.n_rows, gpb, 4 * kNumSM), TPB, 0, st>>>(b);
        }
        KLAUNCH(h);
    }
    if (own_fork) SDP_CHECK(classes_join(h));
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

template <bool IND, int EPI, bool VF = false>
int32_t launch_csr(sdplrp_handle *h, RowArgs a, const RowClasses &cls, const TileLayout &longs, double *sums, bool long_empty = false,
                   i64 hot_override = -1, int class_mask = 7) {
    const int r = h->r;
    const bool vec2 = (r % 2 == 0);
    const int nv = vec2 ? r / 2 : r;
    a.r = r;
    a.G = pick_group(nv);
    if (a.own_hi <= 0) {   // (a local pattern sets its own row range)
        a.own_lo = h->row_lo;
        a.own_hi = h->row_hi;
    }
    a.G0 = (nv <= 32 && h->spmm_g0) ? nv : a.G;   // class 0: exactly one lane per piece
    a.hot_rows = (int)(hot_override >= 0 ? hot_override : tile_hot_rows(h));
    const int units = (nv + a.G - 1) / a.G;
    a.Gw = (h->spmm_g0 && nv <= 16 && units == 1) ? nv : a.G;
    if (units > 4) return fail(h, SDPLRP_ERR_ARG, "rank too large for the sparse kernels (r <= 256 even / 128 odd)");
    if (vec2) {
        if (units == 1) return launch_classes<2, 1, IND, EPI, VF>(h, a, cls, longs, sums, long_empty, class_mask);
        return launch_classes<2, 4, IND, EPI, VF>(h, a, cls, longs, sums, long_empty, class_mask);
    }
    if (units == 1) return launch_classes<1, 1, IND, EPI, VF>(h, a, cls, longs, sums, long_empty, class_mask);
    return launch_classes<1, 4, IND, EPI, VF>(h, a, cls, longs, sums, long_empty, class_mask);
}

// mid[i] = first position of row i whose column is >= hub_cols (columns are ascending inside a row, hubs first)
__global__ void k_row_split(i64 n, const int *__restrict__ ptr, const int *__restrict__ idx, int hub_cols, int *__restrict__ mid) {
    for (i64 i = blockIdx.x * (i64)blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        int lo = ptr[i], hi = ptr[i + 1];
        while (lo < hi) {
            const int m = lo + ((hi - lo) >> 1);
            if (idx[m] < hub_cols) lo = m + 1; else hi = m;
        }
        mid[i] = lo;
    }
}

// Two-phase gather pass (option "spmm_phases", off by default; DESIGN.md section 8, profiles/r1_hub_tail_analysis.md):
// every row first takes its hub columns (an L2-sized prefix of the gathered factor), then -- in a second sweep over the
// rows -- its tail columns, so that the random tail fills do not evict the hub rows while they are still being reused.
// Only for the hub-first internal order on one GPU (the multi-GPU deal spreads the hubs over the rank blocks).
static i64 phase_hub_cols(const sdplrp_handle *h) {
    if (h->spmm_phases <= 0 || !h->relabeled || h->dealt || h->world > 1 || h->nnzF <= 0) return 0;
    const i64 want = h->spmm_phases == 1 ? (i64)(64.0 * 1024 * 1024) / (8 * (i64)std::max(1, h->r)) : (i64)h->spmm_phases;
    return std::min<i64>(want, h->n);
}
static int32_t ensure_row_mid(sdplrp_handle *h, i64 hub_cols) {
    if (h->row_mid && h->row_mid_cols == hub_cols) return SDPLRP_OK;
    SDP_CHECK(dev_alloc(h, &h->row_mid, h->n));
    k_row_split<<<grid_for(h->n, TPB, 8 * kNumSM), TPB, 0, h->stream>>>(h->n, h->full_ptr, h->full_idx, (int)hub_cols, h->row_mid);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    h->row_mid_cols = hub_cols;
    return SDPLRP_OK;
}

int32_t add_lowrank(sdplrp_handle *h, const double *X, double *Y, double scale) {
    if (h->lr.empty()) return SDPLRP_OK;
    const int r = h->r;
    SDP_CHECK(lr_scratch(h));
    for (const LowRank &L : h->lr) {
        SDP_CHECK(lr_project(h, L, X, h->lr_tmp));
        k_lr_apply<<<grid_for((h->row_hi - h->row_lo) * r, TPB, kRedBlocks), TPB, 0, h->stream>>>(
            h->row_lo, h->row_hi, r, (int)L.s, h->n, h->lr_tmp, L.dD, L.dB, h->y, (int)L.gid, scale, Y);
        KLAUNCH(h);
    }
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

}  // namespace

int32_t grad_form_y(sdplrp_handle *h) {
    k_form_y<<<grid_for(h->m + 1, TPB, kRedBlocks), TPB, 0, h->stream>>>(h->m, h->sigma, h->lambda, h->lambda_ub, h->pvio_raw, h->y);
    KLAUNCH(h);
    h->y_obj = 1.0;
    h->S_current = false;  // the hot loop never materialises S; Lanczos / At! re-assemble on demand
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

// At_preprocess!: materialise S = y_obj*C + S_dyn(y) on the full pattern (seam-level / Lanczos)
int32_t grad_assemble_S(sdplrp_handle *h) {
    h->S_current = true;
    SDP_CHECK(comm_gather_cvec(h, h->y));  // multi-GPU: S is replicated, so every rank needs every y_i
    if (h->nA <= 0) return SDPLRP_OK;
    cudaStream_t st = h->stream;
    const double yobj = (h->obj_mat >= 0) ? h->y_obj : 0.0;
    if (!h->S_static_valid || h->S_static_scale != yobj) {
        if (h->nnzF > 0) {
            k_S_static<<<grid_for(h->nnzF, TPB, 8 * kNumSM), TPB, 0, st>>>(h->nnzF, yobj, h->Cfull, h->S);
            KLAUNCH(h);
        }
        h->S_static_valid = true;
        h->S_static_scale = yobj;
    }
    if (h->n_dyn > 0) {
        k_S_dynamic<0><<<grid_for(h->n_dyn, TPB, 8 * kNumSM), TPB, 0, st>>>(h->n_dyn, yobj, h->dyn_slot, h->dyn_ptr, h->dyn_nsd_end, h->dyn_gid, h->dyn_val,
                                                                           h->dyn_pos_a, h->dyn_pos_b, h->triuS_static, h->y, h->S);
        KLAUNCH(h);
    }
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

int32_t grad_triuS(sdplrp_handle *h, double *out) {
    if (h->nnzT <= 0) return SDPLRP_OK;
    cudaStream_t st = h->stream;
    const double yobj = (h->obj_mat >= 0) ? h->y_obj : 0.0;
    k_scale_copy<<<grid_for(h->nnzT, TPB, 8 * kNumSM), TPB, 0, st>>>(h->nnzT, yobj, h->triuS_static, out);
    KLAUNCH(h);
    if (h->n_dyn > 0) {
        k_S_dynamic<1><<<grid_for(h->n_dyn, TPB, 8 * kNumSM), TPB, 0, st>>>(h->n_dyn, yobj, h->dyn_slot, h->dyn_ptr, h->dyn_nsd_end, h->dyn_gid, h->dyn_val,
                                                                           h->dyn_pos_a, h->dyn_pos_b, h->triuS_static, h->y, out);
        KLAUNCH(h);
    }
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

// seam-level At!(Y, X): Y = scale * (X*S + sum_g y_g X B D B') over the owned rows, S as last assembled
int32_t grad_spmm(sdplrp_handle *h, const double *X, double *Y, double scale, bool /*want_norm*/) {
    SDP_CHECK(grad_spmm_sparse(h, X, Y, scale));
    return add_lowrank(h, X, Y, scale);
}

// the sparse part alone (DIMACS error 6 of the reference leaves the low-rank terms out, src/coreop.jl:448-451)
int32_t grad_spmm_sparse(sdplrp_handle *h, const double *X, double *Y, double scale) {
    const int r = h->r;
    if (h->nA > 0 && gather_supported(h) && h->nnzF > 0) {
        SDP_CHECK(gather_plan_build(h, h->full_plan, h->full_ptr, h->row_lo, h->row_hi, gather_tile_size(h)));
        SDP_CHECK(gather_spmm(h, h->full_plan, h->full_ptr, h->full_idx, h->S, X, nullptr, nullptr, Y, 0, scale, nullptr));
    } else if (h->nA > 0) {
        RowArgs a = {};
        a.ptr = h->full_ptr; a.idx = h->full_idx; a.val = h->S; a.src = nullptr;
        a.X = X; a.Y = Y; a.scale = scale;
        SDP_CHECK((launch_csr<false, 0>(h, a, h->full_cls, h->full_long, nullptr)));
    } else {
        CUDA_TRY(h, cudaMemsetAsync(Y + h->row_lo * r, 0, (size_t)(h->row_hi - h->row_lo) * r * sizeof(double), h->stream));
    }
    return SDPLRP_OK;
}

// Y = C*X over the owned rows with the fused sums  out0 = <X, Y>, out1 = <X, Z>  (Z may be null)
// Several GPUs, halo plan active: Y = C*X over the own rows from the LOCAL pattern.  The caller started the exchange of the
// ghost rows of X (halo_begin).  Phase A: the [own | hub-ghost] columns of the short and medium rows as soon as the (small)
// hub class has arrived; phase B, once the tail class is in: their tail-ghost columns on top (with the fused dots of the
// pass) and the long rows whole.
static int32_t grad_obj_spmm_halo(sdplrp_handle *h, const double *X, double *Y, const double *Z, double *sums6) {
    const HaloPlan &p = h->halo;
    const size_t off = (size_t)h->row_lo * h->r;
    RowArgs a = {};
    a.ptr = p.lptr; a.idx = p.lidx; a.val = p.lval; a.src = nullptr;
    // the gathered operand is the compact array [own rows | hub ghosts | tail ghosts] that halo_begin filled (own rows copied,
    // ghosts received in place): one base pointer for every column, as on one GPU (a two-base select in the gather address
    // cost the row kernels 20-25 %: 2.30 -> 2.85 ms for the short-row kernel of C5)
    (void)X;
    a.X = p.xc; a.Y = Y + off; a.Z = Z ? Z + off : nullptr; a.scale = 1.0;
    a.own_lo = 0; a.own_hi = p.nloc;
    CUDA_TRY(h, cudaMemsetAsync(sums6, 0, 6 * sizeof(double), h->stream));
    // Two-phase (the tail exchange runs under phase A) or one sweep over whole rows once both classes are in?  The phases cost a
    // second visit of every short / medium row (measured: 1.27-1.33x the sweep) and can only hide what phase A lasts.  "auto"
    // compares the two with rates measured on B200 / NVLink 5 (profiles/r2_multigpu.md): exchange at 450 GB/s, sweep at 39
    // gathered rows/ns, constraint pass 0.1 ms + 3 TB/s under the exchange.  C5: one sweep at 2 and 8 GPUs, two phases at 4.
    bool single_sweep = h->halo_mode == 2;
    if (h->halo_mode == 3) {
        const double exch = (double)(p.n_ghost[0] + p.n_ghost[1]) * h->r * 8.0 / 450e9 * 1e3;      // ms
        const double sweep = (double)p.lnnz / 39e9 * 1e3;
        const double ls = 0.1 + 2.0 * (double)p.nloc * h->r * 8.0 / 3e12 * 1e3;
        const double hidden = std::min(std::max(0.0, exch - ls - 0.1), 0.58 * 1.27 * sweep);
        const double extra = 0.33 * sweep + 0.1;
        single_sweep = hidden < extra + 0.15;
    }
    if (single_sweep) {   // one sweep over whole rows once both classes are in (no second visit of the rows, exchange exposed)
        SDP_CHECK(halo_wait(h, 0));
        SDP_CHECK(halo_wait(h, 1));
        return launch_csr<false, 2>(h, a, p.cls, p.longs, sums6);
    }
    SDP_CHECK(halo_wait(h, 0));
    RowArgs a1 = a;
    a1.end_arr = p.lmid;                                   // phase A: plain store of the [own | hub] part
    SDP_CHECK((launch_csr<false, 0>(h, a1, p.cls, p.longs, nullptr, false, -1, 3)));
    SDP_CHECK(halo_wait(h, 1));
    RowArgs a2 = a;
    a2.beg_arr = p.lmid;                                   // phase B: tail part on top, dots on the total ...
    SDP_CHECK(classes_fork(h));
    int32_t rc = launch_csr<false, 4>(h, a2, p.cls, p.longs, sums6, false, -1, 3);
    if (rc == SDPLRP_OK) rc = launch_csr<false, 2>(h, a, p.cls, p.longs, sums6, false, -1, 4);   // ... next to the long rows: whole, chunked
    const int32_t rj = classes_join(h);
    return rc != SDPLRP_OK ? rc : rj;
}

int32_t grad_obj_spmm(sdplrp_handle *h, const double *X, double *Y, const double *Z, double *sums6) {
    if (halo_active(h)) return grad_obj_spmm_halo(h, X, Y, Z, sums6);
    if (gather_supported(h) && h->nnzF > 0) {   // asynchronous tile pipeline (gather.cu)
        SDP_CHECK(gather_plan_build(h, h->full_plan, h->full_ptr, h->row_lo, h->row_hi, gather_tile_size(h)));
        CUDA_TRY(h, cudaMemsetAsync(sums6 + 4, 0, 2 * sizeof(double), h->stream));
        return gather_spmm(h, h->full_plan, h->full_ptr, h->full_idx, h->Cfull, X, X, Z, Y, 2, 1.0, sums6);
    }
    RowArgs a = {};
    a.ptr = h->full_ptr; a.idx = h->full_idx; a.val = h->Cfull; a.src = nullptr;
    a.X = X; a.Y = Y; a.Z = Z; a.scale = 1.0;
    const i64 hub_cols = phase_hub_cols(h);
    if (hub_cols > 0 && hub_cols < h->n) {
        SDP_CHECK(ensure_row_mid(h, hub_cols));
        a.end_arr = h->row_mid;                       // phase one: hub columns (long rows: everything, chunked), plain store
        SDP_CHECK((launch_csr<false, 0>(h, a, h->full_cls, h->full_long, nullptr, false, hub_cols)));
        a.beg_arr = h->row_mid; a.end_arr = nullptr;  // phase two: tail columns on top, with the fused dots of the pass
        return launch_csr<false, 4>(h, a, h->full_cls, h->full_long, sums6, true, hub_cols);
    }
    if (obj_value_free(h)) {   // C = v * (0/1 pattern) off the diagonal, v = +-2^k: the value stream is not read
        a.val = nullptr; a.vf_diag = h->vf_diag; a.vf_scale = h->vf_val;
        return launch_csr<false, 2, true>(h, a, h->full_cls, h->full_long, sums6);
    }
    return launch_csr<false, 2>(h, a, h->full_cls, h->full_long, sums6);
}

// the hot-loop gradient: G = 2*(y_obj*CR + S_dyn(y)*R + low rank), ||G||_F^2 -> SC_GNORM2
//   1. dynS = constraint part of S at every dynamic slot (deterministic slot -> contributors gather)
//   2. streaming pass: G_i = 2*(y_obj*CR_i + S_dyn(i,i)*R_i) with the norm fused
//   3. only if some constraint has off-diagonal entries: G_i += 2*sum_j S_dyn(i,j)*R_j over the off-diagonal dynamic pattern
//   4. only with low-rank constraints: the BDB' terms; the norm is then taken in a separate pass
int32_t grad_hot(sdplrp_handle *h) {
    cudaStream_t st = h->stream;
    const int r = h->r;
    const bool need_dynS = h->n_dyn > 0 && h->n_dyn_nsd > 0;  // false for MaxCut-type problems: nothing but row-list constraints
    if (need_dynS) {
        k_S_dynamic<2><<<grid_for(h->n_dyn, TPB, 8 * kNumSM), TPB, 0, st>>>(h->n_dyn, 0.0, h->dyn_slot, h->dyn_ptr, h->dyn_nsd_end, h->dyn_gid, h->dyn_val,
                                                                           h->dyn_pos_a, h->dyn_pos_b, h->triuS_static, h->y, h->dynS);
        KLAUNCH(h);
    }
    const bool vec2 = (r % 2 == 0);
    const int nv = vec2 ? r / 2 : r;
    const i64 total = (h->row_hi - h->row_lo) * nv;
    const double *CR = (h->obj_mat >= 0) ? h->CR : nullptr;
    const int grid = grid_for(total, TPB * 2, kRedBlocks);
    if (vec2) k_grad_diag<2><<<grid, TPB, 0, st>>>(h->row_lo, h->row_hi, r, h->y_obj, CR, h->R, h->rowc_ptr, h->rowc_val, h->y, h->dyn_diag, need_dynS ? h->dynS : nullptr, h->G, h->partials, h->ticket, h->dscal + SC_GNORM2);
    else k_grad_diag<1><<<grid, TPB, 0, st>>>(h->row_lo, h->row_hi, r, h->y_obj, CR, h->R, h->rowc_ptr, h->rowc_val, h->y, h->dyn_diag, need_dynS ? h->dynS : nullptr, h->G, h->partials, h->ticket, h->dscal + SC_GNORM2);
    KLAUNCH(h);
    bool renorm = false;
    if (h->n_dynF > 0) {
        RowArgs a = {};
        a.ptr = h->dynrow_ptr; a.idx = h->dynrow_col; a.val = h->dynS; a.src = h->dynrow_src;
        a.X = h->R; a.Y = h->G; a.scale = 2.0;
        SDP_CHECK((launch_csr<true, 3>(h, a, h->dyn_cls, h->dyn_long, nullptr)));
        renorm = true;
    }
    if (!h->lr.empty()) {
        SDP_CHECK(add_lowrank(h, h->R, h->G, 2.0));
        renorm = true;
    }
    if (renorm) SDP_CHECK(lb_norm2(h, h->G, SC_GNORM2));
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

// sdplrp_step + sdplrp_g in one go (same results, 1 row pass instead of 3 + 4 m-vector passes):
//   Rt += alpha*dirt, CR += alpha*CD, residual recurrence, y, G, ||G||^2, ||pvio||^2.
// Caller guarantees: linesearch_coeffs ran for the current D (A_RD, A_DD, CD valid) and CR is valid (or C is not sparse).
int32_t grad_step_fused(sdplrp_handle *h, double alpha) {
    cudaStream_t st = h->stream;
    const int r = h->r;
    const bool split = h->obj_mat >= 0;
    double *raw_in = h->pvio_raw, *raw_out = h->pvio_raw_alt;
    double *pn2_rest = h->dscal + SC_SUMS + 2;
    SDP_CHECK(vec_tail_rest(h, alpha, raw_in, raw_out, pn2_rest));  // slots [n_sd, m]: raw, y, obj; its share of ||pvio||^2
    h->y_obj = 1.0;
    h->S_current = false;
    const bool need_dynS = h->n_dyn > 0 && h->n_dyn_nsd > 0;
    if (need_dynS) {
        k_S_dynamic<2><<<grid_for(h->n_dyn, TPB, 8 * kNumSM), TPB, 0, st>>>(h->n_dyn, 0.0, h->dyn_slot, h->dyn_ptr, h->dyn_nsd_end, h->dyn_gid, h->dyn_val,
                                                                           h->dyn_pos_a, h->dyn_pos_b, h->triuS_static, h->y, h->dynS);
        KLAUNCH(h);
    }
    const bool vec2 = (r % 2 == 0);
    const int nv = vec2 ? r / 2 : r;
    const i64 total = (h->row_hi - h->row_lo) * nv;
    // CTAs per SM: measured on C5, one GPU: 4 / 5 / 6 / 7 / 8 -> 1.156 / 1.101 / 0.975 / 1.305 / 1.198 ms (profiles/r2_call11_summary.txt);
    // the multi-GPU numbers of the round were taken with 4, which stays the value there
    const int ctas = h->tail_ctas > 0 ? h->tail_ctas : (h->world == 1 ? 6 : 4);
    const int grid = grid_for(total, TPB * 2, ctas * kNumSM);   // K = 2 sums: h->partials holds up to 8 CTAs per SM
    const double *CD = split ? h->CD : nullptr;
    double *CR = split ? h->CR : nullptr;
#define SG_ARGS h->row_lo, h->row_hi, r, alpha, h->sigma, h->y_obj, h->D, h->R, CD, CR, h->rowc_ptr, h->rowc_val, h->lambda, h->lambda_ub, \
                h->pvio_lb, raw_in, raw_out, h->A_RD, h->A_DD, h->y, h->dyn_diag, need_dynS ? h->dynS : nullptr, h->G, pn2_rest, h->partials, \
                h->ticket, h->dscal + SC_GNORM2, h->dscal + SC_PNORM2
    if (vec2) k_step_grad<2><<<grid, TPB, 0, st>>>(SG_ARGS);
    else k_step_grad<1><<<grid, TPB, 0, st>>>(SG_ARGS);
#undef SG_ARGS
    KLAUNCH(h);
    std::swap(h->pvio_raw, h->pvio_raw_alt);
    comm_mark_partial(h, SDPLRP_MAT_R);
    comm_mark_partial(h, SDPLRP_MAT_G);
    if (h->n_dynF > 0) SDP_CHECK(comm_require_full(h, SDPLRP_MAT_R));  // the off-diagonal dynamic part gathers rows of other ranks
    bool renorm = false;
    if (h->n_dynF > 0) {
        RowArgs a = {};
        a.ptr = h->dynrow_ptr; a.idx = h->dynrow_col; a.val = h->dynS; a.src = h->dynrow_src;
        a.X = h->R; a.Y = h->G; a.scale = 2.0;
        SDP_CHECK((launch_csr<true, 3>(h, a, h->dyn_cls, h->dyn_long, nullptr)));
        renorm = true;
    }
    if (!h->lr.empty()) {
        SDP_CHECK(add_lowrank(h, h->R, h->G, 2.0));
        renorm = true;
    }
    if (renorm) SDP_CHECK(lb_norm2(h, h->G, SC_GNORM2));
    SDP_CHECK(comm_reduce_scalars(h, SC_GNORM2, 2));  // ||G||^2 and ||pvio||^2 shares of the ranks
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

// objective slots of A_RD / A_DD from the sums of CD = C*D; pvio_raw[m] from those of CR = C*R
int32_t grad_obj_slots(sdplrp_handle *h, const double *sums6, double *a_rd_m, double *a_dd_m) {
    k_obj_slots<<<1, 1, 0, h->stream>>>(3, sums6, a_rd_m, a_dd_m);
    KLAUNCH(h);
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}

// y = S*x (+ low rank), x and y are n x ncols column-major device arrays
int32_t grad_spmv(sdplrp_handle *h, const double *x, double *y, i64 ncols) {
    cudaStream_t st = h->stream;
    const i64 n = h->n;
    for (i64 q = 0; q < ncols; q++) {
        const double *xq = x + q * n;
        double *yq = y + q * n;
        if (h->nA > 0) {
            k_spmv<<<grid_for(n, TPB / SPMV_L, 16 * kNumSM), TPB, 0, st>>>(n, h->full_ptr, h->full_idx, h->S, xq, yq);
            KLAUNCH(h);
        } else {
            CUDA_TRY(h, cudaMemsetAsync(yq, 0, (size_t)n * sizeof(double), st));
        }
        for (const LowRank &L : h->lr) {
            for (i64 k = 0; k < L.s; k++) {
                k_lr_dot<<<kRedBlocks, TPB, 0, st>>>(n, L.dB + k * n, xq, h->partials, h->ticket, h->dscal + SC_LANCZOS + 8);
                KLAUNCH(h);
                k_lr_axpy_vec<<<grid_for(n, TPB, kRedBlocks), TPB, 0, st>>>(n, L.dB + k * n, h->dscal + SC_LANCZOS + 8, L.dD, (int)k, h->y, (int)L.gid, yq);
                KLAUNCH(h);
            }
        }
    }
    CUDA_TRY(h, cudaGetLastError());
    return SDPLRP_OK;
}
