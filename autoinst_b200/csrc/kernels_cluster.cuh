// kernels_cluster.cuh — stage 3, persistent variant: ONE thread-block cluster runs the whole Lanczos
// iteration of ONE node (init, matvec, re-orthogonalisation, convergence checks, Ritz vector) without
// returning to the host.  Replaces eigsh(A, 2, sigma=1e-10) + argsort (normalized_cut.py:49-53) for
// nodes of up to CL_NMAX points; larger nodes keep the grid-wide multi-launch path (kernels_lanczos.cuh).
//
// The C CTAs of a cluster own C row slices of the node's block.  Per step:
//   matvec of the slice (W streamed from L2/HBM, z = S v for the whole node in shared memory), alpha out of its
//   epilogue and exchanged (pushed into every CTA, mbarrier bar_a), the three-term recurrence with the squared norm and
//   the z push in the same pass, the norm exchanged (pushed, bar_n, which also counts the z rows), then partial
//   re-orthogonalisation: the omega recurrence decides whether this step also takes ONE classical Gram-Schmidt pass
//   against u1 = D^1/2 1 and every Lanczos vector (partial dots over the slice exchanged through a cluster barrier and
//   remote reads, update, z and norm pushed again).  Every exchange is summed by every CTA in rank order, so all CTAs hold
//   bit-identical alpha/beta and take identical decisions.  A step without the pass: no cluster barrier, two mbarrier
//   waits and three block barriers, no sweep over the basis.
// MODE 7 (default) keeps the slice as CSR in shared memory instead of streaming W, and a node that converged there also
// takes its N-cut decision in the epilogue (cl_fused_cut).
// Every sum is float64 and evaluated in a fixed order: results do not depend on scheduling.
#pragma once
#include <cooperative_groups.h>
#include "common.cuh"
#include "kernels_graph.cuh"
#include "kernels_lanczos.cuh"
#include "kernels_ncut.cuh"

namespace ancuts {
namespace cg = cooperative_groups;

constexpr int CL_KMAX = 256;             // steps the cluster kernel can take; nodes needing more fall back
constexpr int CL_KS = CL_KMAX + 4;
constexpr int CL_RPMAX = 512;            // rows per CTA (two per thread)
constexpr int CL_NMAX = 4096;            // largest node handled here (8 CTAs x 512 rows)
constexpr int CL_THREADS = 512;          // 1024 threads (64 registers, 2 KB ring stages) measured 9 % slower (DESIGN.md 5a)
constexpr int CL_WARPS = CL_THREADS / 32;
constexpr int CL_HALF = CL_THREADS / 2;     // shifts per eigenvalue and bisection round
constexpr int CL_CLASSES = 6;            // node size bins (kernels_graph.cuh::cluster_class); cluster sizes 1, 2, 4, 8
constexpr double CL_REORTH_TOL = 0x1p-26;   // sqrt(eps): an estimated |v_j . v_i| above it triggers the full Gram-Schmidt pass
constexpr int CL_SHIFTS = CL_HALF / 2;   // shifts per eigenvalue and multisection round (cluster_tridiag_eigs)
constexpr int CL_DYN_SMEM = 194 * 1024;  // z for the whole node + as many basis rows of the slice as fit
                                         // (one CTA per SM; 256 threads x 2 CTAs per SM measured 25 % slower)

struct ClusterShared {
    double hpart[CL_KS];         // this CTA's partial dots of the Gram-Schmidt pass, read by the peers
    double npart[2];             // set-up: [1] = this CTA's "slice does not fit" flag, read by the peers
    double apart[8];             // step exchanges, slot [r] written by rank r with st.async: partials of alpha ...
    double nslot[8];             // ... and of the squared norm
    uint64_t bar_a, bar_n;       // their mbarriers (arrival count 1); bar_n also counts the z rows the peers push
    double spart[4];             // at the end: partial (sum, min, max, sum of squares) of the Ritz vector
    double hs[CL_KS];            // reduced projection coefficients
    double alpha[CL_KS], beta[CL_KS];
    double be2[CL_KS], dd[CL_KS], du[CL_KS], yv[CL_KS];
    short hexp[CL_KS], pexp[CL_KS];   // exponent offsets of dd / du (cluster_tridiag_vec)
    double prev_th[2];           // the two eigenvalues at the previous check (seed of the next multisection)
    float om[CL_KS];             // omega recurrence (partial re-orthogonalisation): om[i] estimates v_k . v_i for the newest
                                 // Lanczos vector v_k (float: only compared with sqrt(eps)); thread i also keeps om[i] and
                                 // its predecessor v_{k-1} . v_i in registers
    unsigned long long fdiff[NB + 1];   // fused cut: this CTA's difference array of cut weights, read by the peers
    unsigned long long fsum[NB + 1];    //            the node's difference array
    double fvol[NB];                    //            volume per bucket
    int fcnt[NB];                       //            points per bucket
    int fdec[4];                        //            decision: best threshold, split, side 0 passes, side 1 passes
    double ysl[2][CL_RPMAX];     // this CTA's slice of the current vector (ping) and of the matvec result (pong)
    double wred[CL_WARPS];       // per-warp partials of alpha (matvec epilogue)
    double wred2[CL_WARPS];      // per-warp partials of the norm (update): its own array, no barrier separates the two uses
    double sv[CL_RPMAX];         // D^-1/2 of the slice
    double red[32];
    double bounds[4];
    double gb[3];
    int cnts[2 * CL_SHIFTS];        // Sturm counts of the multisection (two eigenvalues x CL_SHIFTS shifts); fused cut: 16 x 11
    long long tmark;             // debug phase clock: end of the multisection rounds inside cluster_tridiag
    double prev_res;             // adaptive check schedule: residual estimate and step of the last check
    int prev_k;
    int next_check;
    int sp_nnz;                  // MODE 7: stored entries of the CSR slice (accounting)
};

// Adaptive convergence checks.  The fixed schedule (every 16 steps) runs 8 steps past convergence on average
// (14 % of the steps of the benchmark workload; no node converges before step 38).  Here the residual estimates
// of the last two checks give a geometric rate, the next check is placed at CL_CHECK_SAFETY x the predicted
// number of steps (Lanczos converges faster than geometrically at the end), clamped to [LO, HI].  numpy model
// over 87 nodes: 1.009 x the minimum number of steps (fixed 16: 1.14) with the same number of checks.
constexpr int CL_CHECK_FIRST = 28;
constexpr int CL_CHECK_LO = 2;
constexpr int CL_CHECK_HI = 12;
constexpr double CL_CHECK_SAFETY = 0.7;

__device__ __forceinline__ double block_sum_512(double v, double* red) {
    v = warp_sum(v);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < CL_WARPS; ++i) t += red[i];
    return t;
}
__device__ __forceinline__ double block_min_512(double v, double* red) {
    v = warp_min(v);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double t = red[0];
#pragma unroll
    for (int i = 1; i < CL_WARPS; ++i) t = fmin(t, red[i]);
    return t;
}

// Sturm count without divisions: the characteristic polynomials of the leading blocks,
// p_i = (a_i - x) p_{i-1} - b_{i-1}^2 p_{i-2}, change sign between consecutive i exactly where the pivots
// q_i = p_i / p_{i-1} of sturm_count() are negative.  One dependent FMA per element instead of one division
// (a float64 division is a ~12-instruction dependent sequence; the convergence checks were 8-13 % of the CTA time).
// |a_i - x| <= 2.3 and b^2 <= 1 bound the growth to 3.3x per step, so the pair is rescaled every 4 elements;
// an exact zero takes the sign opposite to its predecessor (the q = -pivmin rule).
// Signs are compared on the high words (integer pipe): an exact +-0 then takes the sign of its zero, and the total
// over the two steps around it is the same as with the q = -pivmin rule (p_{i+1} = -b^2 p_{i-1} there).
// al and be2 must be readable up to index k + 3 (CL_KS = CL_KMAX + 4 entries): the loads of the next group of four
// are unconditional so that they sit in front of the dependent FMA chain of the current one.
__device__ __forceinline__ int sturm_count_poly(const double* al, const double* be2, int k, double x) {
    double pm = 1.0, p = al[0] - x;
    int cnt = (int)((unsigned)__double2hiint(p) >> 31);       // p_{-1} = 1 > 0
#define STURM_STEP(c, e) do {                                                             \
        const double pn_ = fma((c), p, -((e) * pm));                                      \
        cnt += (int)((unsigned)(__double2hiint(pn_) ^ __double2hiint(p)) >> 31);          \
        pm = p; p = pn_;                                                                  \
    } while (0)
    int i = 1;
    double a0 = al[1], a1 = al[2], a2 = al[3], a3 = al[4], b0 = be2[0], b1 = be2[1], b2 = be2[2], b3 = be2[3];
    while (i + 3 < k) {
        const double c0 = a0 - x, c1 = a1 - x, c2 = a2 - x, c3 = a3 - x;
        const double e0 = b0, e1 = b1, e2 = b2, e3 = b3;
        i += 4;
        a0 = al[i]; a1 = al[i + 1]; a2 = al[i + 2]; a3 = al[i + 3];
        b0 = be2[i - 1]; b1 = be2[i]; b2 = be2[i + 1]; b3 = be2[i + 2];
        STURM_STEP(c0, e0); STURM_STEP(c1, e1); STURM_STEP(c2, e2); STURM_STEP(c3, e3);
        const int ex = (__double2hiint(p) >> 20) & 0x7ff;          // biased exponent
        if (ex > 1023 + 256) { p *= 0x1p-256; pm *= 0x1p-256; }
        else if (ex < 1023 - 256 && ex != 0) { p *= 0x1p256; pm *= 0x1p256; }
    }
    if (i < k) STURM_STEP(a0 - x, b0);                             // at most three elements left: no rescaling needed
    if (i + 1 < k) STURM_STEP(a1 - x, b1);
    if (i + 2 < k) STURM_STEP(a2 - x, b2);
#undef STURM_STEP
    return cnt;     // number of eigenvalues < x
}

// Tridiagonal analysis by the whole CTA (512 threads), part 1: the two largest eigenvalues of the k x k tridiagonal by
// multisection with CL_SHIFTS shifts per eigenvalue and round, until the brackets are one float64 step wide
// (129^8 > 2^56: eight rounds from the Gershgorin bracket).  From the second check of a node on, round 0 is SEEDED:
// the eigenvalues of T_k interlace those of T_{k'} for k' < k, so theta_i(k) >= theta_i(k'), and after the first few
// dozen steps they move by less than 1e-6 between checks; the shifts of round 0 then sit at prev + (hi - prev) 2^(-0.4 j),
// which brackets the new value to 30 % of the distance it moved, and 3-5 uniform rounds finish instead of 8.
// th[0], th[1] = eigenvalues (also kept in S.prev_th for the next check).
// CL_SHIFTS = 128: half as many warps on the FP64 pipe as with 256, same 8 rounds

__device__ __forceinline__ double cl_shift(double lo, double hi, int t, bool seeded) {
    if (t < 0) return lo;
    if (t >= CL_SHIFTS) return hi;
    if (!seeded) return lo + (hi - lo) * ((double)(t + 1) * (1.0 / (double)(CL_SHIFTS + 1)));
    return lo + (hi - lo) * exp2(-0.4 * (double)(CL_SHIFTS - t));      // t = CL_SHIFTS - 1 -> 0.76 (hi - lo); the bound hi follows
}

__device__ void cluster_tridiag_eigs(ClusterShared& S, int k, double* th) {
    const int tid = threadIdx.x;
    // Gershgorin bracket of the spectrum, by the whole CTA
    double lo_t = 1e300, hi_t = -1e300;
    for (int i = tid; i < k; i += CL_THREADS) {
        const double b = S.beta[i];
        S.be2[i] = b * b;
        const double rad = (i > 0 ? fabs(S.beta[i - 1]) : 0.0) + (i < k - 1 ? fabs(b) : 0.0);
        lo_t = fmin(lo_t, S.alpha[i] - rad);
        hi_t = fmax(hi_t, S.alpha[i] + rad);
    }
    lo_t = block_min_512(lo_t, S.red);
    hi_t = -block_min_512(-hi_t, S.red);
    const bool seeded = S.prev_k > 0;
    if (tid == 0) {
        const double w = fmax(fmax(fabs(lo_t), fabs(hi_t)), 1e-300);
        S.gb[0] = lo_t - 1e-10 * w;
        S.gb[1] = hi_t + 1e-10 * w;
        S.gb[2] = 0x1p-52 * w;                       // bracket width at which the multisection stops
        for (int e = 0; e < 2; ++e) {
            S.bounds[2 * e] = seeded ? fmax(S.prev_th[e] - 1e-12 * w, lo_t - 1e-10 * w) : lo_t - 1e-10 * w;
            S.bounds[2 * e + 1] = hi_t + 1e-10 * w;
        }
    }
    __syncthreads();
    const double eps = S.gb[2];
    const int which = tid / CL_SHIFTS, ts = tid % CL_SHIFTS;
    const bool act = which < 2 && (k - 1 - which) >= 0;
    const int m = k - 1 - which;
    for (int round = 0; round < 12; ++round) {
        const bool sd = seeded && round == 0;
        double lo = 0.0, hi = 0.0;
        if (which < 2) { lo = S.bounds[2 * which]; hi = S.bounds[2 * which + 1]; }
        if (act) S.cnts[tid] = sturm_count_poly(S.alpha, S.be2, k, cl_shift(lo, hi, ts, sd));
        __syncthreads();
        if (act && ts < 32) {                // one warp per eigenvalue finds the last shift with count <= m
            int best = -1;
            for (int i = ts; i < CL_SHIFTS; i += 32) if (S.cnts[which * CL_SHIFTS + i] <= m) best = max(best, i);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
            if (ts == 0) {
                S.bounds[2 * which] = cl_shift(lo, hi, best, sd);
                S.bounds[2 * which + 1] = cl_shift(lo, hi, best + 1, sd);
            }
        }
        __syncthreads();
        // every thread sees the same four bounds: uniform exit
        const bool done0 = (S.bounds[1] - S.bounds[0]) <= eps;
        const bool done1 = (k < 2) || (S.bounds[3] - S.bounds[2]) <= eps;
        if (done0 && done1) break;
    }
    const double th1 = 0.5 * (S.bounds[0] + S.bounds[1]);
    const double th2 = (k > 1) ? 0.5 * (S.bounds[2] + S.bounds[3]) : -1e300;
    __syncthreads();
    if (tid == 0) { S.prev_th[0] = th1; S.prev_th[1] = (k > 1) ? th2 : S.gb[0]; S.tmark = clock64(); }
    th[0] = th1;
    th[1] = th2;
}

// Part 2: eigenvector of th1 from the factorisation of T - th1 I twisted at the FIRST index, division-free.
// Bottom-up determinants of the trailing blocks, r_k = 1, r_{k-1} = a_{k-1} - th, r_i = (a_i - th) r_{i+1} - b_i^2 r_{i+2}:
// the trailing blocks of T do not contain the converged part of the Krylov space, their eigenvalues stay below th1
// (interlacing), so consecutive r have opposite signs and both terms of the recurrence add up (no cancellation; the
// forward recurrence from the first index cancels catastrophically once the Ritz value has converged).  The pivots of
// the twisted factorisation are r_i / r_{i+1} and the vector is z_i = (prod_{j<i} -b_j) r_{i+1} / r_1: ONE dependent
// FMA and one multiply per element instead of a float64 division (a ~30-instruction dependent sequence; the serial
// part of a check was 2 % of the CTA time in the dense form and a quarter of it in the shared-memory sparse form).
// Thread 0 runs the r chain, thread 32 the product chain (exponents tracked separately so that neither overflows),
// then all threads form z and the norm.  Agreement with LAPACK on every component: 1e-14 (numpy model, 160 steps).
// Returns the residual estimate beta_{k-1} |y_{k-1}|; S.yv = unit eigenvector.
__device__ double cluster_tridiag_vec(ClusterShared& S, int k, double th1) {
    const int tid = threadIdx.x;
    // S.dd[i] = r_{i+1} (scaled), S.hexp[i] = its exponent offset; S.du[i] = prod_{j<i} -b_j (scaled), S.pexp[i]
    if (tid == 0) {
        double rp = 1.0, rc = S.alpha[k - 1] - th1;          // r_k, r_{k-1}
        int e = 0;
        S.dd[k - 1] = 1.0; S.hexp[k - 1] = 0;                // r_k goes with z_{k-1}
        if (k >= 2) { S.dd[k - 2] = rc; S.hexp[k - 2] = 0; } // r_{k-1} goes with z_{k-2}
        for (int i = k - 2; i >= 0; --i) {                   // r_i from r_{i+1} = rc, r_{i+2} = rp
            const double rn = fma(S.alpha[i] - th1, rc, -(S.be2[i] * rp));
            rp = rc; rc = rn;
            const int ex = (__double2hiint(rc) >> 20) & 0x7ff;
            if (ex > 1023 + 256) { rc *= 0x1p-256; rp *= 0x1p-256; e += 256; }
            else if (ex < 1023 - 256 && ex != 0) { rc *= 0x1p256; rp *= 0x1p256; e -= 256; }
            if (i >= 1) { S.dd[i - 1] = rc; S.hexp[i - 1] = e; }     // r_i goes with z_{i-1}
        }
        (void)rc;                                            // r_0 = the twist pivot's numerator: only a common factor
    } else if (tid == 32) {
        double p = 1.0;
        int f = 0;
        for (int i = 0; i < k; ++i) {
            S.du[i] = p; S.pexp[i] = f;
            if (i < k - 1) {
                p *= -S.beta[i];
                const int ex = (__double2hiint(p) >> 20) & 0x7ff;
                if (ex < 1023 - 256 && ex != 0) { p *= 0x1p256; f -= 256; }
            }
        }
    }
    __syncthreads();
    // z_i = P_i r_{i+1} up to a common factor.  The largest recorded exponent is the reference, so that nothing overflows
    // even when the start vector was almost orthogonal to the Ritz vector (z_0 tiny against later components); anything
    // 2^-1000 below the largest component is zero for the Ritz sum.
    double emax_t = -1e9;
    for (int i = tid; i < k; i += CL_THREADS) emax_t = fmax(emax_t, (double)(S.pexp[i] + S.hexp[i]));
    const int emax = (int)(-block_min_512(-emax_t, S.red));
    double ss = 0.0;
    for (int i = tid; i < k; i += CL_THREADS) {
        const int ex = S.pexp[i] + S.hexp[i] - emax;
        double z = S.du[i] * S.dd[i];
        z = (ex < -1000) ? 0.0 : ldexp(z, ex);
        S.yv[i] = z;
        ss = fma(z, z, ss);
    }
    ss = block_sum_512(ss, S.red);
    const double inv = 1.0 / sqrt(ss);
    for (int i = tid; i < k; i += CL_THREADS) S.yv[i] *= inv;
    __syncthreads();
    return fabs(S.beta[k - 1] * S.yv[k - 1]);
}

template <int C>
__device__ __forceinline__ void cl_sync(cg::cluster_group& cl) {
    if (C > 1) cl.sync(); else __syncthreads();
}

// Basis rows restricted to this CTA's slice: the first rows_s rows live in shared memory, later rows
// (long runs) spill to the global basis V.
struct SliceBasis {
    double* smem;          // rows_s rows of stride nrp
    double* glob;          // e.V + first global position of the slice; row stride P
    size_t P;
    int rows_s;
    int nrp;
    __device__ __forceinline__ double* row(int j) const {
        return (j < rows_s) ? smem + (size_t)j * nrp : glob + (size_t)j * P;
    }
    __device__ __forceinline__ double get(int j, int i) const {
        return (j < rows_s) ? smem[(size_t)j * nrp + i] : glob[(size_t)j * P + i];
    }
    __device__ __forceinline__ void put(int j, int i, double v) const {
        row(j)[i] = v;
    }
};

// partial dots of the slice vector y with basis rows [0, rows): S.hpart[j].  One warp per row,
// all loads of a row in flight at once (nr <= CL_RPMAX = 16 * 32).
// (Forming the three-term values inside this pass -- every warp from yraw, v_k, v_{k-1}, no barrier in between -- was built
// and measured: bit-identical results, 3 % SLOWER: sixteen warps re-read v_k and v_{k-1}, from L2 once the basis has outgrown
// its shared-memory part.)
template <int M>
__device__ __forceinline__ double cl_dot_row(const double* __restrict__ vr, const double (&yr)[M], int lane, int nr) {
    // the slice has more than 32 (M - 4) rows: only the last four blocks of 32 need the bound check
    double t[M];
#pragma unroll
    for (int m = 0; m < M; ++m) { const int i = lane + 32 * m; t[m] = (m < M - 4 || i < nr) ? vr[i] : 0.0; }
    double s = 0.0;
#pragma unroll
    for (int m = 0; m < M; ++m) s += t[m] * yr[m];
    return warp_sum(s);
}
template <int M>
__device__ __forceinline__ void cl_partial_dots_m(ClusterShared& S, const double* __restrict__ y, const SliceBasis& B,
                                                  int rows, int nr) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double yr[M];
#pragma unroll
    for (int m = 0; m < M; ++m) { int i = lane + 32 * m; yr[m] = (i < nr) ? y[i] : 0.0; }
    // rows in shared memory, then rows in global memory: two loops, so that the loads are LDS / LDG instead of generic
    const int rs = min(rows, B.rows_s);
    int j = warp;
    for (; j < rs; j += CL_WARPS) {
        const double s = cl_dot_row<M>(B.smem + (size_t)j * B.nrp, yr, lane, nr);
        if (lane == 0) S.hpart[j] = s;
    }
    for (; j < rows; j += CL_WARPS) {
        const double s = cl_dot_row<M>(B.glob + (size_t)j * B.P, yr, lane, nr);
        if (lane == 0) S.hpart[j] = s;
    }
}
// slices of up to 128 / 256 / 384 / 512 rows: the loads and products beyond the slice (zeros) are not issued; same sums
__device__ __forceinline__ void cl_partial_dots(ClusterShared& S, const double* __restrict__ y, const SliceBasis& B,
                                                int rows, int nr) {
    static_assert(CL_RPMAX == 512, "four tiers of 128 rows");
    if (nr <= 128) cl_partial_dots_m<4>(S, y, B, rows, nr);
    else if (nr <= 256) cl_partial_dots_m<8>(S, y, B, rows, nr);
    else if (nr <= 384) cl_partial_dots_m<12>(S, y, B, rows, nr);
    else cl_partial_dots_m<16>(S, y, B, rows, nr);
}

template <int C>
__device__ __forceinline__ void cl_reduce_h(cg::cluster_group& cl, ClusterShared& S, int rows, int buf) {
    for (int j = threadIdx.x; j < rows; j += CL_THREADS) {
        double h = 0.0;
        if (C > 1) {
#pragma unroll
            for (int r = 0; r < C; ++r) h += cl.map_shared_rank(&S.hpart[0], r)[j];     // rank order
        } else {
            h = S.hpart[j];
        }
        S.hs[j] = h;
    }
    __syncthreads();
}

// y_i -= sum_j hs[j] V[j][i] for the slice; returns this thread's share of |y|^2 (the norm rides on the update pass)
__device__ __forceinline__ double cl_update_norm(const double* __restrict__ hs, double* __restrict__ y, const SliceBasis& B,
                                                 int rows, int nr) {
    // Rows [0, rows_s) of the basis sit in shared memory (stride nrp), the rest in global memory (stride P).  A group of
    // rows that lies on one side is walked with a stepping pointer; B.get's per-element select and two 64-bit address
    // products were 22 % of all instructions the kernel executed (ncu source view).  Same groups, same two chains, same
    // order as before: bit-identical sums.
    double q = 0.0;
    const int rs = B.rows_s;
    for (int i = threadIdx.x; i < nr; i += CL_THREADS) {
        double v = y[i];
        int j = 0;
        double c0 = 0.0, c1 = 0.0;                        // the correction sum_j hs[j] V[j][i] in two chains (fixed order)
        for (; j + 12 <= rows; j += 12) {                 // 12 basis rows in flight: the rows behind the shared-memory part come
            double t[12];                                 // from L2 / HBM while other SMs stream W, one round trip per group
            if (j + 12 <= rs) {
                const double* p = B.smem + (size_t)j * B.nrp + i;
#pragma unroll
                for (int u = 0; u < 12; ++u) { t[u] = *p; p += B.nrp; }
            } else if (j >= rs) {
                const double* p = B.glob + (size_t)j * B.P + i;
#pragma unroll
                for (int u = 0; u < 12; ++u) { t[u] = *p; p += B.P; }
            } else {
#pragma unroll
                for (int u = 0; u < 12; ++u) t[u] = B.get(j + u, i);
            }
#pragma unroll
            for (int u = 0; u < 12; u += 2) { c0 = fma(hs[j + u], t[u], c0); c1 = fma(hs[j + u + 1], t[u + 1], c1); }
        }
        for (; j + 4 <= rows; j += 4) {
            double t[4];
            if (j + 4 <= rs) {
                const double* p = B.smem + (size_t)j * B.nrp + i;
#pragma unroll
                for (int u = 0; u < 4; ++u) { t[u] = *p; p += B.nrp; }
            } else if (j >= rs) {
                const double* p = B.glob + (size_t)j * B.P + i;
#pragma unroll
                for (int u = 0; u < 4; ++u) { t[u] = *p; p += B.P; }
            } else {
#pragma unroll
                for (int u = 0; u < 4; ++u) t[u] = B.get(j + u, i);
            }
#pragma unroll
            for (int u = 0; u < 4; u += 2) { c0 = fma(hs[j + u], t[u], c0); c1 = fma(hs[j + u + 1], t[u + 1], c1); }
        }
        for (; j < rows; ++j) c0 = fma(hs[j], B.get(j, i), c0);
        v -= c0 + c1;
        y[i] = v;
        q = fma(v, v, q);
    }
    return q;
}

// ---- the two exchanges of a Lanczos step (C > 1) are one-way pushes onto mbarriers, no cluster barrier:
//   alpha: thread 0 posts expect_tx(8 C) on its bar_a and st.async's its partial into apart[rank] of every CTA, itself
//          included; every thread waits for the phase and sums apart[0 .. C) in rank order.
//   norm:  the three-term pass st.async's z into the peers' z buffers, counted on their bar_n; thread 0 posts
//          expect_tx(8 (n - nr + C)) -- the z rows of all peers plus the C norm partials -- and pushes its partial into
//          nslot[rank] of every CTA.  A full Gram-Schmidt pass pushes z and the norm again in a phase of its own.
// Ordering (why no push lands in a phase it does not belong to, and no slot or z element is overwritten before it is read):
//   a peer's alpha push of step k+1 follows its matvec k+1, which waited for OUR z of step k, which we push after our
//   bar_a wait of step k; its z / norm push of step k+1 needs our alpha of step k+1, which we push after our last bar_n wait
//   of step k; its pushes of a full pass follow the pass's cluster barrier, which we enter after our first bar_n wait of the
//   step.  So every phase completes before a push of the next phase of the same barrier can arrive (a push that arrives
//   before the local expect_tx only makes the transaction count negative for a while; the phase cannot complete before
//   that arrival).  A peer rewrites our apart slots only after our next norm push, and our nslot slots only after our
//   next alpha push or the full pass's cluster barrier; a block barrier separates every thread's read of the slots from
//   each of these.  Our z pushes follow the peers' alpha partials of the step, so their matvec, the only reader of z, has
//   ended.  The phase parities follow from the step count: bar_a completes once per step (k & 1), bar_n once more per full
//   pass ((k + full passes) & 1).
// The sums start at 0.0 and add the ranks in order, as the cluster-barrier form with remote reads did: the same bits.
// ANCUTS_EXCHANGE_GUARD (debug builds): a wait gives up after a bounded number of polls and the step loop stops with
// e.ctr[19] counted, so a protocol error fails the call instead of hanging the GPU.
__device__ __forceinline__ bool cl_wait(uint64_t* bar, uint32_t parity) {
#ifdef ANCUTS_EXCHANGE_GUARD
    bool ok = false;
    for (uint32_t it = 0; it < (1u << 22) && !ok; ++it) ok = mbarrier_try_wait_cluster(bar, parity);
    return !__syncthreads_or(!ok);
#else
    while (!mbarrier_try_wait_cluster(bar, parity)) {}
    return true;
#endif
}
// x = sum over the cluster of every CTA's x, through `slots` and `bar` (bytes: what this CTA receives in the phase)
template <int C>
__device__ __forceinline__ bool cl_exchange(double* slots, uint64_t* bar, uint32_t parity, uint32_t bytes, int rank, double& x) {
    if (threadIdx.x == 0) {
        mbarrier_expect_tx(bar, bytes);
        const uint32_t sa = smem_addr_u32(slots + rank), ba = smem_addr_u32(bar);
#pragma unroll 1
        for (int r = 0; r < C; ++r) st_async_f64(mapa_u32(sa, r), x, mapa_u32(ba, r));
    }
    const bool ok = cl_wait(bar, parity);
    double t = 0.0;
#pragma unroll
    for (int r = 0; r < C; ++r) t += slots[r];
    x = t;
    return ok;
}

// z = S y for the next matvec: element j of the node's z vector into the z buffer of every CTA of the cluster.  The own
// copy is a plain store (the block barrier of the norm sum orders it before the next matvec), the peers' copies are
// counted on their bar_n.
template <int C>
__device__ __forceinline__ void cl_put_z(ClusterShared& S, double* zs, int rank, int j, double zv) {
    zs[j] = zv;
    if (C > 1) {
        const uint32_t za = smem_addr_u32(zs + j), ba = smem_addr_u32(&S.bar_n);
#pragma unroll 1
        for (int r = 0; r < C; ++r)
            if (r != rank) st_async_f64(mapa_u32(za, r), zv, mapa_u32(ba, r));
    }
}
template <int C>
__device__ __forceinline__ void cl_push_z(ClusterShared& S, double* zs, int rank, const double* y, int r0, int nr, int pad) {
    for (int i = threadIdx.x; i < nr; i += CL_THREADS) cl_put_z<C>(S, zs, rank, r0 + i + pad, S.sv[i] * y[i]);
}

// sum over the CTA of one value per thread: warp partials in S.wred2, ONE block barrier, fixed order
__device__ __forceinline__ double cl_block_sum1(ClusterShared& S, double v) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) S.wred2[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < CL_WARPS; ++i) t += S.wred2[i];
    return t;
}

// norm of the node's vector from the CTAs' squared partial norms q; the phase also completes the peers' z pushes
template <int C>
__device__ __forceinline__ bool cl_norm_exchange(ClusterShared& S, uint32_t parity, int n, int nr, int rank, double& q) {
    bool ok = true;
    if (C > 1) ok = cl_exchange<C>(S.nslot, &S.bar_n, parity, 8u * (uint32_t)(n - nr + C), rank, q);
    q = sqrt(q);
    return ok;
}

// float -> double widening on the integer pipe, for weights in {0} U [2^-126, 2): the bits move 29 places and the
// exponent is re-biased; +0 becomes 2^-127 (5.9e-39), which every later float64 sum absorbs exactly.
// cvt.f64.f32 runs on the XU pipe at 4 lanes per clock and scheduler: ncu shows it half busy during the matvec and
// the warps waiting on it, so in the MIX variant every second element is widened with three integer instructions.
__device__ __forceinline__ double widen_int(float f) {
    const unsigned b = __float_as_uint(f);
    return __hiloint2double((int)((b >> 3) + 0x38000000u), (int)(b << 29));
}
template <bool MIX>
__device__ __forceinline__ double widen_alt(float f) { return MIX ? widen_int(f) : (double)f; }

// ---- guarded matvec (MODE 0, stage entry points on the caller's W): register-staged loads, entries outside the block
// are selected away (they may be uninitialised or belong to other nodes).
// yout_i = s_i * invb * (sum_j w_ij z_j + z_i) for the rows [r0, r0+nr); returns (lane 0) the warp's share of
// alpha = v . (M v), v_i = yin_i * invb.
__device__ __forceinline__ double cl_matvec_guard(ClusterShared& S, const double* zs, const double* __restrict__ yin,
                                                  double* __restrict__ yout, const NodeView& v, int r0, int nr, int pad,
                                                  double invb) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c_lo = v.ro, c_hi = v.ro + v.n, a0 = c_lo & ~3;
    double pa = 0.0;
    for (int rb = warp * 2; rb < nr; rb += CL_WARPS * 2) {
        const float* rpt[2];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) rpt[rr] = v.W + (size_t)(v.ro + r0 + min(rb + rr, nr - 1)) * v.ld;
        double acc[2] = {0.0, 0.0};
        for (int c = a0 + lane * 4; c < c_hi; c += 512) {
            float4 w[2][4];
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const int cg_ = c + 128 * g;
                const bool has = cg_ < c_hi;
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) w[rr][g] = has ? ld_stream4(rpt[rr] + cg_) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const int cg_ = c + 128 * g;
                if (cg_ < c_hi) {
                    const double2 z0 = *reinterpret_cast<const double2*>(&zs[cg_ - a0]);
                    const double2 z1 = *reinterpret_cast<const double2*>(&zs[cg_ - a0 + 2]);
                    const bool v0 = (cg_ >= c_lo), v1 = (cg_ + 1 >= c_lo) & (cg_ + 1 < c_hi);
                    const bool v2 = (cg_ + 2 >= c_lo) & (cg_ + 2 < c_hi), v3 = (cg_ + 3 >= c_lo) & (cg_ + 3 < c_hi);
#pragma unroll
                    for (int rr = 0; rr < 2; ++rr) {
                        double q0 = (v0 ? (double)w[rr][g].x : 0.0) * z0.x + (v1 ? (double)w[rr][g].y : 0.0) * z0.y;
                        double q1 = (v2 ? (double)w[rr][g].z : 0.0) * z1.x + (v3 ? (double)w[rr][g].w : 0.0) * z1.y;
                        acc[rr] += q0 + q1;
                    }
                }
            }
        }
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const double t = warp_sum(acc[rr]);
            const int i = rb + rr;
            if (lane == 0 && i < nr) {
                const double yn = S.sv[i] * invb * (t + zs[r0 + i + pad]);      // (w + I) z
                yout[i] = yn;
                pa = fma(yin[i] * invb, yn, pa);
            }
        }
    }
    return pa;
}

// ---- TMA-fed matvec (MODE 4 / 6): every warp owns a ring of RING_ST stages in shared memory; a stage holds up to
// RING_COLS columns of the warp's RING_R current rows (4 KB).  Lane 0 issues one bulk copy per row and stage
// (cp.async.bulk, completion counted on the stage's mbarrier); the warp waits for the stage, multiplies it with z
// from shared memory and hands the slot back.  Registers limit a register-staged form to 4 KB per warp in flight and
// only in bursts (issue 8 loads, wait, multiply: ncu put 32 % of that kernel's stall samples on the first use of the
// loaded registers); the ring keeps 4-8 KB per warp in flight all the time.  It takes the shared memory that held
// basis rows: Gram-Schmidt then reads the basis from L2, which costs less than the matvec gains.
// W does not change between steps, so the first stages of the NEXT matvec are fetched during Gram-Schmidt.
// The blocks come from k_gather_blocks_cur / k_zero_blocks, which zero the <= 3-column fringe of every block, and
// zs is zero there: no selects.  (Measured and dropped, DESIGN.md 5a: 1 KB stages x 4, register-staged loads with L2
// bulk prefetch, per-lane prefetch, L2 prefetch of the next matvec's stages, all loads of a stage hoisted.)
#ifndef ANCUTS_RING_ROWS
#define ANCUTS_RING_ROWS 4
#endif
constexpr int RING_ST = 2;
constexpr int RING_R = ANCUTS_RING_ROWS;                     // rows per stage.  4: every z value read from shared memory serves
                                                             // four rows (0.713 of the HBM peak against 0.684 with 2, profiles/r2i_lib_*)
constexpr int RING_COLS = 1024 / RING_R;                     // floats per row and stage (a stage is 4 KB)
constexpr int RING_STAGE_FLOATS = RING_R * RING_COLS;
constexpr int RING_WARP_FLOATS = RING_ST * RING_STAGE_FLOATS;
constexpr int RING_BYTES = CL_WARPS * RING_WARP_FLOATS * 4;      // 128 KB

struct RingGeom {
    int a0, width, nseg, npass, T;
};
__device__ __forceinline__ RingGeom ring_geom(const NodeView& v, int nr) {
    RingGeom q;
    const int warp = threadIdx.x >> 5;
    q.a0 = v.ro & ~3;
    q.width = (v.ro + v.n - q.a0 + 3) & ~3;            // columns fetched per row (multiple of 4)
    q.nseg = (q.width + RING_COLS - 1) / RING_COLS;
    q.npass = (warp * RING_R < nr) ? (nr - warp * RING_R + CL_WARPS * RING_R - 1) / (CL_WARPS * RING_R) : 0;
    q.T = q.npass * q.nseg;
    return q;
}
// lane 0: fetch stage (p, sg) of the matvec into the slot of global stage index gi
__device__ __forceinline__ void ring_issue(const NodeView& v, const RingGeom& q, int r0, int nr, int p, int sg,
                                           float* ring_w, uint64_t* bars_w, uint32_t gi) {
    const int warp = threadIdx.x >> 5;
    const int rb = warp * RING_R + p * (CL_WARPS * RING_R);
    const int c = sg * RING_COLS;
    const uint32_t bytes = (uint32_t)min(RING_COLS, q.width - c) * 4u;
    const uint32_t slot = gi % RING_ST;
    float* dst = ring_w + slot * RING_STAGE_FLOATS;
    uint64_t* bar = bars_w + slot;
    mbarrier_expect_tx(bar, (uint32_t)RING_R * bytes);
#pragma unroll
    for (int rr = 0; rr < RING_R; ++rr) {
        const float* src = v.W + (size_t)(v.ro + r0 + min(rb + rr, nr - 1)) * v.ld + q.a0 + c;
        bulk_copy_g2s(dst + rr * RING_COLS, src, bytes, bar);
    }
}
// the first min(RING_ST, T) stages of a matvec (before the first step and after every matvec)
__device__ __forceinline__ void ring_prologue(const NodeView& v, const RingGeom& q, int r0, int nr, float* ring_w,
                                              uint64_t* bars_w, uint32_t g) {
    if ((threadIdx.x & 31) == 0) {
        int p = 0, sg = 0;
        for (int t = 0; t < min(RING_ST, q.T); ++t) {
            ring_issue(v, q, r0, nr, p, sg, ring_w, bars_w, g + t);
            if (++sg == q.nseg) { sg = 0; ++p; }
        }
    }
}
__device__ __forceinline__ void ring_drain(const RingGeom& q, uint64_t* bars_w, uint32_t g) {
    for (int t = 0; t < min(RING_ST, q.T); ++t) mbarrier_wait(bars_w + ((g + t) % RING_ST), ((g + t) / RING_ST) & 1u);
}

// returns (lane 0) the warp's share of alpha = v . (M v), v_i = yin_i * invb
template <bool MIX>
__device__ __forceinline__ double cl_matvec_ring(ClusterShared& S, const double* zs, const double* __restrict__ yin,
                                                 double* __restrict__ yout, const NodeView& v, const RingGeom& q,
                                                 int r0, int nr, int pad, double invb, float* ring_w, uint64_t* bars_w,
                                                 uint32_t& g) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ip = 0, isg = 0;                               // next stage to issue = stage t + RING_ST
    for (int t = 0; t < min(RING_ST, q.T); ++t) if (++isg == q.nseg) { isg = 0; ++ip; }
    int t = 0;
    double pa = 0.0;
    for (int p = 0; p < q.npass; ++p) {
        double acc[RING_R], acb[RING_R];               // two FMA chains per row: one FP64 instruction per element
#pragma unroll
        for (int rr = 0; rr < RING_R; ++rr) { acc[rr] = 0.0; acb[rr] = 0.0; }
        for (int sg = 0; sg < q.nseg; ++sg, ++t) {
            const uint32_t slot = g % RING_ST;
            mbarrier_wait(bars_w + slot, (g / RING_ST) & 1u);
            const float* buf = ring_w + slot * RING_STAGE_FLOATS;
#pragma unroll
            for (int gq = 0; gq < RING_COLS / 128; ++gq) {
                const int cs = 128 * gq + 4 * lane;                // column inside the stage
                const int cofs = sg * RING_COLS + cs;              // column - a0
                if (cofs < q.width) {
                    const double2 z0 = *reinterpret_cast<const double2*>(&zs[cofs]);
                    const double2 z1 = *reinterpret_cast<const double2*>(&zs[cofs + 2]);
#pragma unroll
                    for (int rr = 0; rr < RING_R; ++rr) {
                        const float4 w = *reinterpret_cast<const float4*>(buf + rr * RING_COLS + cs);
                        acc[rr] = fma((double)w.x, z0.x, acc[rr]); acb[rr] = fma(widen_alt<MIX>(w.y), z0.y, acb[rr]);
                        acc[rr] = fma((double)w.z, z1.x, acc[rr]); acb[rr] = fma(widen_alt<MIX>(w.w), z1.y, acb[rr]);
                    }
                }
            }
            __syncwarp();
            ++g;
            if (lane == 0 && t + RING_ST < q.T) {
                ring_issue(v, q, r0, nr, ip, isg, ring_w, bars_w, g + RING_ST - 1);
                if (++isg == q.nseg) { isg = 0; ++ip; }
            }
        }
        const int rb = warp * RING_R + p * (CL_WARPS * RING_R);
        double tsum[RING_R];
#pragma unroll
        for (int rr = 0; rr < RING_R; ++rr) tsum[rr] = warp_sum(acc[rr] + acb[rr]);
        if (lane == 0) {
#pragma unroll
            for (int rr = 0; rr < RING_R; ++rr) {
                if (rb + rr < nr) {
                    const double y = S.sv[rb + rr] * invb * (tsum[rr] + zs[r0 + rb + rr + pad]);      // (w + I) z
                    yout[rb + rr] = y;
                    pa = fma(yin[rb + rr] * invb, y, pa);
                }
            }
        }
    }
    ring_prologue(v, q, r0, nr, ring_w, bars_w, g);
    return pa;
}

// ---- shared-memory sparse matvec (MODE 7, ANCUTS_OPT_MATVEC = 0, the default): W is 99.5 % zeros (27-66 stored entries per row
// against n <= 4096 columns), yet the dense form streams every block from HBM once per Lanczos step.  Here the CTA reads
// its row slice of the dense block ONCE at the start of the node (the entries per row were counted by k_degree on its own
// pass) and keeps it as CSR in shared memory (float32 value + uint16 column, rows in slice order, columns ascending) for
// all the steps: 4 n^2 bytes per node instead of k (4 n^2 + 8 n).  No ring, so the basis rows get the shared memory the ring took.  Same float64 products; the sum of a
// row is taken by four lanes over its entries round-robin and combined (l0 + l1) + (l2 + l3): a fixed order, but not
// the dense kernels' order, so alpha/beta differ from the dense form in the last bits (parity is against the oracle).
// A slice that does not fit (dense little nodes far above 100 entries per row) sends the node to the grid-wide path.
struct SparseSlice {
    const float* val; const unsigned short* col; const int* ptr;
    // col holds the BYTE offset of the entry's z value inside the CTA's z buffer, 8 * (column + pad) <= 8 * 4099: the matvec
    // adds it to the buffer's address and loads (two integer instructions per entry less than index -> address)
    __device__ __forceinline__ int column(int q, int pad) const { return (int)(col[q] >> 3) - pad; }
};
constexpr int SP_LANES = 4;

// Entries of TWO rows inside the block's aligned window, written by one warp: eight 128-bit loads in flight per lane
// (512 columns of both rows) before the first use.  Entries of a row keep the column order.  A row pointer may be NULL.
__device__ __forceinline__ void sp_fill_rows(const float* __restrict__ rowa, const float* __restrict__ rowb, int a0, int c_lo,
                                             int c_hi, int lane, float* val, unsigned short* col, int basea, int baseb,
                                             int pad) {
    for (int c0 = a0; c0 < c_hi; c0 += 512) {
        float4 w[2][4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int c = c0 + 128 * g + lane * 4;
            w[0][g] = (rowa && c < c_hi) ? ld_stream4(rowa + c) : make_float4(0.f, 0.f, 0.f, 0.f);
            w[1][g] = (rowb && c < c_hi) ? ld_stream4(rowb + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                if (c0 + 128 * g >= c_hi) break;                              // warp-uniform
                const int c = c0 + 128 * g + lane * 4;
                const float in[4] = {w[rr][g].x, w[rr][g].y, w[rr][g].z, w[rr][g].w};
                unsigned m = 0;
#pragma unroll
                for (int q = 0; q < 4; ++q) m |= (in[q] != 0.0f && c + q >= c_lo && c + q < c_hi) ? (1u << q) : 0u;
                const int cnt = __popc(m);
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
                int& base = rr ? baseb : basea;
                int pos = base + incl - cnt;
#pragma unroll
                for (int q = 0; q < 4; ++q) if (m & (1u << q)) { val[pos] = in[q]; col[pos] = (unsigned short)((c + q - c_lo + pad) << 3); ++pos; }
                base += __shfl_sync(0xffffffffu, incl, 31);
            }
        }
    }
    // rows start at multiples of four entries (the matvec loads four values and four columns at once): a row is filled up
    // with zeros that point at the first z slot
    if (lane < 3) {
        if (rowa && lane < ((4 - (basea & 3)) & 3)) { val[basea + lane] = 0.0f; col[basea + lane] = 0; }
        if (rowb && lane < ((4 - (baseb & 3)) & 3)) { val[baseb + lane] = 0.0f; col[baseb + lane] = 0; }
    }
}

// returns (every lane) the thread's share of alpha = v . (M v), v_i = yin_i * invb; the caller reduces it over the warp
__device__ __forceinline__ double cl_matvec_sparse(ClusterShared& S, const double* zs, const double* __restrict__ yin,
                                                   double* __restrict__ yout, const SparseSlice& sp, int r0, int nr, int pad,
                                                   double invb) {
    const int tid = threadIdx.x, sub = tid & (SP_LANES - 1);
    double pa = 0.0;
    for (int base = 0; base < nr; base += CL_THREADS / SP_LANES) {         // warp-uniform loop: the shuffles need all lanes
        const int i = base + tid / SP_LANES;
        double acc = 0.0;
        if (i < nr) {
            // four adjacent entries per lane and trip: one 128-bit load for the values, one 64-bit load for the columns (rows
            // start at multiples of four entries), two chains
            const int b = sp.ptr[i], e = sp.ptr[i + 1];
            const char* zb = reinterpret_cast<const char*>(zs);
            double acc1 = 0.0;
            for (int q = b + 4 * sub; q < e; q += 4 * SP_LANES) {
                const float4 w = *reinterpret_cast<const float4*>(sp.val + q);
                const uint2 cc = *reinterpret_cast<const uint2*>(sp.col + q);
                acc = fma((double)w.x, *reinterpret_cast<const double*>(zb + (cc.x & 0xffffu)), acc);
                acc1 = fma((double)w.y, *reinterpret_cast<const double*>(zb + (cc.x >> 16)), acc1);
                acc = fma((double)w.z, *reinterpret_cast<const double*>(zb + (cc.y & 0xffffu)), acc);
                acc1 = fma((double)w.w, *reinterpret_cast<const double*>(zb + (cc.y >> 16)), acc1);
            }
            acc += acc1;
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        if (sub == 0 && i < nr) {
            const double y = S.sv[i] * invb * (acc + zs[r0 + i + pad]);      // (w + I) z
            yout[i] = y;
            pa = fma(yin[i] * invb, y, pa);
        }
    }
    return pa;
}

// ---- fused cut (segment calls, nodes whose CSR slice is in shared memory): what k_ev_final, k_bucket, k_scan, k_decide,
// k_sides and, for the next rebuild, k_cc_union do in six launches and two dense passes over the node's block
// (get_min_ncut / ncut_cost / cut_cost, normalized_cut.py:4-34, the decision :56 and the component split of DESIGN.md 4.2)
// happens here from the CSR slice: the Ritz vector of the whole node was pushed into every CTA's z buffer, every CTA derives
// sign, thresholds, buckets and volumes redundantly (identical values), the ten cut weights come from the slice's stored
// entries with the same fixed-point integer atomics as k_scan (identical sums), and after the decision the entries whose
// end points share a side that goes on are joined in the union-find forest.  The cut weights are bit-equal to the separate
// kernels'; the volumes are summed in another (fixed) order, so costs may differ in the last bits.
template <int C>
__device__ void cl_fused_cut(cg::cluster_group& cl, ClusterShared& S, const Eng& e, const double* zs, const SparseSlice& sp,
                             const NodeView& v, int a, int rank, int r0, int nr, int pad, int steps, const double* th) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = v.n;
    const int r = e.a_rid[a];
    // statistics of the Ritz vector in rank order (S.spart of every CTA is complete: the caller synchronised the cluster)
    double ts = 0.0, tmn = 1e300, tmx = -1e300, tq = 0.0;
#pragma unroll
    for (int q = 0; q < C; ++q) {
        const double* np_ = (C > 1) ? cl.map_shared_rank(&S.spart[0], q) : &S.spart[0];
        ts += np_[0]; tmn = fmin(tmn, np_[1]); tmx = fmax(tmx, np_[2]); tq += np_[3];
    }
    // k_ev_final: unit norm, sign sum(ev) >= 0, np.allclose(min, max), np.linspace(endpoint=False)
    const double scale = 1.0 / sqrt(tq);
    const double sg = (ts < 0.0) ? -scale : scale;
    double mn = tmn, mx = tmx;
    if (ts < 0.0) { const double t = mn; mn = -mx; mx = -t; }
    mn *= scale; mx *= scale;
    const bool nocut = fabs(mn - mx) <= 1e-8 + 1e-5 * fabs(mx);
    const double step = (mx - mn) / (double)NCUT;
    double thr[NCUT];
#pragma unroll
    for (int q = 0; q < NCUT; ++q) thr[q] = __dadd_rn(__dmul_rn((double)q, step), mn);
    // k_bucket: bucket of every point of the node (all CTAs), signed unit-norm ev and bucket of the slice to global memory
    unsigned char* bk = reinterpret_cast<unsigned char*>(&S.ysl[0][0]);       // 8 KB: n <= 4096 buckets
    double volp[NB];
    int cntp[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) { volp[b] = 0.0; cntp[b] = 0; }
    for (int j = tid; j < n; j += CL_THREADS) {
        const double x = zs[j + pad] * sg;
        int b = 0;
#pragma unroll
        for (int q = 0; q < NCUT; ++q) b += (x > thr[q]) ? 1 : 0;
        bk[j] = (unsigned char)b;
        const double dg = e.deg[v.start + j];
#pragma unroll
        for (int b2 = 0; b2 < NB; ++b2) { volp[b2] += (b == b2) ? dg : 0.0; cntp[b2] += (b == b2) ? 1 : 0; }
        if (j >= r0 && j < r0 + nr) { e.ev[v.start + j] = x; e.bucket[v.start + j] = (uint8_t)b; }
    }
    // block reduction of the 11 volumes and counts in a fixed order: S.du = 16 x 11 doubles, S.cnts = 16 x 11 ints
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        const double vs = warp_sum(volp[b]);
        int cs = cntp[b];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cs += __shfl_xor_sync(0xffffffffu, cs, o);
        if (lane == 0) { S.du[warp * NB + b] = vs; S.cnts[warp * NB + b] = cs; }
    }
    // the difference array is summed per warp first (64-bit shared-memory atomics of 512 threads on eleven addresses were
    // 2.7 % of the kernel's stall samples); S.hpart is free after the last Gram-Schmidt exchange: 16 x 12 counters
    unsigned long long* wdiff = reinterpret_cast<unsigned long long*>(&S.hpart[0]);
    static_assert(CL_WARPS * (NB + 1) <= CL_KS, "per-warp difference arrays alias S.hpart");
    static_assert(CL_WARPS * NB <= 2 * CL_SHIFTS, "per-warp counts fit S.cnts");
    if (tid < CL_WARPS * (NB + 1)) wdiff[tid] = 0ull;
    __syncthreads();
    if (tid < NB) {
        double vs = 0.0; int cs = 0;
        for (int w = 0; w < CL_WARPS; ++w) { vs += S.du[w * NB + tid]; cs += S.cnts[w * NB + tid]; }
        S.fvol[tid] = vs; S.fcnt[tid] = cs;
    }
    __syncthreads();
    double vtot = 0.0;
#pragma unroll
    for (int b = 0; b < NB; ++b) vtot += S.fvol[b];
    const int shift = fix_shift(vtot);
    const double fscale = ldexp(1.0, shift);
    // k_scan on the CSR slice: every stored entry of the upper triangle adds its weight to the difference array
    if (!nocut) {
        for (int base = 0; base < nr; base += CL_THREADS / SP_LANES) {
            const int i = base + tid / SP_LANES;
            if (i < nr) {
                const int gi = r0 + i, bi = bk[gi];
                for (int q = sp.ptr[i] + (tid & (SP_LANES - 1)); q < sp.ptr[i + 1]; q += SP_LANES) {
                    const int c = sp.column(q, pad);
                    if (c > gi) {
                        const int bj = bk[c];
                        if (bj != bi) {
                            const long long w = __double2ll_rn((double)sp.val[q] * fscale);
                            atomicAdd(&wdiff[warp * (NB + 1) + min(bi, bj)], (unsigned long long)w);
                            atomicAdd(&wdiff[warp * (NB + 1) + max(bi, bj)], (unsigned long long)(-w));
                        }
                    }
                }
            }
        }
    }
    __syncthreads();
    if (tid <= NB) {
        unsigned long long t = 0ull;
        for (int w = 0; w < CL_WARPS; ++w) t += wdiff[w * (NB + 1) + tid];
        S.fdiff[tid] = t;
    }
    cl_sync<C>(cl);
    if (tid <= NB) {
        unsigned long long t = 0ull;
#pragma unroll
        for (int q = 0; q < C; ++q) t += (C > 1) ? cl.map_shared_rank(&S.fdiff[0], q)[tid] : S.fdiff[tid];
        S.fsum[tid] = t;
    }
    __syncthreads();
    // k_decide (every CTA, identical inputs): N-cut value of the ten cuts, first strictly smallest, mcut < T, side sizes
    if (tid == 0) {
        int best = -1;
        double bestc = INFINITY;
        double costs[NCUT];
        if (!nocut) {
            const double unfix = ldexp(1.0, -shift);
            long long run = 0;
            for (int q = 0; q < NCUT; ++q) {
                run += (long long)S.fsum[q];
                const double cut = (double)run * unfix;
                double assoc_b = 0.0, assoc_a = 0.0;
                for (int b = 0; b <= q; ++b) assoc_b += S.fvol[b];
                for (int b = q + 1; b < NB; ++b) assoc_a += S.fvol[b];
                const double cost = (cut / assoc_a) + (cut / assoc_b);
                costs[q] = cost;
                if (cost < bestc) { bestc = cost; best = q; }
            }
        } else {
            for (int q = 0; q < NCUT; ++q) costs[q] = INFINITY;
        }
        const bool split = (best >= 0) && (bestc < e.T);
        int n_a = 0;
        if (best >= 0) for (int b = best + 1; b < NB; ++b) n_a += S.fcnt[b];
        const int n_b = n - n_a;
        const double no = (double)e.c_norig[v.chunk] + 1e-8;
        const int p0 = (split && n_a > 2 && (double)n_a / no > CHILD_SPLIT_LIM) ? 1 : 0;
        const int p1 = (split && n_b > 2 && (double)n_b / no > CHILD_SPLIT_LIM) ? 1 : 0;
        S.fdec[0] = best; S.fdec[1] = split ? 1 : 0; S.fdec[2] = p0; S.fdec[3] = p1;
        if (rank == 0) {
            e.a_bestk[a] = best;
            e.a_mcut[a] = bestc;
            for (int q = 0; q < NCUT; ++q) e.a_costs[a * NCUT + q] = costs[q];
            if (split) {
                e.r_pass[2 * r + 0] = p0 ? 2 : 0;            // 2 = passes and its components are already joined (k_cc_union skips it)
                e.r_pass[2 * r + 1] = p1 ? 2 : 0;
                e.r_status[r] = ST_SPLIT;
                const int s_ = atomicAdd(&e.ctr[5], 1);
                e.split_ids[s_] = r;
                atomicMax(&e.ctr[7], n);
            } else {
                e.r_status[r] = ST_LEAF;
            }
            if (e.stats != nullptr) {
                const int s_ = atomicAdd(&e.ctr[6], 1);
                if (s_ < e.stats_cap) {
                    ancuts_node_stat st;
                    st.chunk = v.chunk; st.n = n; st.steps = steps; st.converged = 1;
                    st.best_k = best; st.split = split ? 1 : 0; st.level = e.r_level[r]; st.n_side = n_a;
                    st.lambda2 = 1.0 - th[0]; st.mcut = bestc;
                    e.stats[s_] = st;
                }
            }
            e.a_fused[a] = 1;
            atomicAdd(&e.ctr[17], 1);
        }
    }
    __syncthreads();
    if (!S.fdec[1]) return;
    // k_sides + k_cc_union on the slice: side 0 = mask side (ev > t); entries inside a side that goes on are joined
    const int best = S.fdec[0];
    for (int i = tid; i < nr; i += CL_THREADS) e.side[v.start + r0 + i] = (bk[r0 + i] > best) ? 0 : 1;
    for (int base = 0; base < nr; base += CL_THREADS / SP_LANES) {
        const int i = base + tid / SP_LANES;
        if (i < nr) {
            const int gi = r0 + i;
            const int si = (bk[gi] > best) ? 0 : 1;
            if (S.fdec[2 + si]) {
                for (int q = sp.ptr[i] + (tid & (SP_LANES - 1)); q < sp.ptr[i + 1]; q += SP_LANES) {
                    const int c = sp.column(q, pad);
                    if (c > gi && ((bk[c] > best) ? 0 : 1) == si) uf_union(e.parent, v.start + gi, v.start + c);
                }
            }
        }
    }
}

// grid: count * C CTAs, cluster (C,1,1); ids[cluster index] = active slot.
// MODE 0: guarded register-staged matvec (caller's W read in place); 4: TMA ring; 6: TMA ring + integer widening of
// every second element (weights in {0} U [2^-126, 2): the library's own affinities); 7: row slice as CSR in shared memory.
template <int C, int MODE>
__global__ void __launch_bounds__(CL_THREADS, 1)
k_lanczos_cluster(Eng e, int cur, const int* __restrict__ ids, int dyn_doubles) {
    extern __shared__ __align__(16) double zs[];   // z = S v for the whole node on the 16-byte window of W's columns;
                                                   // behind it: the warps' W rings, then the first rows of the basis,
                                                   // restricted to this CTA's slice
    __shared__ ClusterShared S;
    cg::cluster_group cl = cg::this_cluster();
    const int rank = (C > 1) ? (int)cl.block_rank() : 0;
    const int a = ids[blockIdx.x / C];
    const NodeView v = node_view(e, e.a_rid[a], cur);
    const int n = v.n;
    const int rp = (n + C - 1) / C;
    const int r0 = min(n, rank * rp), r1 = min(n, r0 + rp);
    const int nr = r1 - r0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t P = (size_t)e.P;
    const int g0 = v.start + r0;                       // global position of the slice
    const int pad = v.ro & 3;                          // zs[j + pad] <-> column v.ro + j
    constexpr bool RING = (MODE == 4 || MODE == 6);
    constexpr bool SP = (MODE == 7);
    const int nz = (n + 8 + 3) & ~3;                   // doubles used by zs
    SparseSlice sp;
    sp.val = nullptr; sp.col = nullptr; sp.ptr = nullptr;
    int sp_doubles = 0;
    if (SP) {
        // ---- build the CSR slice: entries per row (counted by k_degree on its pass over the block), scan, fill ----
        const int c_lo = v.ro, c_hi = v.ro + n, a0 = c_lo & ~3;
        __shared__ int sp_wtot[CL_WARPS + 1];
        const int stored = (tid < nr) ? e.rownnz[g0 + tid] : 0;    // stored entries per row, counted by k_degree
        const int mine = (stored + 3) & ~3;                        // rows start at multiples of four entries (cl_matvec_sparse)
        const int fill = __syncthreads_count((mine - stored) & 1) + 2 * __syncthreads_count((mine - stored) & 2);
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) sp_wtot[warp] = incl;
        __syncthreads();
        if (tid == 0) {
            int run = 0;
            for (int w = 0; w < CL_WARPS; ++w) { int t = sp_wtot[w]; sp_wtot[w] = run; run += t; }
            sp_wtot[CL_WARPS] = run;
        }
        __syncthreads();
        const int total = sp_wtot[CL_WARPS];
        int* ptr = reinterpret_cast<int*>(zs + nz);
        const int ptr_d = (((nr + 1 + 1) / 2) + 1) & ~1;                     // doubles; even: the values start 16-byte aligned
        const int val_d = (total + 1) / 2, col_d = (total + 3) / 4;
        sp_doubles = ptr_d + val_d + col_d;
        double misfit = (nz + sp_doubles > dyn_doubles) ? 1.0 : 0.0;
        if (C > 1) {                                                         // the whole cluster takes the same decision
            if (tid == 0) S.npart[1] = misfit;
            cl.sync();
            misfit = 0.0;
#pragma unroll
            for (int r = 0; r < C; ++r) misfit += cl.map_shared_rank(&S.npart[0], r)[1];
            cl.sync();                                                       // peers have read the flag: the slot is free again
        }
        if (misfit != 0.0) {
            // a slice that does not fit (dense little graphs far above 100 entries per row, 512-row slices of the largest
            // nodes): this node streams W with the register-staged matvec instead, in the same kernel
            sp_doubles = 0;
        } else {
            float* val = reinterpret_cast<float*>(zs + nz + ptr_d);
            unsigned short* col = reinterpret_cast<unsigned short*>(zs + nz + ptr_d + val_d);
            if (tid < nr) ptr[tid] = sp_wtot[warp] + incl - mine;
            if (tid == 0) ptr[nr] = total;
            __syncthreads();
            if (e.node_csr) {
                // the node's CSR rows hold exactly the entries sp_fill_rows keeps, in the same order: copy them
                for (int i = warp; i < nr; i += CL_WARPS) {
                    const int b = e.csr_ptr[g0 + i], cnt = e.csr_ptr[g0 + i + 1] - b, o = ptr[i];
                    for (int k = lane; k < cnt; k += 32) {
                        val[o + k] = e.csr_val[b + k];
                        col[o + k] = (unsigned short)((e.csr_col[b + k] + pad) << 3);
                    }
                    if (lane < ((4 - (cnt & 3)) & 3)) { val[o + cnt + lane] = 0.0f; col[o + cnt + lane] = 0; }
                }
            } else {
                for (int i = warp; i < nr; i += 2 * CL_WARPS) {
                    const int i2 = i + CL_WARPS;
                    sp_fill_rows(v.W + (size_t)(v.ro + r0 + i) * v.ld, i2 < nr ? v.W + (size_t)(v.ro + r0 + i2) * v.ld : nullptr,
                                 a0, c_lo, c_hi, lane, val, col, ptr[i], i2 < nr ? ptr[i2] : 0, pad);
                }
            }
            sp.val = val; sp.col = col; sp.ptr = ptr;
            if (tid == 0) S.sp_nnz = total - fill;       // accounting only: shared memory, not a register across the steps
            __syncthreads();
        }
    }
    SliceBasis B;
    {
        B.nrp = (max(nr, 1) + 3) & ~3;
        const int nfront = RING ? RING_BYTES / 8 : sp_doubles;              // the warps' W rings or the CSR slice sit in front
        B.smem = zs + nz + nfront;
        B.rows_s = max(0, (dyn_doubles - nz - nfront) / B.nrp);
        B.glob = e.V + g0;
        B.P = P;
    }
    const int kcap = min(min(CL_KMAX, e.kmax), n - 1);
    __shared__ uint64_t ring_bar[CL_WARPS * RING_ST];
    float* ring_w = reinterpret_cast<float*>(zs + nz) + (size_t)warp * RING_WARP_FLOATS;
    uint64_t* bars_w = ring_bar + warp * RING_ST;
    const RingGeom rq = ring_geom(v, nr);
    uint32_t ring_g = 0;                               // stages consumed by this warp so far
    if (RING) {
        if (lane == 0) {
            for (int i = 0; i < RING_ST; ++i) mbarrier_init(bars_w + i, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        ring_prologue(v, rq, r0, nr, ring_w, bars_w, ring_g);     // W is ready: start streaming during the set-up
    }
    // ---- init (every CTA redundantly: bit-identical scalars, no exchange needed) ----
    double s = 0.0;
    for (int i = tid; i < n; i += CL_THREADS) s += e.deg[v.start + i];
    const double vol = block_sum_512(s, S.red);
    const double ivol = 1.0 / sqrt(vol);
    s = 0.0;
    const StartVec sv0(e, v.chunk, v.start);
    for (int i = tid; i < n; i += CL_THREADS) s += sqrt(e.deg[v.start + i]) * ivol * sv0.at(v.start + i, i);
    const double dot = block_sum_512(s, S.red);
    s = 0.0;
    for (int i = tid; i < n + 8; i += CL_THREADS) {
        int j = i - pad;
        double z = 0.0;
        if (j >= 0 && j < n) {
            double u = sqrt(e.deg[v.start + j]) * ivol;
            double x = sv0.at(v.start + j, j) - dot * u;
            z = e.sinv[v.start + j] * x;
            s += x * x;
        }
        zs[i] = z;
    }
    double bprev = sqrt(block_sum_512(s, S.red));
    double* yc = S.ysl[0];                               // current (unnormalised) Lanczos vector of the slice
    double* yn = S.ysl[1];                               // matvec result, orthogonalised in place
    for (int i = tid; i < nr; i += CL_THREADS) {
        int j = r0 + i;
        double u = sqrt(e.deg[v.start + j]) * ivol;
        B.put(0, i, u);                                  // basis row 0 = u1
        yc[i] = sv0.at(v.start + j, j) - dot * u;
        S.sv[i] = e.sinv[v.start + j];
    }
    __syncthreads();
    if (C > 1) {                                         // the mbarriers of the step exchanges, initialised before any peer pushes
        if (tid == 0) {
            mbarrier_init(&S.bar_a, 1);
            mbarrier_init(&S.bar_n, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        cl.sync();
    }

    float om_c = (tid == 0) ? 1.0f : 0.0f, om_p = 0.0f;  // omega_{k, tid}, omega_{k-1, tid}; omega_{0,0} = v_0 . v_0 = 1
    if (tid == 0) S.om[0] = 1.0f;
    double om_u = 0x1p-52, om_u_prev = 0x1p-52;          // omega of u1 against the two newest Lanczos vectors
    bool reorth_next = false;                            // the step after a full pass takes one too
    int nfull = 0;                                       // steps that took the full pass (accounting)
    int k = 0;
    int conv = 0;
    double th[2] = {0.0, 0.0};
    const bool adapt = e.check_adapt != 0;
    if (tid == 0) { S.prev_res = 1.0; S.prev_k = 0; S.next_check = adapt ? CL_CHECK_FIRST : e.check_every; }
    // optional phase clock (debug): cycles of thread 0 of rank 0 between the block-wide syncs that end each phase
    // (a barrier's wait is charged to the phase AFTER it: BAR.SYNC does not block at issue)
    const bool prof = (e.dbg != nullptr) && tid == 0 && rank == 0;
    long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tlast = prof ? clock64() : 0;
#define CL_PHASE(i) do { if (prof) { long long t_ = clock64(); tph[i] += t_ - tlast; tlast = t_; } } while (0)
    // a guard build's wait gave up (cl_wait): count it and leave the step loop
#define CL_EXCHANGE_FAILED() do { if (tid == 0) atomicAdd(&e.ctr[19], 1); } while (0)
    while (true) {
        const double invb = 1.0 / bprev;
        // basis row k+1 = current vector (slice).  The matvec below only reads yc and writes yn: no barrier in between.
        double* vk = B.row(k + 1);
        for (int i = tid; i < nr; i += CL_THREADS) vk[i] = yc[i] * invb;
        CL_PHASE(0);
        // ---- matvec of the slice; alpha = v_k . (M v_k) rides on its epilogue ----
        double pa;
        if (RING) pa = cl_matvec_ring<MODE == 6>(S, zs, yc, yn, v, rq, r0, nr, pad, invb, ring_w, bars_w, ring_g);
        else if (SP && sp.ptr) pa = warp_sum(cl_matvec_sparse(S, zs, yc, yn, sp, r0, nr, pad, invb));
        else pa = cl_matvec_guard(S, zs, yc, yn, v, r0, nr, pad, invb);
        if (lane == 0) S.wred[warp] = pa;
        __syncthreads();
        CL_PHASE(1);
        double a1 = 0.0;
#pragma unroll
        for (int i = 0; i < CL_WARPS; ++i) a1 += S.wred[i];
        if (C > 1 && !cl_exchange<C>(S.apart, &S.bar_a, (uint32_t)k & 1u, 8u * C, rank, a1)) { CL_EXCHANGE_FAILED(); break; }
        // ---- three-term recurrence y = M v_k - alpha v_k - beta v_{k-1}; its squared norm and z = S y for the next matvec
        //      ride on the same pass.  z: every CTA PUSHES its slice into the z vector of all CTAs of the cluster through
        //      distributed shared memory (every matvec of this step has ended before its alpha partial was pushed, so the
        //      peers' z is free; the stores complete the phase of the norm exchange below). ----
        double q = 0.0;
        {
            const double bk = (k > 0) ? S.beta[k - 1] : 0.0;
            // own elements of v_k and v_{k-1} (u1 when k = 0: bk = 0)
            const double* vp = B.row(k);
            for (int i = tid; i < nr; i += CL_THREADS) {
                const double y = (yn[i] - a1 * vk[i]) - bk * vp[i];
                yn[i] = y;
                q = fma(y, y, q);
                cl_put_z<C>(S, zs, rank, r0 + i + pad, S.sv[i] * y);
            }
        }
        q = cl_block_sum1(S, q);
        CL_PHASE(2);
        double beta = q;
        if (!cl_norm_exchange<C>(S, (uint32_t)(k + nfull) & 1u, n, nr, rank, beta)) { CL_EXCHANGE_FAILED(); break; }
        // ---- partial re-orthogonalisation (Simon 1984, as in PROPACK): the omega recurrence estimates v_{k+1} . v_i of
        //      the new vector against every Lanczos vector from alpha and beta alone, O(k) per step.  The full classical
        //      Gram-Schmidt pass against u1 and the whole basis runs only when an estimate passes sqrt(eps), and on the step
        //      after one (the pair v_{k+1}, v_{k+2} is made orthogonal); a pass resets the estimates to eps.  u1 = D^1/2 1 is
        //      an exact eigenvector of M (eigenvalue 1), so its own estimate follows
        //      beta_k w' = (1 - alpha_k) w_k - beta_{k-1} w_{k-1}, and it too is removed only by the full passes.
        //      Every CTA evaluates the recurrence from its bit-identical alpha / beta in the same order, so the decision is
        //      the same in the whole cluster without an exchange.  numpy model (tests/test_partial_reorth.py): the same
        //      steps and the same Ritz vector to 1e-9 as the pass on every step, with the pass on ~5 % of the steps. ----
        {
            constexpr double EPS = 0x1p-52;
            const double bn = beta;
            const double bkm = (k > 0) ? S.beta[k - 1] : 0.0;
            // thread i: omega_{k+1, i} from omega_{k, i-1 .. i+1} (S.om, own entry om_c) and omega_{k-1, i} (om_p)
            float om_new = 0.0f;
            bool hi = false;
            if (tid < k) {                               // one estimate per thread (k <= CL_KMAX < CL_THREADS)
                const double bi = S.beta[tid];
                double t = bi * (double)S.om[tid + 1] + (S.alpha[tid] - a1) * (double)om_c - bkm * (double)om_p;
                if (tid > 0) t += S.beta[tid - 1] * (double)S.om[tid - 1];
                const double noise = 0.6 * EPS * (fabs(bi) + bn);       // rounding of the step's products, as in the model
                t = (t + (t < 0.0 ? -noise : noise)) / bn;
                om_new = (float)t;
                hi = !(fabs(t) <= CL_REORTH_TOL);         // NaN (beta = 0 at a breakdown) takes the pass too
            } else if (tid == k) {
                om_new = (float)(EPS * 0.5 * (double)n);
            } else if (tid == k + 1) {
                om_new = 1.0f;
            }
            {
                double t = (1.0 - a1) * om_u - bkm * om_u_prev;
                t = (t + (t < 0.0 ? -2.0 * EPS * bn : 2.0 * EPS * bn)) / bn;
                om_u_prev = om_u;
                om_u = t;
            }
            const bool full = __syncthreads_or(hi) || reorth_next || !(fabs(om_u) <= CL_REORTH_TOL);
            // every thread has read S.om (the barrier above): the new row replaces it
            if (full) {
                if (tid <= k) om_new = (float)EPS;
                om_u = EPS;
            }
            om_p = om_c;
            om_c = om_new;
            if (tid <= k + 1) S.om[tid] = om_new;
            CL_PHASE(6);
            if (full) {
                reorth_next = !reorth_next;
                nfull += 1;
                // ---- the full pass on y: ONE classical Gram-Schmidt pass against u1 and every Lanczos vector (rows
                //      0 .. k+1).  After the three-term part it only removes small components, so one pass is as good as
                //      two (test_design_choices.py).  The pass leaves alpha v_k to the three-term part: a pass that also
                //      had to remove it loses orthogonality within dozens of steps; its own coefficient corrects alpha. ----
                const int rows = k + 2;
                cl_partial_dots(S, yn, B, rows, nr);      // yn is complete: the barrier of the norm sum ordered its stores
                cl_sync<C>(cl);
                const double* hsrc = S.hpart;             // one CTA per node: its partial dots are the coefficients
                if (C > 1) { cl_reduce_h<C>(cl, S, rows, 1); hsrc = S.hs; }
                a1 += hsrc[rows - 1];
                CL_PHASE(4);
                q = cl_update_norm(hsrc, yn, B, rows, nr);
                cl_push_z<C>(S, zs, rank, yn, r0, nr, pad);
                beta = cl_block_sum1(S, q);
                // a bar_n phase of its own (nfull already counts this pass): z and the norm arrive as after the three-term pass
                if (!cl_norm_exchange<C>(S, (uint32_t)(k + nfull) & 1u, n, nr, rank, beta)) { CL_EXCHANGE_FAILED(); break; }
                CL_PHASE(5);
            }
        }
        if (tid == 0) { S.alpha[k] = a1; S.beta[k] = beta; }
        bprev = beta;
        k += 1;
        { double* t_ = yc; yc = yn; yn = t_; }
        // no barrier here: what the next step reads of this one -- yc, z, alpha / beta, omega -- is separated from its writes
        // by the block barriers of the norm sum and the decision above or by the one that ends the next matvec (S.wred /
        // S.wred2 are separate arrays); the peers' z arrived with the bar_n phase
        const bool breakdown = beta < 1e-13;
        if (breakdown || k >= kcap || k == S.next_check) {
            __syncthreads();                 // alpha[k-1], beta[k-1] of thread 0
            cluster_tridiag_eigs(S, k, th);
            if (prof) { tph[3] += S.tmark - tlast; tlast = S.tmark; }     // slot 3: multisection part of the check
            const double res = cluster_tridiag_vec(S, k, th[0]);
            double gap = fmax(th[0] - th[1], 1e-300);
            bool c1 = (k >= n - 1) || breakdown || (res <= e.tol * gap);
            if (c1) { conv = 1; break; }
            if (k >= kcap) break;
            if (tid == 0) {                  // every CTA of the cluster holds the same alpha/beta: identical schedules
                int adv = e.check_every;
                if (adapt) {
                    adv = CL_CHECK_HI;
                    const double pr = S.prev_res;
                    if (res < pr && res > 0.0) {
                        const double rate = log(res / pr) / (double)(k - S.prev_k);          // < 0
                        const double need = CL_CHECK_SAFETY * log(e.tol * gap / res) / rate;   // > 0: not converged yet
                        adv = (int)fmin((double)CL_CHECK_HI, fmax((double)CL_CHECK_LO, ceil(need)));
                    }
                    S.prev_res = res;
                    S.prev_k = k;
                }
                S.next_check = k + adv;
            }
            __syncthreads();
            CL_PHASE(7);
        }
    }
    CL_PHASE(7);
    if (RING) ring_drain(rq, bars_w, ring_g);     // stages fetched ahead for a step that will not run
    if (prof) {
        const int ci = (C == 1) ? 0 : (C == 2) ? 1 : (C == 4) ? 2 : 3;
        for (int i = 0; i < 8; ++i) atomicAdd(&e.dbg[ci * 8 + i], (unsigned long long)tph[i]);
    }
#undef CL_PHASE
#undef CL_EXCHANGE_FAILED
    if (rank == 0 && tid == 0) {             // share of the steps that took the full Gram-Schmidt pass
        atomicAdd(&e.acct[SG_CL_STEPS], (unsigned long long)k);
        atomicAdd(&e.acct[SG_CL_FULL], (unsigned long long)nfull);
    }
    // ---- Ritz vector of the slice, statistics for the cut kernels ----
    if (conv) {
        const bool fuse = SP && sp.ptr != nullptr && e.fuse_cut != 0;
        double xs = 0.0, xq = 0.0, xmn = 1e300, xmx = -1e300;
        for (int i = tid; i < nr; i += CL_THREADS) {
            double x = 0.0;
            int j = 0;
            {   // basis rows 1 .. k: shared-memory part, then global part (stepping pointers, same order of the sum)
                const double* p = B.smem + (size_t)B.nrp + i;
                for (; j < k && j + 1 < B.rows_s; ++j) { x += S.yv[j] * *p; p += B.nrp; }
                p = B.glob + (size_t)(j + 1) * B.P + i;
                for (; j < k; ++j) { x += S.yv[j] * *p; p += B.P; }
            }
            e.ev[g0 + i] = x;
            xs += x; xq += x * x; xmn = fmin(xmn, x); xmx = fmax(xmx, x);
            if (fuse) {                               // the whole node's Ritz vector into every CTA's z buffer (no matvec follows)
                if (C > 1) {
#pragma unroll
                    for (int q = 0; q < C; ++q) cl.map_shared_rank(zs, q)[r0 + i + pad] = x;
                } else {
                    zs[i + pad] = x;
                }
            }
        }
        double sm_ = block_sum_512(xs, S.red);
        double sq = block_sum_512(xq, S.red);
        double mn = block_min_512(xmn, S.red);
        double mx = -block_min_512(-xmx, S.red);
        if (tid == 0) { S.spart[0] = sm_; S.spart[1] = mn; S.spart[2] = mx; S.spart[3] = sq; }
        cl_sync<C>(cl);
        if (rank == 0 && tid == 0) {
            double ts = 0.0, tmn = 1e300, tmx = -1e300, tq = 0.0;
            for (int r = 0; r < C; ++r) {
                const double* np_ = (C > 1) ? cl.map_shared_rank(&S.spart[0], r) : &S.spart[0];
                ts += np_[0]; tmn = fmin(tmn, np_[1]); tmx = fmax(tmx, np_[2]); tq += np_[3];
            }
            const int s0 = e.a_slot0[a], nch = e.a_nch[a];
            double* o = e.p_stat + (size_t)s0 * 4;
            o[0] = ts; o[1] = tmn; o[2] = tmx; o[3] = tq;
            for (int c = 1; c < nch; ++c) { double* oc = e.p_stat + (size_t)(s0 + c) * 4; oc[0] = 0.0; oc[1] = 1e300; oc[2] = -1e300; oc[3] = 0.0; }
            e.a_k[a] = k;
            e.a_kcap[a] = kcap;
            e.a_conv[a] = 1;
            e.a_theta[2 * a] = th[0];
            e.a_theta[2 * a + 1] = th[1];
            e.a_done[a] = DONE_YES;
            e.a_path[a] = 0;                    // Ritz vector and statistics are already in place
            if (!SP || !sp.ptr) atomicAdd(&e.acct[SG_MATVEC], (unsigned long long)k * (4ull * n * n + 8ull * n));
        }
        if (SP && sp.ptr && tid == 0) {      // what this form really moves: the slice once from HBM, then k sweeps over its entries
            atomicAdd(&e.acct[SG_MATVEC], 4ull * (unsigned long long)nr * n);
            atomicAdd(&e.acct[SG_SPARSE_STEPS], (unsigned long long)k * (unsigned long long)S.sp_nnz);
            atomicAdd(&e.acct[SG_SPARSE_NNZ], (unsigned long long)S.sp_nnz);
        }
        if (fuse) cl_fused_cut<C>(cl, S, e, zs, sp, v, a, rank, r0, nr, pad, k, th);
        else if (rank == 0 && tid == 0 && e.unfused) e.unfused[atomicAdd(&e.ctr[18], 1)] = a;     // the cut kernels take it
    } else if (rank == 0 && tid == 0) {
        e.a_done[a] = DONE_NO;                  // left for the multi-launch path (more steps)
        e.a_path[a] = 1;
        atomicAdd(&e.ctr[4], 1);
        if (e.unfused) e.unfused[atomicAdd(&e.ctr[18], 1)] = a;
    }
    cl_sync<C>(cl);                             // peers may still be reading this CTA's shared memory
}

}  // namespace ancuts
