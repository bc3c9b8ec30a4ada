// kernels_graph.cuh — affinity (exact CUDA-core tile kernel), degrees, connected components,
// range-table rebuild and block gather.  Reference lines are cited per kernel.
#pragma once
#include "common.cuh"

namespace ancuts {

// size bin of a node for the persistent Lanczos kernel (kernels_cluster.cuh); -1 = too large.
// The host maps bins to cluster sizes per level (engine.cu: latency mapping when the level fits one
// wave of CTAs, throughput mapping with fewer CTAs per node otherwise).
__host__ __device__ inline int cluster_class(int n) {
    if (n <= 320) return 0;
    if (n <= 512) return 1;
    if (n <= 640) return 2;
    if (n <= 1024) return 3;
    if (n <= 2048) return 4;
    if (n <= 4096) return 5;
    return -1;
}

struct NodeView {
    int start;      // global position of the first point
    int n;
    int chunk;
    int ro;         // chunk-local offset = row/column of the block inside the chunk's matrix
    int ld;
    const float* W; // chunk matrix in the current buffer
};

__device__ __forceinline__ NodeView node_view(const Eng& e, int r, int cur) {
    NodeView v;
    v.start = e.r_start[r];
    v.n = e.r_n[r];
    v.chunk = e.r_chunk[r];
    v.ro = v.start - e.c_base[v.chunk];
    v.ld = e.c_ld[v.chunk];
    v.W = cur ? e.c_W1[v.chunk] : e.c_W0[v.chunk];
    return v;
}

// ---------------------------------------------------------------------------------------------
// Stage 1 (exact): A_ij = [sd_ij <= prox] * exp(-(alpha*sd_ij + theta*td_ij + gamma*dd_ij))
//   ncuts_utils.py:60-66 (spatial, float64 compare), :135-149 (TARL, zero rows neutralised),
//   :125-133 (DINOv2, zero rows NOT neutralised), :151-156 (product).
// One 64x64 tile per CTA.  Pass 1 evaluates the float64 spatial test for every pair; pairs inside
// the mask are queued in shared memory.  Pass 2 spreads the queued pairs over 8-lane groups which
// evaluate the feature distances by direct differences (float32 inputs, float64 accumulation).
// ---------------------------------------------------------------------------------------------
constexpr int AT = 64;

__global__ void __launch_bounds__(256)
k_zero_rows(int n, const float* __restrict__ f, int dim, uint8_t* __restrict__ zero) {
    int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= n) return;
    bool any = false;
    for (int k = lane; k < dim; k += 32) any |= (f[(size_t)row * dim + k] != 0.0f);
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) zero[row] = any ? 0 : 1;          // ~tarl.any(1), ncuts_utils.py:143
}

__device__ __forceinline__ double feat_dist8(const float* __restrict__ a, const float* __restrict__ b,
                                             int dim, int lane8) {
    double s = 0.0;
    for (int k = lane8 * 4; k < dim; k += 32) {
        float4 x = *reinterpret_cast<const float4*>(a + k);
        float4 y = *reinterpret_cast<const float4*>(b + k);
        double d0 = (double)x.x - (double)y.x, d1 = (double)x.y - (double)y.y;
        double d2 = (double)x.z - (double)y.z, d3 = (double)x.w - (double)y.w;
        s += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
    }
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    return sqrt(s);
}

// DINOv2 term over several cameras: S = dd_0 + dd_1 + ... with dd_c = ||a_c - b_c||, a_c = a + c * dim (rows are point-major,
// camera c's dim values at c * dim).  The reference multiplies exp(-gamma dd_c) over the cameras (ncuts_utils.py:129-133); the
// kernels evaluate the single exponential exp(-gamma S).  One float64 sum of squares and one sqrt per camera, the distances added
// in camera order.  The loads of up to CAM_BATCH cameras are issued before their shuffle reductions, so a second camera adds
// bandwidth rather than another dependent round trip.  One camera takes feat_dist8 itself (S = dd_0, bit for bit).
constexpr int CAM_BATCH = 4;

__device__ __forceinline__ double feat_dist8_cams(const float* __restrict__ a, const float* __restrict__ b,
                                                  int dim, int cams, int lane8) {
    if (cams == 1) return feat_dist8(a, b, dim, lane8);
    double S = 0.0;
    for (int c0 = 0; c0 < cams; c0 += CAM_BATCH) {
        double s[CAM_BATCH];
#pragma unroll
        for (int c = 0; c < CAM_BATCH; ++c) s[c] = 0.0;
        for (int k = lane8 * 4; k < dim; k += 32) {
#pragma unroll
            for (int c = 0; c < CAM_BATCH; ++c) {
                if (c0 + c < cams) {
                    const size_t o = (size_t)(c0 + c) * dim + k;
                    float4 x = *reinterpret_cast<const float4*>(a + o);
                    float4 y = *reinterpret_cast<const float4*>(b + o);
                    double d0 = (double)x.x - (double)y.x, d1 = (double)x.y - (double)y.y;
                    double d2 = (double)x.z - (double)y.z, d3 = (double)x.w - (double)y.w;
                    s[c] += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
                }
            }
        }
#pragma unroll
        for (int c = 0; c < CAM_BATCH; ++c) {
            if (c0 + c < cams) {                       // uniform over the warp: cams is a kernel argument
                s[c] += __shfl_xor_sync(0xffffffffu, s[c], 4);
                s[c] += __shfl_xor_sync(0xffffffffu, s[c], 2);
                s[c] += __shfl_xor_sync(0xffffffffu, s[c], 1);
                S += sqrt(s[c]);
            }
        }
    }
    return S;
}

__global__ void __launch_bounds__(256)
k_affinity_exact(int n, const double* __restrict__ pts, const float* __restrict__ tarl, int tdim,
                 const float* __restrict__ dino, int ddim, int dcams, const uint8_t* __restrict__ tarl_zero,
                 double alpha, double theta, double gamma, double prox,
                 float* __restrict__ W, long long ld, const int* __restrict__ only_if = nullptr) {
    if (only_if && !*only_if) return;       // conditional fallback after the two-pass form (pair queue overflow)
    __shared__ double pr[AT][3];
    __shared__ double pc[AT][3];
    __shared__ float pr32[AT][3];           // coordinates relative to the tile's first row point: float32 pre-filter
    __shared__ float pc32[AT][3];
    __shared__ __align__(16) float tile[AT][AT];
    __shared__ unsigned short queue[AT * AT];
    __shared__ int qn;

    const int row0 = blockIdx.y * AT, col0 = blockIdx.x * AT;
    const int tid = threadIdx.x;
    if (tid == 0) qn = 0;
    for (int i = tid; i < AT * 3; i += 256) {
        int p = i / 3, k = i % 3;
        int gr = row0 + p, gc = col0 + p;
        double org = pts[(size_t)min(row0, n - 1) * 3 + k];
        double a = gr < n ? pts[(size_t)gr * 3 + k] : 0.0;
        double b = gc < n ? pts[(size_t)gc * 3 + k] : 0.0;
        pr[p][k] = a;
        pc[p][k] = b;
        pr32[p][k] = (float)(a - org);
        pc32[p][k] = (float)(b - org);
    }
    __syncthreads();
    // pairs whose float32 distance exceeds prox by more than this margin are outside for certain (the
    // float32 error of the relative coordinates is orders of magnitude smaller); every pair that might be
    // inside still takes the exact float64 test below, so the result is unchanged
    const float lim32 = (float)((prox + 1e-2) * (prox + 1e-2) * 1.001);

    const bool feats = (theta != 0.0 && tarl != nullptr) || (gamma != 0.0 && dino != nullptr);
    const int cg = (tid & 15) * 4, rg = tid >> 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int r = rg + 16 * k;
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
            int c = cg + c4;
            float out = 0.0f;
            float fx = pr32[r][0] - pc32[c][0], fy = pr32[r][1] - pc32[c][1], fz = pr32[r][2] - pc32[c][2];
            if (row0 + r < n && col0 + c < n && !(fx * fx + fy * fy + fz * fz > lim32)) {
                double dx = pr[r][0] - pc[c][0], dy = pr[r][1] - pc[c][1], dz = pr[r][2] - pc[c][2];
                // cdist accumulates the squares one after another in float64 without contraction
                double s = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
                double sd = __dsqrt_rn(s);
                if (sd <= prox) {                                    // ncuts_utils.py:61, inclusive
                    double a = alpha != 0.0 ? alpha * sd : 0.0;      // :63-66
                    if (feats) {
                        out = (float)a;
                        int q = atomicAdd(&qn, 1);
                        queue[q] = (unsigned short)(r * AT + c);
                    } else {
                        out = (float)exp(-a);
                    }
                }
            }
            tile[r][c] = out;
        }
    }
    __syncthreads();

    if (feats) {
        const int total = qn;
        const int grp = tid >> 3, lane8 = tid & 7;
        const int rounds = (total + 31) / 32;
        for (int it = 0; it < rounds; ++it) {
            int q = it * 32 + grp;
            bool live = q < total;
            int idx = live ? queue[q] : 0;
            int r = idx / AT, c = idx % AT;
            int gi = row0 + r, gj = col0 + c;
            if (!live) { gi = 0; gj = 0; }                            // keep the 8-lane shuffles uniform
            // alpha * spatial distance again in float64 (the tile holds it rounded to float32, one ulp of W off the
            // rounded reference)
            const double dx = pr[r][0] - pc[c][0], dy = pr[r][1] - pc[c][1], dz = pr[r][2] - pc[c][2];
            const double sd = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
            double arg = alpha != 0.0 ? alpha * sd : 0.0;
            if (theta != 0.0 && tarl != nullptr) {
                double td = feat_dist8(tarl + (size_t)gi * tdim, tarl + (size_t)gj * tdim, tdim, lane8);
                if (tarl_zero[gi] | tarl_zero[gj]) td = 0.0;          // ncuts_utils.py:145-146
                arg += theta * td;
            }
            if (gamma != 0.0 && dino != nullptr) {
                const size_t ds = (size_t)dcams * ddim;
                double dd = feat_dist8_cams(dino + gi * ds, dino + gj * ds, ddim, dcams, lane8);
                arg += gamma * dd;                                    // :129-133
            }
            if (live && lane8 == 0) tile[r][c] = (float)exp(-arg);
        }
        __syncthreads();
    }

#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int r = rg + 16 * k;
        int gr = row0 + r, gc = col0 + cg;
        if (gr < n && gc < ld) {
            float4 v = *reinterpret_cast<const float4*>(&tile[r][cg]);
            *reinterpret_cast<float4*>(W + (size_t)gr * ld + gc) = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Stage 1, two-pass form used when feature terms are present (default).  The one-kernel form above evaluates the
// feature distances of a tile inside the tile's CTA: tiles on the diagonal hold thousands of in-mask pairs, tiles
// elsewhere none, and the dense tiles became the tail of the launch (0.18 ms at N = 8.6 k against a 0.05 ms store
// floor).  Here pass 1 only tests distances on the upper triangle, zero-fills W and appends the in-mask pairs
// (i < j) to a queue; pass 2 spreads the queue evenly over the grid, one 8-lane group per pair, and writes both
// W_ij and W_ji (cdist is symmetric bit for bit).  Pass 1 also joins i and j in the union-find forest of the
// root-level connected components, which saves the first k_cc_union pass over the dense matrix.
// ---------------------------------------------------------------------------------------------
struct PairQ { int i, j; double a; };      // a = alpha * spatial distance (float64)

// forward declarations (defined with the component kernels below)
__device__ __forceinline__ void uf_union(int* parent, int a, int b);

// Measured on B200 (N = 8.6 k): the zero stores of this kernel are free (replacing them by one cudaMemsetAsync at
// 7.5 TB/s did not shorten it); ncu showed it issue-bound at 47 instructions per pair, hence the register pre-filter
// below.  Hits are collected in a register bit mask and appended with one atomic per warp.  Merging the components
// inside the tile first (shared-memory union-find, then one global union per non-root) was measured SLOWER than one
// global union per pair (24.3 vs 20.8 ms of affinity time per 128 chunks) and is not used.
__global__ void __launch_bounds__(256)
k_affinity_pairs(int n, const double* __restrict__ pts, double alpha, double prox, float* __restrict__ W, long long ld,
                 PairQ* __restrict__ q, int qcap, int* __restrict__ qctr, int* parent, int pos0) {
    const int row0 = blockIdx.y * AT, col0 = blockIdx.x * AT;
    const int tid = threadIdx.x;
    const int cg = (tid & 15) * 4, rg = tid >> 4;
    if (row0 > col0) {                               // mirror entries: written by pass 2
        if (!W) return;                              // deferred mode: W is written block by block after the root split
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int gr = row0 + rg + 16 * k, gc = col0 + cg;
            if (gr < n && gc < ld) __stcs(reinterpret_cast<float4*>(W + (size_t)gr * ld + gc), make_float4(0.f, 0.f, 0.f, 0.f));
        }
        return;
    }
    __shared__ double pr[AT][3];
    __shared__ double pc[AT][3];
    __shared__ float pr32[AT][3];
    __shared__ float pc32[AT][3];
    __shared__ unsigned short queue[AT * AT];
    __shared__ int qn, qbase;

    if (tid == 0) qn = 0;
    for (int i = tid; i < AT * 3; i += 256) {
        int p = i / 3, k = i % 3;
        int gr = row0 + p, gc = col0 + p;
        double org = pts[(size_t)min(row0, n - 1) * 3 + k];
        double a = gr < n ? pts[(size_t)gr * 3 + k] : 0.0;
        double b = gc < n ? pts[(size_t)gc * 3 + k] : 0.0;
        pr[p][k] = a;
        pc[p][k] = b;
        pr32[p][k] = (float)(a - org);
        pc32[p][k] = (float)(b - org);
    }
    __syncthreads();
    const float lim32 = (float)((prox + 1e-2) * (prox + 1e-2) * 1.001);     // see k_affinity_exact
    // float32 pre-filter on register copies of the coordinates (7 instructions per pair; ncu showed 47 per pair and
    // the issue slots 66 % busy when the index tests and shared-memory reads sat inside the pair loop), then the
    // exact float64 test for the few candidates only
    float cx[4], cy[4], cz[4], rx[4], ry[4], rz[4];
#pragma unroll
    for (int c4 = 0; c4 < 4; ++c4) { cx[c4] = pc32[cg + c4][0]; cy[c4] = pc32[cg + c4][1]; cz[c4] = pc32[cg + c4][2]; }
#pragma unroll
    for (int k = 0; k < 4; ++k) { rx[k] = pr32[rg + 16 * k][0]; ry[k] = pr32[rg + 16 * k][1]; rz[k] = pr32[rg + 16 * k][2]; }
    unsigned cand = 0;                               // bit 4k + c4: pair (rg + 16k, cg + c4)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
            float fx = rx[k] - cx[c4], fy = ry[k] - cy[c4], fz = rz[k] - cz[c4];
            if (!(fx * fx + fy * fy + fz * fz > lim32)) cand |= 1u << (4 * k + c4);
        }
    }
    const bool interior = (col0 >= row0 + AT) && (col0 + AT <= n);      // every pair has i < j < n
    const bool diag_tile = (row0 == col0);
    unsigned hits = 0;
    while (cand) {
        const int b = __ffs(cand) - 1;
        cand &= cand - 1;
        const int r = rg + 16 * (b >> 2), c = cg + (b & 3);
        if (!interior && !(row0 + r < col0 + c && col0 + c < n)) continue;
        double dx = pr[r][0] - pc[c][0], dy = pr[r][1] - pc[c][1], dz = pr[r][2] - pc[c][2];
        double s2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
        if (__dsqrt_rn(s2) <= prox) hits |= 1u << b;                     // ncuts_utils.py:61, inclusive
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (!W) break;
        const int gi = row0 + rg + 16 * k, gc = col0 + cg;
        float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
        if (diag_tile && gi < n) {                                       // unit diagonal: exp(-0)
            if (gi == gc) out.x = 1.0f;
            if (gi == gc + 1) out.y = 1.0f;
            if (gi == gc + 2) out.z = 1.0f;
            if (gi == gc + 3) out.w = 1.0f;
        }
        if (gi < n && gc < ld) __stcs(reinterpret_cast<float4*>(W + (size_t)gi * ld + gc), out);
    }
    // append the hits: exclusive prefix over the warp, one atomic per warp
    {
        const int lane = tid & 31;
        const int cnt = __popc(hits);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        const int wtot = __shfl_sync(0xffffffffu, incl, 31);
        int wbase = 0;
        if (lane == 31 && wtot > 0) wbase = atomicAdd(&qn, wtot);
        wbase = __shfl_sync(0xffffffffu, wbase, 31);
        int pos = wbase + incl - cnt;
        while (hits) {
            const int b = __ffs(hits) - 1;
            hits &= hits - 1;
            queue[pos++] = (unsigned short)((rg + 16 * (b >> 2)) * AT + cg + (b & 3));
        }
    }
    __syncthreads();
    const int total = qn;
    if (total == 0) return;
    if (tid == 0) {
        int b = atomicAdd(&qctr[0], total);
        if (b + total > qcap) { atomicExch(&qctr[1], 1); b = -1; }      // the caller falls back to the one-kernel form
        qbase = b;
    }
    __syncthreads();
    const int base = qbase;
    if (base < 0) return;
    for (int t = tid; t < total; t += 256) {
        int idx = queue[t];
        int r = idx / AT, c = idx % AT;
        double dx = pr[r][0] - pc[c][0], dy = pr[r][1] - pc[c][1], dz = pr[r][2] - pc[c][2];
        double sd = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
        PairQ e;
        e.i = row0 + r; e.j = col0 + c;
        e.a = alpha != 0.0 ? alpha * sd : 0.0;                           // ncuts_utils.py:63-66
        q[base + t] = e;
        // root-level connected components (saves the first k_cc_union pass over the dense matrix)
        if (parent) uf_union(parent, pos0 + e.i, pos0 + e.j);
    }
}

// ---------------------------------------------------------------------------------------------
// Cell grid of the cell-sorted pair search below: pitch >= prox, at most PG_DIM cells per axis (one CTA bins the points
// of a chunk by counting sort in shared memory).  Same inclusive float64 test and operation order as k_affinity_pairs
// (ncuts_utils.py:60-61); every pair is queued exactly once; queue order is arbitrary, W and the union-find forest do
// not depend on it.  (Round 1 walked the 27 neighbour cells with one warp per point and one union per found pair:
// 190 us per chunk, union-find bound; replaced by the tile sweep over the sorted points.)
// ---------------------------------------------------------------------------------------------
constexpr int PG_DIM = 25;
constexpr int PG_CELLS = PG_DIM * PG_DIM * PG_DIM;       // 15625 counters = 61 KB of shared memory
constexpr int PG_STRIDE = PG_CELLS + 7;                  // ints per chunk in the global cell table (start offsets + end)
struct PairGrid { double lo[3]; double inv_h; int n[3]; int pad; };

__device__ __forceinline__ int pg_cell1(const PairGrid& g, double x, int a) {
    int c = (int)floor((x - g.lo[a]) * g.inv_h);
    return max(0, min(g.n[a] - 1, c));
}

// ---------------------------------------------------------------------------------------------
// Pair search on the CELL-SORTED points (ANCUTS_OPT_PAIR_SEARCH = 0, the default), batched over the chunks of a call:
//   k_pair_grid_b   one CTA per chunk: counting sort into cells of pitch >= prox (x fastest), points stored in cell order
//   k_tile_boxes    bounding box of every run of PS_T consecutive sorted points ("tile")
//   k_pair_sweep    one CTA per tile pair (ti <= tj) of a chunk: pairs of tiles whose boxes are farther apart than prox
//                   exit at once (in cell order a tile covers a few adjacent cell rows, so only ~1/5 of the tile pairs
//                   survive), the others take the float32 pre-filter in registers (64 pairs per thread) and the exact
//                   float64 test of k_affinity_pairs; hits go to the chunk's queue with their CELL-SORTED ranks, which are
//                   the positions of the points at the root of the tree (k_init_positions takes the sorted order)
//   k_pair_unions   root-level components: one union per queued pair, in queue order
// Same pairs, same float64 distances as the shuffled 64 x 64 sweep (k_affinity_pairs walks all N^2 / 2 pairs in 8.7 k
// CTAs per chunk of 16 pairs per thread and is bound by its per-CTA overhead: 96 us per 8.4 k-point chunk).
// ---------------------------------------------------------------------------------------------
constexpr int PS_T = 128;                              // points per tile side

__global__ void __launch_bounds__(1024)
k_pair_grid_b(const int* __restrict__ c_n, const int* __restrict__ c_base, const double* __restrict__ pts_all, double prox,
              int* __restrict__ cells_all, int* __restrict__ sorted_all, int* __restrict__ tmp_all,
              double* __restrict__ spts_all, PairGrid* __restrict__ grids) {
    extern __shared__ int hist[];
    __shared__ double red[6][32];
    __shared__ PairGrid g;
    __shared__ int wsum[32];
    const int chunk = blockIdx.x;
    const int n = c_n[chunk];
    const size_t pos0 = (size_t)c_base[chunk];
    const double* pts = pts_all + pos0 * 3;
    int* cell_start = cells_all + (size_t)chunk * PG_STRIDE;
    int* sorted = sorted_all + pos0;
    int* tmp = tmp_all + pos0;
    double* spts = spts_all + pos0 * 3;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double mn[3] = {1e300, 1e300, 1e300}, mx[3] = {-1e300, -1e300, -1e300};
    for (int i = tid; i < n; i += 1024) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { double x = pts[(size_t)i * 3 + a]; mn[a] = fmin(mn[a], x); mx[a] = fmax(mx[a], x); }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double lo = warp_min(mn[a]), hi = -warp_min(-mx[a]);
        if (lane == 0) { red[a][warp] = lo; red[3 + a][warp] = hi; }
    }
    for (int c = tid; c < PG_CELLS; c += 1024) hist[c] = 0;
    __syncthreads();
    if (tid == 0) {
        double ext = 0.0;
        for (int a = 0; a < 3; ++a) {
            double lo = red[a][0], hi = red[3 + a][0];
            for (int w = 1; w < 32; ++w) { lo = fmin(lo, red[a][w]); hi = fmax(hi, red[3 + a][w]); }
            g.lo[a] = lo; red[3 + a][0] = hi;
            ext = fmax(ext, hi - lo);
        }
        const double pitch = fmax(fmax(prox, ext / (double)(PG_DIM - 1)), 1e-300);
        g.inv_h = 1.0 / pitch;
        for (int a = 0; a < 3; ++a) g.n[a] = min(PG_DIM, (int)floor((red[3 + a][0] - g.lo[a]) * g.inv_h) + 1);
        g.pad = 0;
        grids[chunk] = g;
    }
    __syncthreads();
    for (int i = tid; i < n; i += 1024) {
        const int c = (pg_cell1(g, pts[(size_t)i * 3 + 2], 2) * g.n[1] + pg_cell1(g, pts[(size_t)i * 3 + 1], 1)) * g.n[0]
                      + pg_cell1(g, pts[(size_t)i * 3], 0);
        atomicAdd(&hist[c], 1);
    }
    __syncthreads();
    constexpr int PER = (PG_CELLS + 1023) / 1024;          // 16 consecutive cells per thread, then a scan of the partial sums
    const int c0 = tid * PER;
    int loc[PER];
    int s = 0;
#pragma unroll
    for (int k = 0; k < PER; ++k) { int c = c0 + k; int v = (c < PG_CELLS) ? hist[c] : 0; loc[k] = s; s += v; }
    int incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = wsum[lane];
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
        wsum[lane] = wi - w;
    }
    __syncthreads();
    const int base = wsum[warp] + incl - s;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        int c = c0 + k;
        if (c < PG_CELLS) { hist[c] = base + loc[k]; cell_start[c] = base + loc[k]; }
    }
    if (tid == 0) cell_start[PG_CELLS] = n;
    __syncthreads();
    // The slot inside a cell follows the atomics; the sorted order is the order of the points in every node of the tree
    // (k_init_positions), so it has to be the same in every run: a second pass ranks the points of a cell by input index.
    for (int i = tid; i < n; i += 1024) {
        const int c = (pg_cell1(g, pts[(size_t)i * 3 + 2], 2) * g.n[1] + pg_cell1(g, pts[(size_t)i * 3 + 1], 1)) * g.n[0]
                      + pg_cell1(g, pts[(size_t)i * 3], 0);
        tmp[atomicAdd(&hist[c], 1)] = i;
    }
    __syncthreads();
    for (int q = tid; q < n; q += 1024) {
        const int i = tmp[q];
        const int c = (pg_cell1(g, pts[(size_t)i * 3 + 2], 2) * g.n[1] + pg_cell1(g, pts[(size_t)i * 3 + 1], 1)) * g.n[0]
                      + pg_cell1(g, pts[(size_t)i * 3], 0);
        const int start = cell_start[c], end = hist[c];            // hist[c] has advanced to the end of the cell
        int rank = 0;
        for (int t = start; t < end; ++t) rank += (tmp[t] < i) ? 1 : 0;
        const int pos = start + rank;
        sorted[pos] = i;
        spts[(size_t)pos * 3] = pts[(size_t)i * 3];
        spts[(size_t)pos * 3 + 1] = pts[(size_t)i * 3 + 1];
        spts[(size_t)pos * 3 + 2] = pts[(size_t)i * 3 + 2];
    }
}

// grid: (tiles of the largest chunk, chunks), PS_T threads
__global__ void __launch_bounds__(PS_T)
k_tile_boxes(const int* __restrict__ c_n, const int* __restrict__ c_base, const int* __restrict__ c_tile0,
             const double* __restrict__ spts_all, double* __restrict__ tbox) {
    __shared__ double red[6][PS_T / 32];
    const int chunk = blockIdx.y, t = blockIdx.x;
    const int n = c_n[chunk];
    if (t * PS_T >= n) return;
    const int i = min(t * PS_T + (int)threadIdx.x, n - 1);              // the last tile repeats its last point
    const double* q = spts_all + ((size_t)c_base[chunk] + i) * 3;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double lo = warp_min(q[a]), hi = warp_max(q[a]);
        if (lane == 0) { red[a][warp] = lo; red[3 + a][warp] = hi; }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        const int a = threadIdx.x;
        double v = red[a][0];
        for (int w = 1; w < PS_T / 32; ++w) v = (a < 3) ? fmin(v, red[a][w]) : fmax(v, red[a][w]);
        tbox[((size_t)c_tile0[chunk] + t) * 6 + a] = v;
    }
}

// grid: (tile pairs of the largest chunk, chunks), 256 threads; tile pair L -> (ti <= tj) with L = tj (tj + 1) / 2 + ti
__global__ void __launch_bounds__(256)
k_pair_sweep(const int* __restrict__ c_n, const int* __restrict__ c_base, const int* __restrict__ c_tile0,
             const double* __restrict__ spts_all, const double* __restrict__ tbox,
             double alpha, double prox, PairQ* __restrict__ q_all, const long long* __restrict__ q_off,
             const int* __restrict__ q_cap, int* __restrict__ qctr_all) {
    const int chunk = blockIdx.y;
    const int n = c_n[chunk];
    const int T = (n + PS_T - 1) / PS_T;
    const int L = blockIdx.x;
    int tj = (int)((sqrt(8.0 * (double)L + 1.0) - 1.0) * 0.5);
    while ((tj + 1) * (tj + 2) / 2 <= L) ++tj;                           // guard the float square root
    while (tj * (tj + 1) / 2 > L) --tj;
    const int ti = L - tj * (tj + 1) / 2;
    if (tj >= T) return;
    {
        const double* ba = tbox + ((size_t)c_tile0[chunk] + ti) * 6;
        const double* bb = tbox + ((size_t)c_tile0[chunk] + tj) * 6;
        double g2 = 0.0;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const double d = fmax(0.0, fmax(ba[a] - bb[3 + a], bb[a] - ba[3 + a]));
            g2 += d * d;
        }
        if (g2 > prox * prox * 1.000001) return;                         // no pair of the two tiles can be inside the mask
    }
    __shared__ double pr[PS_T][3];
    __shared__ double pc[PS_T][3];
    __shared__ float pr32[PS_T][3];
    __shared__ float pc32[PS_T][3];
    __shared__ unsigned short queue[PS_T * PS_T];
    __shared__ int qn, qbase;
    const int tid = threadIdx.x;
    const size_t pos0 = (size_t)c_base[chunk];
    const double* sp = spts_all + pos0 * 3;
    const int row0 = ti * PS_T, col0 = tj * PS_T;
    if (tid == 0) qn = 0;
    for (int i = tid; i < PS_T * 3; i += 256) {
        const int pnt = i / 3, k = i % 3;
        const int gr = row0 + pnt, gc = col0 + pnt;
        const double org = sp[(size_t)row0 * 3 + k];
        const double a = gr < n ? sp[(size_t)gr * 3 + k] : 1e30;        // padding points are far from everything
        const double b = gc < n ? sp[(size_t)gc * 3 + k] : -1e30;
        pr[pnt][k] = a; pc[pnt][k] = b;
        pr32[pnt][k] = (float)(a - org); pc32[pnt][k] = (float)(b - org);
    }
    __syncthreads();
    const float lim32 = (float)((prox + 1e-2) * (prox + 1e-2) * 1.001);     // see k_affinity_exact
    const int rg = (tid >> 4) * 8, cg = (tid & 15) * 8;                 // 8 x 8 pairs per thread
    float cx[8], cy[8], cz[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) { cx[c] = pc32[cg + c][0]; cy[c] = pc32[cg + c][1]; cz[c] = pc32[cg + c][2]; }
    const bool diag = (ti == tj);
    const int lane = tid & 31;
#pragma unroll 1
    for (int r = 0; r < 8; ++r) {
        const float rx = pr32[rg + r][0], ry = pr32[rg + r][1], rz = pr32[rg + r][2];
        unsigned cand = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const float fx = rx - cx[c], fy = ry - cy[c], fz = rz - cz[c];
            if (!(fx * fx + fy * fy + fz * fz > lim32)) cand |= 1u << c;
        }
        unsigned hits = 0;
        const int row = rg + r;
        while (cand) {
            const int c = __ffs(cand) - 1;
            cand &= cand - 1;
            const int col = cg + c;
            if (diag && col <= row) continue;                            // every pair once
            const double dx = pr[row][0] - pc[col][0], dy = pr[row][1] - pc[col][1], dz = pr[row][2] - pc[col][2];
            const double s2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
            if (__dsqrt_rn(s2) <= prox) hits |= 1u << c;                 // ncuts_utils.py:61, inclusive
        }
        // append this row's hits: exclusive prefix over the warp, one shared-memory atomic per warp
        const int cnt = __popc(hits);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        const int wtot = __shfl_sync(0xffffffffu, incl, 31);
        int wbase = 0;
        if (lane == 31 && wtot > 0) wbase = atomicAdd(&qn, wtot);
        wbase = __shfl_sync(0xffffffffu, wbase, 31);
        int pos = wbase + incl - cnt;
        while (hits) {
            const int c = __ffs(hits) - 1;
            hits &= hits - 1;
            queue[pos++] = (unsigned short)(row * PS_T + cg + c);
        }
    }
    __syncthreads();
    const int total = qn;
    if (total == 0) return;
    int* qctr = qctr_all + 2 * chunk;
    if (tid == 0) {
        int b = atomicAdd(&qctr[0], total);
        if (b + total > q_cap[chunk]) { atomicExch(&qctr[1], 1); b = -1; }   // the caller falls back to the dense form
        qbase = b;
    }
    __syncthreads();
    const int base = qbase;
    if (base < 0) return;
    PairQ* q = q_all + q_off[chunk];
    for (int t = tid; t < total; t += 256) {
        const int idx = queue[t];
        const int r = idx / PS_T, c = idx % PS_T;
        const double dx = pr[r][0] - pc[c][0], dy = pr[r][1] - pc[c][1], dz = pr[r][2] - pc[c][2];
        const double sd = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
        PairQ e;
        e.i = row0 + r; e.j = col0 + c;                                  // cell-sorted ranks (ti <= tj, col > row on the diagonal): i < j
        e.a = alpha != 0.0 ? alpha * sd : 0.0;                           // ncuts_utils.py:63-66
        q[base + t] = e;
    }
}

// grid: (blocks, chunks).  The queue is walked in order.  While it held input indices the entries were visited in a scattered
// order ((t * 2147483629) mod total), because neighbouring threads hooked into the same component at the same time; since
// the queue holds cell-sorted ranks (neighbouring entries, neighbouring tree nodes, coalesced loads) the plain order is the
// faster one: pair stage + feature pass 8.19 -> 7.52 ms per 128 chunks.
__global__ void __launch_bounds__(256)
k_pair_unions(const PairQ* __restrict__ q_all, const long long* __restrict__ q_off, const int* __restrict__ q_cap,
              const int* __restrict__ qctr_all, const int* __restrict__ c_base, int* parent) {
    const int chunk = blockIdx.y;
    if (qctr_all[2 * chunk + 1]) return;
    const long long total = min(qctr_all[2 * chunk], q_cap[chunk]);
    const PairQ* q = q_all + q_off[chunk];
    const int pos0 = c_base[chunk];
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const PairQ e = q[t];
        uf_union(parent, pos0 + e.i, pos0 + e.j);
    }
}

// pass 2: one 8-lane group per pair.  Block blk of nblk takes its piece of the `total` queued pairs.
// The queue holds chunk-local indices; the chunk's rows of tarl, dino, tarl_zero, order and inv start at row `base`.
// order != NULL: the queue holds cell-sorted ranks (= root positions); order[rank] = input index, where the features are
// inv != NULL (deferred mode): the pair is written at the positions its points have AFTER the root split
// (inv[old global position] = new global position), and only if their range goes on to the eigensolver.
__device__ __forceinline__ void
affinity_feats_piece(const PairQ* __restrict__ q, int total, int blk, int nblk,
                     const float* __restrict__ tarl, int tdim, const float* __restrict__ dino, int ddim, int dcams,
                     const uint8_t* __restrict__ tarl_zero, double theta, double gamma,
                     float* __restrict__ W, long long ld,
                     const int* __restrict__ inv, int base, const int* __restrict__ rid,
                     const int* __restrict__ r_status, const int* __restrict__ order, float* __restrict__ slot,
                     int* __restrict__ cnt) {
    const int lane8 = threadIdx.x & 7;
    // a block takes a CONTIGUOUS piece of the queue: the sweep appends the hits of one tile pair (128 x 128 points) together,
    // so the piece touches a few hundred feature rows, each about twenty times -- they stay in L1 (a grid-stride walk sent
    // every row read to L2: 147 MB per 8.4 k-point chunk)
    const int per_block = (((total + nblk - 1) / nblk) + 31) & ~31;
    const int b0 = blk * per_block, b1 = min(total, b0 + per_block);
    // two pairs per 8-lane group and trip, written as two independent instruction streams: a pair is a chain of six
    // dependent global-memory round trips (queue entry, order table, feature rows, position table, range id, range state),
    // and a thread only makes about ten trips -- with one pair at a time the kernel ran at the latency of that chain
    for (int i0 = b0; i0 < b1; i0 += 64) {
        int gi[2], gj[2], fi[2], fj[2];
        double a[2], arg[2];
        bool live[2];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int idx = i0 + 32 * s + (threadIdx.x >> 3);
            live[s] = idx < b1;
            gi[s] = 0; gj[s] = 0; a[s] = 0.0;
            if (live[s]) { PairQ e = q[idx]; gi[s] = e.i; gj[s] = e.j; a[s] = e.a; }
        }
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            fi[s] = base + (order ? order[base + gi[s]] : gi[s]);
            fj[s] = base + (order ? order[base + gj[s]] : gj[s]);
            arg[s] = 0.0;
        }
        if (theta != 0.0 && tarl != nullptr) {
            double td[2];
#pragma unroll
            for (int s = 0; s < 2; ++s) td[s] = feat_dist8(tarl + (size_t)fi[s] * tdim, tarl + (size_t)fj[s] * tdim, tdim, lane8);
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                if (tarl_zero[fi[s]] | tarl_zero[fj[s]]) td[s] = 0.0;    // ncuts_utils.py:145-146
                arg[s] += theta * td[s];
            }
        }
        if (gamma != 0.0 && dino != nullptr) {
            double dd[2];
            const size_t ds = (size_t)dcams * ddim;          // row stride: every camera's ddim values
#pragma unroll
            for (int s = 0; s < 2; ++s) dd[s] = feat_dist8_cams(dino + fi[s] * ds, dino + fj[s] * ds, ddim, dcams, lane8);
#pragma unroll
            for (int s = 0; s < 2; ++s) arg[s] += gamma * dd[s];         // :129-133
        }
        if (lane8 == 0) {
            int wi[2], wj[2];
            bool keep[2];
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                wi[s] = gi[s]; wj[s] = gj[s]; keep[s] = live[s];
                if (inv && live[s]) {
                    const int pi = inv[base + gi[s]], pj = inv[base + gj[s]];
                    keep[s] = r_status[rid[pi]] == ST_ACTIVE;
                    wi[s] = pi - base; wj[s] = pj - base;
                }
            }
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                if (slot) {
                    // CSR node form: the value in queue order (0 = not stored), coalesced, and one more entry in the two
                    // rows (k_ncsr_pairs places it with the same test)
                    if (live[s]) {
                        const float w = keep[s] ? (float)exp(-(a[s] + arg[s])) : 0.0f;
                        slot[i0 + 32 * s + (threadIdx.x >> 3)] = w;
                        if (w != 0.0f && rid[base + wi[s]] == rid[base + wj[s]]) {
                            atomicAdd(cnt + base + wi[s], 1);
                            atomicAdd(cnt + base + wj[s], 1);
                        }
                    }
                } else if (keep[s]) {
                    const float w = (float)exp(-(a[s] + arg[s]));
                    W[(size_t)wi[s] * ld + wj[s]] = w;
                    W[(size_t)wj[s] * ld + wi[s]] = w;
                }
            }
        }
    }
}

// one queue (the stage entry, and the host entry's per-chunk passes, which wait for each chunk's features)
__global__ void __launch_bounds__(256)
k_affinity_feats(const PairQ* __restrict__ q, const int* __restrict__ qctr, int qcap,
                 const float* __restrict__ tarl, int tdim, const float* __restrict__ dino, int ddim, int dcams,
                 const uint8_t* __restrict__ tarl_zero, double theta, double gamma,
                 float* __restrict__ W, long long ld,
                 const int* __restrict__ inv = nullptr, int base = 0, const int* __restrict__ rid = nullptr,
                 const int* __restrict__ r_status = nullptr, const int* __restrict__ order = nullptr,
                 float* __restrict__ slot = nullptr, int* __restrict__ cnt = nullptr) {
    if (qctr[1]) return;                             // overflow: everything is redone by the one-kernel form
    affinity_feats_piece(q, min(qctr[0], qcap), blockIdx.x, gridDim.x, tarl, tdim, dino, ddim, dcams, tarl_zero, theta, gamma,
                         W, ld, inv, base, rid, r_status, order, slot, cnt);
}

// deferred pass of a resident batch in one launch, grid (blocks per chunk, chunks): block (x, c) takes the piece of chunk c's
// queue that block x of a k_affinity_feats launch over that queue alone would take, so every W entry gets the same value.
// With one launch per chunk a 128-chunk step ran 128 launches of one wave each (592 blocks of 64 registers fill the 148 SMs
// once) on one stream.  Chunk c's rows start at c_base[c]; its blocks go to Wc[c] with leading dimension c_ld[c], or, with
// slot != NULL (CSR node form), the values to slot[q_off[c] + queue index] and the rows' entry counts to cnt.
__global__ void __launch_bounds__(256)
k_affinity_feats_b(const PairQ* __restrict__ q_all, const long long* __restrict__ q_off, const int* __restrict__ q_cap,
                   const int* __restrict__ qctr_all, const int* __restrict__ c_base,
                   const float* __restrict__ tarl, int tdim, const float* __restrict__ dino, int ddim, int dcams,
                   const uint8_t* __restrict__ tarl_zero, double theta, double gamma,
                   float* const* __restrict__ Wc, const int* __restrict__ c_ld,
                   const int* __restrict__ inv, const int* __restrict__ rid, const int* __restrict__ r_status,
                   const int* __restrict__ order, float* __restrict__ slot, int* __restrict__ cnt) {
    const int c = blockIdx.y;
    const int* qctr = qctr_all + 2 * c;
    if (qctr[1]) return;                             // overflow: everything is redone by the one-kernel form
    affinity_feats_piece(q_all + q_off[c], min(qctr[0], q_cap[c]), blockIdx.x, gridDim.x, tarl, tdim, dino, ddim, dcams,
                         tarl_zero, theta, gamma, slot ? nullptr : Wc[c], c_ld[c], inv, c_base[c], rid, r_status, order,
                         slot ? slot + q_off[c] : nullptr, cnt);
}

// ---------------------------------------------------------------------------------------------
// Stage 2: degrees of W = w + I for every active node:  d_i = 1 + sum_j w_ij  (float64)
//   normalized_cut.py:38,42-43.  One warp per row, aligned 128-bit window loads.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double row_sum_window(const float* __restrict__ rowp, int c_lo, int c_hi, int lane,
                                                 int* nnz_out = nullptr) {
    double acc = 0.0;
    int nz = 0;
    int a0 = c_lo & ~3;
    for (int c = a0 + lane * 4; c < c_hi; c += 128) {
        float4 w = ld_stream4(rowp + c);
        double s = 0.0;
        if (c >= c_lo && c + 3 < c_hi) {
            s = ((double)w.x + (double)w.y) + ((double)w.z + (double)w.w);
            nz += (w.x != 0.0f) + (w.y != 0.0f) + (w.z != 0.0f) + (w.w != 0.0f);
        } else {
            if (c >= c_lo && c < c_hi) { s += (double)w.x; nz += (w.x != 0.0f); }
            if (c + 1 >= c_lo && c + 1 < c_hi) { s += (double)w.y; nz += (w.y != 0.0f); }
            if (c + 2 >= c_lo && c + 2 < c_hi) { s += (double)w.z; nz += (w.z != 0.0f); }
            if (c + 3 >= c_lo && c + 3 < c_hi) { s += (double)w.w; nz += (w.w != 0.0f); }
        }
        acc += s;
    }
    if (nnz_out) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nz += __shfl_xor_sync(0xffffffffu, nz, o);
        *nnz_out = nz;
    }
    return warp_sum(acc);
}

__global__ void __launch_bounds__(256)
k_degree(Eng e, int cur) {
    int a = blockIdx.y;
    NodeView v = node_view(e, e.a_rid[a], cur);
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int row = blockIdx.x * 8 + warp;
    if (row >= v.n) return;
    const float* rowp = v.W + (size_t)(v.ro + row) * v.ld;
    int nnz = 0;
    double s = row_sum_window(rowp, v.ro, v.ro + v.n, lane, &nnz);
    if (lane == 0) {
        double d = 1.0 + s;                         // + identity (normalized_cut.py:38)
        e.deg[v.start + row] = d;
        e.sinv[v.start + row] = 1.0 / sqrt(d);      // :43
        e.rownnz[v.start + row] = nnz;              // stored entries of the row inside its block (shared-memory sparse matvec)
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        atomicAdd(&e.acct[SG_DEGREE], 4ull * v.n * v.n);
}

// plain dense version for the stage-2 entry point (optionally writes M = D^-1/2 (w+I) D^-1/2)
__global__ void __launch_bounds__(256)
k_degree_dense(int n, const float* __restrict__ W, long long ld, double* __restrict__ deg) {
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int row = blockIdx.x * 8 + warp;
    if (row >= n) return;
    double s = row_sum_window(W + (size_t)row * ld, 0, n, lane);
    if (lane == 0) deg[row] = 1.0 + s;
}

// grid: (column tiles of 1024, row tiles of NRM_ROWS).  The row scales of the tile are computed once per
// block into shared memory (one float64 rsqrt per row instead of one per row and thread: the first version
// was bound by the FP64 pipe at 40 % of the HBM peak), the four column scales once per thread.
constexpr int NRM_ROWS = 32;
__global__ void __launch_bounds__(256)
k_normalize_dense(int n, const float* __restrict__ W, long long ld, const double* __restrict__ deg,
                  float* __restrict__ M, long long ldm) {
    __shared__ double srow[NRM_ROWS];
    const int r0 = blockIdx.y * NRM_ROWS;
    if (threadIdx.x < NRM_ROWS) srow[threadIdx.x] = (r0 + threadIdx.x < n) ? rsqrt(deg[r0 + threadIdx.x]) : 0.0;
    __syncthreads();
    int c = (blockIdx.x * 256 + threadIdx.x) * 4;
    if (c >= n) return;
    double sc[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) sc[k] = (c + k < n) ? rsqrt(deg[c + k]) : 0.0;
#pragma unroll
    for (int rb = 0; rb < NRM_ROWS; rb += 8) {
        float4 w[8];
#pragma unroll
        for (int r = 0; r < 8; ++r)
            if (r0 + rb + r < n) w[r] = ld_stream4(W + (size_t)(r0 + rb + r) * ld + c);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            int row = r0 + rb + r;
            if (row >= n) break;
            double si = srow[rb + r];
            float in[4] = {w[r].x, w[r].y, w[r].z, w[r].w};
            float out[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                int cc = c + k;
                out[k] = (cc < n) ? (float)(((double)in[k] + (cc == row ? 1.0 : 0.0)) * si * sc[k]) : 0.0f;
            }
            __stcs(reinterpret_cast<float4*>(M + (size_t)row * ldm + c), make_float4(out[0], out[1], out[2], out[3]));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Connected components of each side of every SPLIT range (lock-free union-find; the larger root
// is hooked under the smaller one, so the final root of a component is its smallest position and
// the result does not depend on scheduling).
//   Replaces the reference's null-space splits of disconnected nodes (normalized_cut.py:49-58 with
//   lambda_2 = 0); see DESIGN.md "degenerate nodes".
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int uf_load(const int* parent, int x) {
    return __ldcg(parent + x);
}
__device__ __forceinline__ int uf_find(int* parent, int x) {
    int p = uf_load(parent, x);
    while (p != x) {
        int gp = uf_load(parent, p);
        if (gp != p) parent[x] = gp;     // path halving; only ever points to an ancestor
        x = p;
        p = gp;
    }
    return x;
}
__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }       // a > b: hook a under b
        if (atomicCAS(parent + a, a, b) == a) return;
    }
}

__global__ void k_cc_init(Eng e) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < e.P) e.parent[g] = g;
}

// grid: (row blocks of 8 rows, split list).  split list = ranges with ST_SPLIT, ids in a_rid-like list
__global__ void __launch_bounds__(256)
k_cc_union(Eng e, int cur, const int* __restrict__ split_ids) {
    int r = split_ids[blockIdx.y];
    NodeView v = node_view(e, r, cur);
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int row = blockIdx.x * 8 + warp;
    if (row >= v.n) return;
    int gi = v.start + row;
    int si = e.side[gi];
    if (e.r_pass[2 * r + si] != 1) return;         // 0: a side at or below the size limit stays whole; 2: joined by cl_fused_cut
    const float* rowp = v.W + (size_t)(v.ro + row) * v.ld;
    int c_lo = v.ro + row + 1, c_hi = v.ro + v.n;  // upper triangle only (w is symmetric)
    int a0 = c_lo & ~3;
    for (int c = a0 + lane * 4; c < c_hi; c += 128) {
        float4 w = ld_stream4(rowp + c);
        float in[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int cc = c + k;
            if (cc >= c_lo && cc < c_hi && in[k] != 0.0f) {
                int gj = v.start + (cc - v.ro);
                if (e.side[gj] == si) uf_union(e.parent, gi, gj);
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        atomicAdd(&e.acct[SG_PARTITION], 2ull * v.n * v.n);
}

__global__ void k_cc_flatten(Eng e) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < e.P) e.croot[g] = uf_find(e.parent, g);
}

// ---------------------------------------------------------------------------------------------
// Range-table rebuild.  Sort key = (range start << 32) | (side << 30 | component root + 1);
// leaves keep key low = 0 so the stable sort leaves them in place.  Mask side first
// (normalized_cut.py:57-59).
// ---------------------------------------------------------------------------------------------
__global__ void k_build_keys(Eng e) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= e.P) return;
    int r = e.rid[g];
    unsigned int lo = 0;
    int start = e.r_start[r];
    if (e.r_status[r] == ST_SPLIT) {
        int s = e.side[g];
        lo = ((unsigned int)s << 30);
        if (e.r_pass[2 * r + s]) lo |= (unsigned int)(e.croot[g] - start + 1);
    }
    e.key[g] = ((unsigned long long)(unsigned int)start << 32) | lo;
    e.val[g] = g;
}

__global__ void k_boundaries(Eng e) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= e.P) return;
    e.flag[p] = (p == 0 || e.key2[p] != e.key2[p - 1]) ? 1 : 0;
}

// after the inclusive scan of flag -> incl
__global__ void k_new_ranges(Eng e) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= e.P) return;
    int nr = e.incl[p] - 1;
    e.rid2[p] = nr;
    e.perm2[p] = e.perm[e.val2[p]];
    if (e.flag[p]) {
        int oldr = e.rid[e.val2[p]];
        e.q_start[nr] = p;
        e.q_chunk[nr] = e.r_chunk[oldr];
        // provisional: remember whether the parent range was being split; level of the child
        e.q_status[nr] = (e.r_status[oldr] == ST_SPLIT) ? ST_ACTIVE : ST_LEAF;
        e.q_level[nr] = e.r_level[oldr] + ((e.r_status[oldr] == ST_SPLIT) ? 1 : 0);
    }
    if (p == e.P - 1) e.ctr[0] = nr + 1;
}

// sizes, stop rule (normalized_cut.py:39-40 with the child default 0.01), active slots
__global__ void k_finish_ranges(Eng e, int num_ranges) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= num_ranges) return;
    int start = e.q_start[r];
    int end = (r + 1 < num_ranges) ? e.q_start[r + 1] : e.P;
    int n = end - start;
    e.q_n[r] = n;
    int st = e.q_status[r];
    if (st == ST_ACTIVE) {
        int c = e.q_chunk[r];
        double frac = (double)n / ((double)e.c_norig[c] + 1e-8);
        bool pass = (n > 2) && (frac > CHILD_SPLIT_LIM);
        if (!pass) st = ST_LEAF;
    }
    e.q_status[r] = st;
    if (st == ST_ACTIVE) {
        int a = atomicAdd(&e.ctr[1], 1);
        int nch = (n + CH - 1) / CH;
        e.a_rid[a] = r;
        e.a_nch[a] = nch;
        e.a_slot0[a] = atomicAdd(&e.ctr[3], nch);
        atomicMax(&e.ctr[2], n);
        e.a_done[a] = DONE_NO;
        e.a_path[a] = 1;
        e.a_fused[a] = 0;
        int cls = cluster_class(n);
        if (cls >= 0) e.cl_ids[cls * e.active_cap + atomicAdd(&e.ctr[8 + cls], 1)] = a;
        else atomicAdd(&e.ctr[14], 1);
    }
}

// gather the blocks of the new ACTIVE ranges from the old buffer into the other one:
//   w[mask][:, mask] etc. (normalized_cut.py:57-58).  Called after the rebuilt table became current;
//   val2[new position] = old position.  grid: (col tiles of 256, row tiles of 16, active)
__global__ void __launch_bounds__(256)
k_gather_blocks_cur(Eng e, int cur /* source buffer */) {
    // (one launch per size bin, so that no block exits at once, was measured: no gain)
    int a = blockIdx.z;
    int r = e.a_rid[a];
    int start = e.r_start[r], n = e.r_n[r], c = e.r_chunk[r];
    int col = blockIdx.x * 256 + threadIdx.x;
    int row0 = blockIdx.y * 16;
    if (row0 >= n) return;
    int base = e.c_base[c], ld = e.c_ld[c];
    const float* src = cur ? e.c_W1[c] : e.c_W0[c];
    float* dst = cur ? e.c_W0[c] : e.c_W1[c];
    int ro = start - base;
    if (col < n) {
        int sc = e.val2[start + col] - base;
        int rows = min(16, n - row0);
        for (int i = 0; i < rows; ++i) {
            int sr = e.val2[start + row0 + i] - base;
            dst[(size_t)(ro + row0 + i) * ld + ro + col] = __ldg(src + (size_t)sr * ld + sc);
        }
    }
    // the matvec reads whole aligned float4 groups: up to 3 columns on either side of the block in the
    // block's own rows.  Nobody else reads those entries; zero them so that the matvec needs no selects.
    if (blockIdx.x == 0 && threadIdx.x < 8) {
        int j = threadIdx.x;
        int fc = ro + ((j < 4) ? -1 - j : n + (j - 4));
        if (fc >= 0 && fc < ld) {
            int rows = min(16, n - row0);
            for (int i = 0; i < rows; ++i) dst[(size_t)(ro + row0 + i) * ld + fc] = 0.f;
        }
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0)
        atomicAdd(&e.acct[SG_PARTITION], 8ull * n * n);
}

// Deferred affinity (segment calls with feature terms): pass 1 only queues the in-mask pairs and joins the root-level
// components; W is never written in input order.  After the root split the blocks of the ACTIVE ranges are zeroed
// with a unit diagonal here (sum n_c^2 floats instead of N^2: the zero fill was the store-bound part of the affinity
// stage, and k_gather_blocks_cur then read the whole N x N matrix once more to pick the blocks out of it) and
// k_affinity_feats scatters the queued pairs to their new positions.
// grid: (ZB_BLOCKS, active): the blocks of a node take its 16-row tiles round-robin and store 128-bit zeros over the
// 4-aligned column window that contains the block and its fringe (a grid sized by the LARGEST node of the level, as the
// gather uses, launches 3 M thread blocks for 2056 nodes of which three quarters exit at once: 1.7 ms for 3 GB of stores).
constexpr int ZB_BLOCKS = 16;
__global__ void __launch_bounds__(256)
k_zero_blocks(Eng e, int cur /* buffer the gather would read; the blocks go to the other one */) {
    int a = blockIdx.y;
    int r = e.a_rid[a];
    int start = e.r_start[r], n = e.r_n[r], c = e.r_chunk[r];
    int base = e.c_base[c], ld = e.c_ld[c];
    float* dst = cur ? e.c_W0[c] : e.c_W1[c];
    int ro = start - base;
    // fringe: four columns on either side (clipped), as in k_gather_blocks_cur
    const int c0 = max(0, (ro - 4) & ~3), c1 = min(ld, (ro + n + 7) & ~3);
    const bool vec = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
    for (int t = blockIdx.x; t * 16 < n; t += gridDim.x) {
        const int row0 = t * 16, rows = min(16, n - row0);
        if (vec) {
            const int w4 = (c1 - c0) >> 2;
            for (int idx = threadIdx.x; idx < rows * w4; idx += 256) {
                const int i = idx / w4, col = c0 + 4 * (idx - i * w4);
                const int d = ro + row0 + i;                       // column of the unit diagonal
                float4 v = make_float4(col == d ? 1.f : 0.f, col + 1 == d ? 1.f : 0.f, col + 2 == d ? 1.f : 0.f,
                                       col + 3 == d ? 1.f : 0.f);
                *reinterpret_cast<float4*>(dst + (size_t)d * ld + col) = v;
            }
        } else {
            const int w = min(ld, ro + n + 4) - max(0, ro - 4), cb = max(0, ro - 4);
            for (int idx = threadIdx.x; idx < rows * w; idx += 256) {
                const int i = idx / w, col = cb + (idx - i * w);
                const int d = ro + row0 + i;
                dst[(size_t)d * ld + col] = (col == d) ? 1.f : 0.f;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        atomicAdd(&e.acct[SG_PARTITION], 4ull * n * n);
}

// inv[old global position] = new global position, from val2[new] = old (after the sort of a rebuild)
__global__ void k_inverse_positions(Eng e, int* __restrict__ inv) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < e.P) inv[e.val2[p]] = p;
}

// ---------------------------------------------------------------------------------------------
// "Next" row N1: 1-nearest-neighbour re-projection of the 0.35 m labels onto the 5 cm points
//   (kDTree_1NN_feature_reprojection, point_cloud_utils.py:144-174; call ncuts_utils.py:185-189).
// Brute force: one thread per query point, the source points staged through shared memory in tiles
// of 1024 (float64 squared distances, first minimum wins), instead of a KD-tree query per point in a
// Python loop.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_nn_reproject(int nq, const double* __restrict__ q, int ns, const double* __restrict__ src,
               const int* __restrict__ src_label, double max_radius, int no_label,
               int* __restrict__ out_label, int* __restrict__ out_index) {
    __shared__ double sx[1024], sy[1024], sz[1024];
    int i = blockIdx.x * 256 + threadIdx.x;
    double px = 0.0, py = 0.0, pz = 0.0;
    if (i < nq) { px = q[(size_t)i * 3]; py = q[(size_t)i * 3 + 1]; pz = q[(size_t)i * 3 + 2]; }
    double best = 1e300;
    int bi = -1;
    for (int t0 = 0; t0 < ns; t0 += 1024) {
        int tn = min(1024, ns - t0);
        __syncthreads();
        for (int j = threadIdx.x; j < tn; j += 256) {
            sx[j] = src[(size_t)(t0 + j) * 3];
            sy[j] = src[(size_t)(t0 + j) * 3 + 1];
            sz[j] = src[(size_t)(t0 + j) * 3 + 2];
        }
        __syncthreads();
        if (i < nq) {
#pragma unroll 4
            for (int j = 0; j < tn; ++j) {
                double dx = px - sx[j], dy = py - sy[j], dz = pz - sz[j];
                double d = dx * dx + dy * dy + dz * dz;
                if (d < best) { best = d; bi = t0 + j; }
            }
        }
    }
    if (i < nq) {
        bool far = (max_radius > 0.0) && (sqrt(best) > max_radius);       // point_cloud_utils.py:166-168
        out_label[i] = (bi < 0 || far) ? no_label : (src_label ? src_label[bi] : bi);
        if (out_index) out_index[i] = bi;
    }
}

// final labels: label = range index relative to the chunk's first range (ncuts_utils.py:177-183)
__global__ void k_emit_labels(Eng e, int* __restrict__ labels, int* __restrict__ nseg) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= e.P) return;
    int r = e.rid[p];
    int c = e.r_chunk[r];
    int base = e.c_base[c];
    int first = e.rid[base];
    labels[base + e.perm[p]] = r - first;
    if (p == base + e.c_n[c] - 1) nseg[c] = r - first + 1;
}

}  // namespace ancuts
