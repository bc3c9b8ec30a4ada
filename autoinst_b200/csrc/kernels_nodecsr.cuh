// kernels_nodecsr.cuh — recursion nodes as CSR (ANCUTS_OPT_NODE_FORM = 0, the default of the points path).
//
// Rows are global positions, columns are positions local to the row's node, every row is sorted by column and holds the
// unit diagonal and the non-zero float32 affinities of its node: exactly the entries sp_fill_rows keeps from a dense block,
// in the same order, so the degrees, the shared-memory slices and everything after them keep their bits.
//   root level: the feature pass writes one value per queued pair (queue order) and counts both directions of every pair
//               at the positions its points have after the root split, k_ncsr_pairs fills the rows, k_ncsr_sort_rows
//               sorts them;
//   later levels: k_ncsr_children compacts the parent's rows (no sort: see there);
//   degrees: ncsr_row_degree, bit-identical to row_sum_window over the dense block, inside the two kernels that write the
//            rows;
//   dense blocks: written by k_ncsr_densify for the nodes that still read dense W (k_ncsr_need lists them).
#pragma once
#include "common.cuh"
#include "kernels_graph.cuh"
#include "kernels_cluster.cuh"

namespace ancuts {

// root level: one stored entry (the unit diagonal) for every position of an ACTIVE range; cnt[P] = 0 closes the scan
__global__ void k_ncsr_diag(Eng e, int* __restrict__ cnt) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < e.P) cnt[g] = (e.r_status[e.rid[g]] == ST_ACTIVE) ? 1 : 0;
    else if (g == e.P) cnt[g] = 0;
}

// d_i = 1 + sum_j w_ij of one CSR row, bit-identical to row_sum_window over the dense block.  That function reads the row
// in 4-float windows aligned at a0 = ro & ~3 (ro = the node's offset in its chunk, pad = ro & 3: local column j sits in
// window (j + pad) >> 2), gives window w to lane w & 31 at trip w >> 5, sums a window ((x+y)+(z+w)) when it lies inside
// the block and in element order otherwise (missing entries are +0), adds the windows of a lane in trip order and reduces
// with warp_sum.  Every value is > 0 (the CSR rows store no zeros), so the windows without entries (sum +0) change nothing,
// and columns ascend, so each lane receives its windows in trip order.  The kernels that write the rows call it right
// after (one warp per row, __syncwarp between): the row is still in cache and no separate pass over the rows is needed.
__device__ __forceinline__ double ncsr_window_sum(float x0, float x1, float x2, float x3, int win, int pad, int n) {
    const int cl = 4 * win - pad;
    if (cl >= 0 && cl + 3 < n) return ((double)x0 + (double)x1) + ((double)x2 + (double)x3);
    double s = 0.0;
    s += (double)x0; s += (double)x1; s += (double)x2; s += (double)x3;
    return s;
}

// Degree, D^-1/2 and stored entries of row g (entries [b, en) of col / val, node of n points at chunk offset pad mod 4).
// wsum: this warp's 32 shared slots, all -1 on entry and on return.  Returns the bytes read (accounting).
__device__ __forceinline__ unsigned long long
ncsr_row_degree(const Eng& e, int g, const int* __restrict__ col, const float* __restrict__ val, int b, int en, int pad, int n,
                double* wsum, int lane) {
    double acc = 0.0;
    // 32 entries per batch; a window has at most four entries, so all windows but the batch's last one are complete in it,
    // and the last one is left for the next batch (which starts at its first entry)
    for (int k0 = b; k0 < en;) {
        const int k = k0 + lane;
        const bool live = k < en;
        const int q = live ? col[k] + pad : 0;
        const float v = live ? val[k] : 0.f;
        const int win = live ? (q >> 2) : -1;
        const bool more = k0 + 32 < en;
        const int wlast = __shfl_sync(0xffffffffu, win, 31);
        const bool take = live && !(more && win == wlast);
        const int wprev = __shfl_up_sync(0xffffffffu, win, 1);
        const bool head = take && (lane == 0 || wprev != win);
        float x[4];
        const int j = q & 3;
        x[0] = j == 0 ? v : 0.f; x[1] = j == 1 ? v : 0.f; x[2] = j == 2 ? v : 0.f; x[3] = j == 3 ? v : 0.f;
#pragma unroll
        for (int d = 1; d < 4; ++d) {               // the other entries of the head's window follow it
            const int wd = __shfl_down_sync(0xffffffffu, win, d), qd = __shfl_down_sync(0xffffffffu, q, d);
            const float vd = __shfl_down_sync(0xffffffffu, v, d);
            if (lane + d < 32 && wd == win) {
                const int jd = qd & 3;
                if (jd == 0) x[0] = vd; else if (jd == 1) x[1] = vd; else if (jd == 2) x[2] = vd; else x[3] = vd;
            }
        }
        // hand each window's sum to its lane (window & 31).  The windows of a batch span fewer than 32 windows in the usual
        // case, so their lanes differ; otherwise windows that share a lane go in window order (rounds)
        const int t = win & 31;
        const double sw = head ? ncsr_window_sum(x[0], x[1], x[2], x[3], win, pad, n) : 0.0;
        const int w0 = __shfl_sync(0xffffffffu, win, 0);
        int rank = 0, rounds = 1;
        if (__reduce_max_sync(0xffffffffu, head ? (unsigned)(win - w0) : 0u) >= 32u) {
            const unsigned hm = __ballot_sync(0xffffffffu, head);
            const unsigned same = __match_any_sync(0xffffffffu, head ? t : -1 - lane) & hm;
            rank = __popc(same & ((1u << lane) - 1u));
            rounds = (int)__reduce_max_sync(0xffffffffu, head ? (unsigned)rank + 1u : 0u);
        }
        for (int rr = 0; rr < rounds; ++rr) {
            if (head && rank == rr) wsum[t] = sw;
            __syncwarp();
            const double got = wsum[lane];
            if (got >= 0.0) { acc += got; wsum[lane] = -1.0; }
            __syncwarp();
        }
        if (!more) break;
        k0 += __ffs(__ballot_sync(0xffffffffu, win == wlast)) - 1;
    }
    const double sum = warp_sum(acc);
    if (lane == 0) {
        const double d = 1.0 + sum;                 // + identity (normalized_cut.py:38)
        e.deg[g] = d;
        e.sinv[g] = 1.0 / sqrt(d);                  // :43
        e.rownnz[g] = en - b;                       // every stored entry is non-zero
    }
    return 8ull * (unsigned long long)(en - b) + 8ull;      // column + value per entry, two row pointers
}

// root level, grid (blocks, chunks): every queued pair with a non-zero value goes to both rows through the rows' fill
// cursors (the feature pass counted them, k_ncsr_fill_diag set the cursors).  A value of 0 is a pair whose range does not
// go on (the feature pass skips it) or whose exp underflowed: the dense block holds a 0 there and sp_fill_rows drops it, so
// it is not stored.  The test is the feature pass's counting test.
__global__ void __launch_bounds__(256)
k_ncsr_pairs(const PairQ* __restrict__ q_all, const long long* __restrict__ q_off, const int* __restrict__ q_cap,
             const int* __restrict__ qctr_all, const int* __restrict__ c_base, const float* __restrict__ slot, Eng e,
             const int* __restrict__ inv, int* __restrict__ cursor, int* __restrict__ col, float* __restrict__ val) {
    const int c = blockIdx.y;
    if (qctr_all[2 * c + 1]) return;
    const int total = min(qctr_all[2 * c], q_cap[c]);
    const PairQ* q = q_all + q_off[c];
    const float* s = slot + q_off[c];
    const int base = c_base[c];
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        const float w = s[t];
        if (w == 0.0f) continue;
        const PairQ p = q[t];
        const int gi = inv[base + p.i], gj = inv[base + p.j];
        const int r = e.rid[gi];
        if (e.rid[gj] != r) continue;               // never taken: a queued pair is one component, the root split keeps it whole
        const int st = e.r_start[r];
        const int a = atomicAdd(cursor + gi, 1), b = atomicAdd(cursor + gj, 1);
        col[a] = gj - st; val[a] = w;
        col[b] = gi - st; val[b] = w;
    }
}

// root level: the diagonal goes first, cursor[g] = next free entry of row g
__global__ void k_ncsr_fill_diag(Eng e, const int* __restrict__ ptr, int* __restrict__ cursor, int* __restrict__ col,
                                 float* __restrict__ val) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= e.P) return;
    const int r = e.rid[g];
    if (e.r_status[r] != ST_ACTIVE) return;
    const int p = ptr[g];
    col[p] = g - e.r_start[r];
    val[p] = 1.0f;
    cursor[g] = p + 1;
}

// root level: rows sorted by column (the fill order is the atomics' order), then the row's degree.  One warp per row;
// columns of a row are distinct.  A row whose columns span fewer than 1024 values (the cell-sorted root order keeps a
// point's neighbours close: the usual case) ranks its entries through a 1024-bit map in shared memory (a popcount prefix
// over the 32 words); other rows count, for every entry, the entries with a smaller column.
__global__ void __launch_bounds__(256)
k_ncsr_sort_rows(Eng e, const int* __restrict__ ptr, const int* __restrict__ col_in, const float* __restrict__ val_in,
                 int* __restrict__ col_out, float* __restrict__ val_out) {
    __shared__ unsigned bits[8][32];
    __shared__ double wsum[8][32];
    __shared__ unsigned long long bytes;
    const int warp = threadIdx.x >> 5, g = blockIdx.x * 8 + warp, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) bytes = 0;
    wsum[warp][lane] = -1.0;
    __syncthreads();
    const int b = (g < e.P) ? ptr[g] : 0, n = (g < e.P) ? ptr[g + 1] - b : 0;
    if (n > 0) {                                    // warp-uniform; rows of ranges that do not go on are empty
        int lo = INT_MAX, hi = -1;
        for (int k = lane; k < n; k += 32) { const int c = col_in[b + k]; lo = min(lo, c); hi = max(hi, c); }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if (hi - lo < 1024) {
            bits[warp][lane] = 0u;
            __syncwarp();
            for (int k = lane; k < n; k += 32) { const int c = col_in[b + k] - lo; atomicOr(&bits[warp][c >> 5], 1u << (c & 31)); }
            __syncwarp();
            const unsigned mine = bits[warp][lane];
            int incl = __popc(mine);
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            const int excl = incl - __popc(mine);
            for (int k0 = 0; k0 < n; k0 += 32) {
                const int k = k0 + lane;
                const int c = (k < n) ? col_in[b + k] - lo : 0;
                const int before = __shfl_sync(0xffffffffu, excl, c >> 5);
                const unsigned word = __shfl_sync(0xffffffffu, mine, c >> 5);
                if (k < n) {
                    const int rank = before + __popc(word & ((1u << (c & 31)) - 1u));
                    col_out[b + rank] = c + lo;
                    val_out[b + rank] = val_in[b + k];
                }
            }
        } else {
            for (int k0 = 0; k0 < n; k0 += 32) {
                const int k = k0 + lane;
                const int ck = (k < n) ? col_in[b + k] : INT_MAX;
                int rank = 0;
                for (int j0 = 0; j0 < n; j0 += 32) {
                    const int cj = (j0 + lane < n) ? col_in[b + j0 + lane] : INT_MAX;
                    const int m = min(32, n - j0);
#pragma unroll 4
                    for (int s = 0; s < m; ++s) rank += (__shfl_sync(0xffffffffu, cj, s) < ck) ? 1 : 0;
                }
                if (k < n) { col_out[b + rank] = ck; val_out[b + rank] = val_in[b + k]; }
            }
        }
        __syncwarp();                               // the sorted row is visible to the whole warp
        const int r = e.rid[g];
        const int start = e.r_start[r];
        const unsigned long long by = ncsr_row_degree(e, g, col_out, val_out, b, b + n, (start - e.c_base[e.r_chunk[r]]) & 3,
                                                      e.r_n[r], wsum[warp], lane);
        if (lane == 0) atomicAdd(&bytes, by);
    }
    __syncthreads();
    if (threadIdx.x == 0 && bytes) atomicAdd(&e.acct[SG_DEGREE], bytes);
}

// Later levels: the rows of every new ACTIVE range from its parent's rows (run_rebuild after the table swap: rid / r_* are
// the new table, rid2 / q_* the previous one, val2[new position] = old position, inv[old position] = new position).  An
// entry stays when both ends are in the same child.  The rebuild's sort is stable and keyed by (range, side, component),
// so inside a child the new positions keep the order of the old ones: the kept entries of a sorted parent row are sorted,
// no re-sort is needed.  One warp per new row; !FILL writes the entry count, FILL compacts in order (ballot prefix) and
// then takes the row's degree.
template <bool FILL>
__global__ void __launch_bounds__(256)
k_ncsr_children(Eng e, const int* __restrict__ inv, const int* __restrict__ optr, const int* __restrict__ ocol,
                const float* __restrict__ oval, int* __restrict__ cnt_or_ptr, int* __restrict__ ncol,
                float* __restrict__ nval) {
    __shared__ double wsum[8][32];
    __shared__ unsigned long long bytes;
    const int warp = threadIdx.x >> 5, p = blockIdx.x * 8 + warp, lane = threadIdx.x & 31;
    if (FILL) {
        if (threadIdx.x == 0) bytes = 0;
        wsum[warp][lane] = -1.0;
        __syncthreads();
    }
    int r = -1;
    if (p < e.P) r = e.rid[p];
    if (r >= 0 && e.r_status[r] != ST_ACTIVE) r = -1;
    if (r < 0) {
        if (!FILL && lane == 0 && p <= e.P) cnt_or_ptr[p] = 0;
    } else {                                        // warp-uniform
    const int go = e.val2[p];
    const int ostart = e.q_start[e.rid2[go]];
    const int nstart = e.r_start[r];
    const int b = optr[go], en = optr[go + 1];
    int out = FILL ? cnt_or_ptr[p] : 0;
    for (int k0 = b; k0 < en; k0 += 32) {
        const int k = k0 + lane;
        bool keep = false;
        int c = 0;
        if (k < en) {
            const int gc = inv[ostart + ocol[k]];
            keep = e.rid[gc] == r;
            c = gc - nstart;
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (FILL && keep) {
            const int o = out + __popc(m & ((1u << lane) - 1u));
            ncol[o] = c;
            nval[o] = oval[k];
        }
        out += __popc(m);
    }
    if (!FILL && lane == 0) cnt_or_ptr[p] = out;
    if (FILL) {
        __syncwarp();                               // the new row is visible to the whole warp
        const int b2 = cnt_or_ptr[p];
        const unsigned long long by = ncsr_row_degree(e, p, ncol, nval, b2, out, (nstart - e.c_base[e.r_chunk[r]]) & 3,
                                                      e.r_n[r], wsum[warp], lane);
        if (lane == 0) atomicAdd(&bytes, by);
    }
    }
    if (FILL) {
        __syncthreads();
        if (threadIdx.x == 0 && bytes) atomicAdd(&e.acct[SG_DEGREE], bytes);
    }
}

// The nodes of the level that read dense W: all of them (all != 0: the grid-wide Lanczos path takes over), those above
// CL_NMAX points, and those whose CSR slice would not fit one CTA's shared memory in the cluster kernel (the same test as
// its prologue, with the cluster size the host maps the node's size bin to: cmap holds 4 bits per bin).  One block per slot.
__global__ void __launch_bounds__(256)
k_ncsr_need(Eng e, int all, unsigned cmap, int* __restrict__ list, int* __restrict__ count) {
    __shared__ int tot[8];
    const int a = blockIdx.x;
    const int r = e.a_rid[a];
    const int start = e.r_start[r], n = e.r_n[r];
    bool need = all != 0 || n > CL_NMAX;
    if (!need) {
        const int C = (int)((cmap >> (4 * cluster_class(n))) & 15u);
        const int rp = (n + C - 1) / C;
        if (threadIdx.x < 8) tot[threadIdx.x] = 0;
        __syncthreads();
        int part[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int q = (e.rownnz[start + i] + 3) & ~3;
#pragma unroll
            for (int k = 0; k < 8; ++k) part[k] += (i / rp == k) ? q : 0;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) if (k < C && part[k]) atomicAdd(&tot[k], part[k]);
        __syncthreads();
        const int nz = (n + 8 + 3) & ~3;
        for (int k = 0; k < C; ++k) {
            const int r0 = min(n, k * rp), nr = min(n, r0 + rp) - r0;
            const int ptr_d = (((nr + 1 + 1) / 2) + 1) & ~1, val_d = (tot[k] + 1) / 2, col_d = (tot[k] + 3) / 4;
            if (nz + ptr_d + val_d + col_d > CL_DYN_SMEM / 8) need = true;
        }
    }
    if (need && threadIdx.x == 0) list[atomicAdd(count, 1)] = a;
}

// Dense blocks of the listed slots from their CSR rows, in the buffer node_view(e, r, cur) reads: zeros over the 4-aligned
// window with its fringe and the unit diagonal (as k_zero_blocks), then the stored entries.  grid: (ZB_BLOCKS, active);
// blocks past the list's length exit.
__global__ void __launch_bounds__(256)
k_ncsr_densify(Eng e, int cur, const int* __restrict__ list, const int* __restrict__ count) {
    if ((int)blockIdx.y >= *count) return;
    const int a = list[blockIdx.y];
    const int r = e.a_rid[a];
    const int start = e.r_start[r], n = e.r_n[r], c = e.r_chunk[r];
    const int base = e.c_base[c], ld = e.c_ld[c];
    float* dst = cur ? e.c_W1[c] : e.c_W0[c];
    const int ro = start - base;
    const int c0 = max(0, (ro - 4) & ~3), c1 = min(ld, (ro + n + 7) & ~3);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t = blockIdx.x; t * 16 < n; t += gridDim.x) {
        const int row0 = t * 16, rows = min(16, n - row0);
        const int w = c1 - c0;
        for (int idx = threadIdx.x; idx < rows * w; idx += 256) {
            const int i = idx / w, col = c0 + (idx - i * w);
            const int d = ro + row0 + i;
            dst[(size_t)d * ld + col] = (col == d) ? 1.f : 0.f;
        }
        __syncthreads();
        for (int i = warp; i < rows; i += 8) {
            const int g = start + row0 + i;
            float* rowp = dst + (size_t)(ro + row0 + i) * ld + ro;
            for (int k = e.csr_ptr[g] + lane; k < e.csr_ptr[g + 1]; k += 32) rowp[e.csr_col[k]] = e.csr_val[k];
        }
        __syncthreads();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        atomicAdd(&e.acct[SG_PARTITION], 4ull * n * n);
}

}  // namespace ancuts
