// kernels_csr.cuh — front end of the recursion for caller-supplied sparse affinity graphs (ancuts_segment_csr_f32).
// The graphs arrive as one concatenated CSR (global row pointers, columns local to the row's graph).  They join the
// deferred-affinity path of the points entry where its pair stage ends: k_csr_unions builds the root-level component
// forest from the stored edges (as k_pair_unions does from the pair queue), run_rebuild splits the root, k_zero_blocks
// writes the blocks of the active ranges with a unit diagonal and k_csr_scatter puts the stored entries at the positions
// their points have after the split (as k_affinity_feats does with the queued pairs).  No n x n root matrix is written.
//
// Every kernel here gives a row to a group of CSR_LANES lanes; the lanes take its stored entries round-robin.
#pragma once
#include "common.cuh"
#include "kernels_graph.cuh"

namespace ancuts {

constexpr int CSR_LANES = 8;

// violation kinds of k_csr_validate (ancuts_segment_csr_f32 turns them into messages)
enum : int {
    CSR_OK = 0, CSR_ROWPTR = 1, CSR_ROWPTR_ENDS = 2, CSR_COLUMN = 3, CSR_UNSORTED = 4, CSR_DUPLICATE = 5,
    CSR_NONFINITE = 6, CSR_DIAGONAL = 7, CSR_NO_MIRROR = 8, CSR_ASYMMETRIC = 9
};

// First violation of a graph, as one 64-bit key for atomicMin: structural faults (row pointers, columns, order, non-finite
// values) rank before the symmetry / diagonal rules, which a structural fault elsewhere in the graph can make fail
// spuriously (a binary search into an unsorted row); within a class the smallest row wins.
__device__ __forceinline__ unsigned long long csr_err_key(int kind, int row) {
    const unsigned long long cls = (kind >= CSR_DIAGONAL) ? 1ull : 0ull;
    return (cls << 62) | ((unsigned long long)(unsigned)row << 8) | (unsigned long long)kind;
}

// {0} U [2^-126, 2) by bits: +0, or a positive normal float below 2.  -0 is outside (its sign bit would survive the integer
// widening of the matvec as a huge exponent), so are negative, denormal and >= 2 values.
__device__ __forceinline__ bool csr_in_own_range(float v) {
    const unsigned b = __float_as_uint(v);
    return b == 0u || (b >= 0x00800000u && b < 0x40000000u);
}

// Validation of the whole batch in one launch.  grid: (row blocks, graphs), block 256 = 32 rows of CSR_LANES lanes.
// err[c] (reset to ~0 by the caller) receives the smallest csr_err_key of graph c; *outside is set when a stored value lies
// outside {0} U [2^-126, 2) (the range the integer widening and the fixed-point fused cut are exact for, see cluster_mode).
//
// Bounds: the only reads are row_ptr[g] and row_ptr[g + 1] for the rows g < P of the call (the ABI gives row_ptr P + 1
// entries), col[q] / val[q] for q inside a row's [lo, hi) AFTER 0 <= lo <= hi <= nnz was checked (a row that fails is
// reported and its entries are not touched), col[q - 1] for lo < q < hi, and, for the mirror entry of (i, j), row j's
// pointers only after 0 <= j < n was checked (so base + j < P) and its entries only inside [lo2, hi2) after the same
// 0 <= lo2 <= hi2 <= nnz check.  A binary search stays inside [lo2, hi2) whatever the order of the columns there.  So no
// row_ptr / col content makes this kernel read outside the caller's arrays; k_csr_unions and k_csr_scatter run only on a
// batch that passed.
__global__ void __launch_bounds__(256)
k_csr_validate(const int* __restrict__ c_base, const int* __restrict__ c_n, int P, const int64_t* __restrict__ row_ptr,
               const int32_t* __restrict__ col, const float* __restrict__ val, long long nnz,
               unsigned long long* __restrict__ err, int* __restrict__ outside) {
    const int c = blockIdx.y;
    const int n = c_n[c], base = c_base[c];
    const int i = blockIdx.x * (256 / CSR_LANES) + threadIdx.x / CSR_LANES;
    const int sub = threadIdx.x & (CSR_LANES - 1);
    const bool live = i < n;                    // no early exit: the group reductions below need every lane of the warp
    const int g = base + (live ? i : 0);
    unsigned long long bad = ~0ull;
    bool out = false;
    if (live && sub == 0) {
        if (g == 0 && row_ptr[0] != 0) bad = min(bad, csr_err_key(CSR_ROWPTR_ENDS, i));
        if (g == P - 1 && row_ptr[P] != nnz) bad = min(bad, csr_err_key(CSR_ROWPTR_ENDS, i));
    }
    const long long lo = live ? row_ptr[g] : 0, hi = live ? row_ptr[g + 1] : 0;
    if (lo < 0 || hi < lo || hi > nnz) {
        if (sub == 0) bad = min(bad, csr_err_key(CSR_ROWPTR, i));
    } else {
        for (long long q = lo + sub; q < hi; q += CSR_LANES) {
            const int j = col[q];
            const float v = val[q];
            if (j < 0 || j >= n) { bad = min(bad, csr_err_key(CSR_COLUMN, i)); continue; }
            if (q > lo) {
                const int jp = col[q - 1];
                if (jp == j) bad = min(bad, csr_err_key(CSR_DUPLICATE, i));
                else if (jp > j) bad = min(bad, csr_err_key(CSR_UNSORTED, i));
            }
            if (!isfinite(v)) { bad = min(bad, csr_err_key(CSR_NONFINITE, i)); continue; }
            if (j == i) {
                if (v != 1.0f) bad = min(bad, csr_err_key(CSR_DIAGONAL, i));
                continue;
            }
            out |= !csr_in_own_range(v);
            // mirror entry (j, i): binary search in row j, bounds-checked as above
            const long long lo2 = row_ptr[base + j], hi2 = row_ptr[base + j + 1];
            bool found = false;
            float v2 = 0.0f;
            if (lo2 >= 0 && lo2 <= hi2 && hi2 <= nnz) {
                long long a = lo2, b = hi2;
                while (a < b) {
                    const long long m = a + ((b - a) >> 1);
                    const int cm = col[m];
                    if (cm == i) { found = true; v2 = val[m]; break; }
                    if (cm < i) a = m + 1; else b = m;
                }
            }
            if (!found) {
                if (v != 0.0f) bad = min(bad, csr_err_key(CSR_NO_MIRROR, i));      // an absent entry is 0
            } else if (__float_as_uint(v) != __float_as_uint(v2) && !(v == 0.0f && v2 == 0.0f)) {
                bad = min(bad, csr_err_key(CSR_ASYMMETRIC, i));
            }
        }
    }
    // the group's minimum, one atomic per row with a fault
#pragma unroll
    for (int o = 1; o < CSR_LANES; o <<= 1) {
        const unsigned long long t = __shfl_xor_sync(0xffffffffu, bad, o);
        bad = min(bad, t);
    }
    const bool any_out = __any_sync(0xffffffffu, out);
    if (sub == 0 && bad != ~0ull) atomicMin(err + c, bad);
    if ((threadIdx.x & 31) == 0 && any_out) atomicOr(outside, 1);
}

// Root-level components: one union per stored nonzero entry with j > i (the graph is symmetric).  uf_union hooks the larger
// root under the smaller, so every component's root is its smallest position whatever the order of the unions: the root
// split depends on the edge set only, as k_cc_union's does on the dense matrix.  grid as k_csr_validate.
__global__ void __launch_bounds__(256)
k_csr_unions(const int* __restrict__ c_base, const int* __restrict__ c_n, const int64_t* __restrict__ row_ptr,
             const int32_t* __restrict__ col, const float* __restrict__ val, int* parent) {
    const int c = blockIdx.y;
    const int n = c_n[c], base = c_base[c];
    const int i = blockIdx.x * (256 / CSR_LANES) + threadIdx.x / CSR_LANES;
    if (i >= n) return;
    const long long lo = row_ptr[base + i], hi = row_ptr[base + i + 1];
    for (long long q = lo + (threadIdx.x & (CSR_LANES - 1)); q < hi; q += CSR_LANES) {
        const int j = col[q];
        if (j > i && val[q] != 0.0f) uf_union(parent, base + i, base + j);
    }
}

// After the root split (run_rebuild, deferred branch): every stored off-diagonal entry (i, j) goes to (inv[base + i],
// inv[base + j]) of the new block when both points sit in the same ACTIVE range -- the rule k_affinity_feats applies.  The
// mirror entry writes the transposed position, so each stored entry is written once.  Stored values are copied bit for bit
// (a stored 0 included): the blocks equal what k_gather_blocks_cur would gather from the densified matrix.  The diagonal
// stays as k_zero_blocks wrote it (1).  Rows in input order (k_init_positions without an order table).  grid as above.
__global__ void __launch_bounds__(256)
k_csr_scatter(Eng e, int cur /* buffer the gather would read; the blocks go to the other one */,
              const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const float* __restrict__ val,
              const int* __restrict__ inv) {
    const int c = blockIdx.y;
    const int n = e.c_n[c], base = e.c_base[c];
    const int i = blockIdx.x * (256 / CSR_LANES) + threadIdx.x / CSR_LANES;
    if (i >= n) return;
    const int pi = inv[base + i];
    const int r = e.rid[pi];
    if (e.r_status[r] != ST_ACTIVE) return;
    float* dst = cur ? e.c_W0[c] : e.c_W1[c];
    const size_t ld = (size_t)e.c_ld[c];
    const long long lo = row_ptr[base + i], hi = row_ptr[base + i + 1];
    for (long long q = lo + (threadIdx.x & (CSR_LANES - 1)); q < hi; q += CSR_LANES) {
        const int j = col[q];
        if (j == i) continue;
        const int pj = inv[base + j];
        if (e.rid[pj] == r) dst[(size_t)(pi - base) * ld + (pj - base)] = val[q];
    }
}

}  // namespace ancuts
