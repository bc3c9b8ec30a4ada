// common.cuh — shared definitions for libautoinst_ncuts (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/autoinst_ncuts.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libautoinst_ncuts is written for sm_100a (B200) only"
#endif

namespace ancuts {

constexpr int NCUT = ANCUTS_NUM_CUTS;   // thresholds per node (normalized_cut.py:54)
constexpr int NB = NCUT + 1;            // buckets 0..NCUT
constexpr int CH = 512;                 // columns per reduction chunk (re-orthogonalisation, stats)
constexpr int ZT = 8192;                // z-tile of the matvec: 64 KB of float64 in shared memory
constexpr int KMAX_DEFAULT = 1024;
constexpr int KMAX_LIMIT = 2048;            // the check kernel keeps 8.5 arrays of kmax+2 float64 in shared memory
constexpr int CHECK_DEFAULT = 16;
constexpr double TOL_DEFAULT = 1e-10;
constexpr double CHILD_SPLIT_LIM = 0.01;   // normalized_cut.py:37 default, not forwarded at :57-58
constexpr int FIX_SHIFT = 40;              // 2^-40 fixed point for order-independent cut sums (fewer bits for huge volumes)
constexpr int CTR_COUNT = 32;              // device counters, see Eng::ctr

enum : int { ST_LEAF = 0, ST_ACTIVE = 1, ST_SPLIT = 2 };
enum : int { DONE_NO = 0, DONE_YES = 1, DONE_HOLD = 2 };

// stages for accounting
enum : int { SG_AFFINITY = 0, SG_DEGREE = 1, SG_MATVEC = 2, SG_REORTH = 3, SG_SCAN = 4, SG_PARTITION = 5, SG_COUNT = 6,
             SG_SPARSE_STEPS = 6, SG_SPARSE_NNZ = 7,     // device accounting has four more slots: sparse matvec form,
             SG_CL_STEPS = 8, SG_CL_FULL = 9,           // Lanczos steps of the cluster kernel and those with the full pass
             SG_ACCT = 10 };

void set_error(const char* fmt, ...);

#define ANCUTS_CUDA(call)                                                                     \
    do {                                                                                      \
        cudaError_t _e = (call);                                                              \
        if (_e != cudaSuccess) {                                                              \
            ancuts::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return ANCUTS_ECUDA;                                                              \
        }                                                                                     \
    } while (0)

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Block-wide sum for 256-thread blocks; result valid in every thread. `red` holds >= 8 doubles.
__device__ __forceinline__ double block_sum_256(double v, double* red) {
    v = warp_sum(v);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i];
    return t;
}

// streaming 128-bit load that does not allocate in L1 (W is read once per pass)
__device__ __forceinline__ float4 ld_stream4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// ---- mbarrier / bulk-copy (TMA) helpers -------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbarrier_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbarrier_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbarrier_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_addr_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a barrier that never completes traps instead of hanging the GPU
__device__ __forceinline__ void mbarrier_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t it = 0; it < (1u << 24); ++it)
        if (mbarrier_try_wait(bar, parity)) return;
    __trap();
}
// ---- one-way cluster exchange: a CTA stores into a peer's shared memory with st.async and the bytes are counted on the
// peer's mbarrier (complete_tx, release at cluster scope); the peer waits on its own barrier (acquire at cluster scope)
// shared::cluster address of `a` (a shared::cta address of this CTA) in the CTA of the given cluster rank
__device__ __forceinline__ uint32_t mapa_u32(uint32_t a, int rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_async_f64(uint32_t dst, double v, uint32_t bar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.f64 [%0], %1, [%2];"
                 ::"r"(dst), "d"(v), "r"(bar) : "memory");
}
__device__ __forceinline__ bool mbarrier_try_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_addr_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// 1-D bulk copy global -> shared memory of this CTA, completion counted in bytes on `bar`
// (16-byte aligned addresses, size a multiple of 16)
__device__ __forceinline__ void bulk_copy_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_addr_u32(bar)) : "memory");
}

// Every per-node / per-position array the kernels touch. Passed by value.
struct Eng {
    // sizes
    int P;            // total points in the batch
    int B;            // chunks
    int KS;           // stride of per-node Krylov arrays = kmax + 4
    int kmax;
    int check_every;
    int check_adapt;  // 1: caller left lanczos_check_every at 0, the cluster kernel places its checks adaptively
    double tol;
    double T;
    // chunk table
    const int* c_base;      // [B] first global position
    const int* c_n;         // [B]
    const int* c_ld;        // [B]
    const int* c_norig;     // [B] num_points_orig for the stop rule
    float* const* c_W0;     // [B] ping
    float* const* c_W1;     // [B] pong
    // range table (every position belongs to exactly one range)
    int* r_start; int* r_n; int* r_chunk; int* r_status; int* r_pass; /* 2 per range */ int* r_slot;
    int* r_level;
    // second copy for the rebuild
    int* q_start; int* q_n; int* q_chunk; int* q_status; int* q_level;
    // per position
    int* rid; int* rid2; int* perm; int* perm2;
    double* deg; double* sinv; double* wbuf; double* ybuf; double* ev;
    double* zbuf;           // S wbuf (input of the matvec), P + 4 entries
    uint8_t* bucket; uint8_t* side;
    int* rownnz;            // stored (non-zero) entries of every row inside its node's block, written by k_degree (or with the CSR rows)
    int* parent; int* croot;
    unsigned long long* key; unsigned long long* key2; int* val; int* val2; int* flag; int* incl;
    double* V;              // (kmax+2) rows of P
    // per active slot
    int* split_ids;       // ranges that split at this level (input of the next rebuild)
    int* a_rid; int* a_k; int* a_kcap; int* a_done; int* a_conv; int* a_slot0; int* a_nch;
    int* a_path;          // 1 = multi-launch Lanczos path (k_ritz needed), 0 = finished by the cluster kernel
    int* a_fused;         // 1 = the cluster kernel also took the cut decision of the node (cl_fused_cut): the cut kernels skip it
    int fuse_cut;         // segment calls: the sparse-form cluster kernels may fuse the cut
    int* unfused;         // active slots the cluster kernels ran but did not decide (ctr[18] entries)
    const int* sel;       // cut kernels: the slots to work on (blockIdx.y / thread index -> slot), NULL = all active slots
    int* cl_ids;          // [class][active_cap] active slots per cluster-size class
    int active_cap;
    double* a_alpha; double* a_beta;     // [slot][KS]
    double* a_y;                         // [slot][KS]
    double* a_bprev; double* a_h1; double* a_h2; int* a_need2;
    double* a_theta;                     // [slot][2]
    double* a_thr;                       // [slot][NCUT]
    double* a_sign; int* a_nocut;
    unsigned long long* a_diff;          // [slot][NB+1]
    int* a_cnt;                          // [slot][NB]
    int* a_bestk; double* a_mcut; double* a_costs; /* [slot][NCUT] */
    // chunk-slot partials
    double* p_dot;        // [cslot][KS]  first Gram-Schmidt pass
    double* p_dot2;       // [cslot][KS]  second pass
    double* p_norm;       // [cslot]
    double* p_stat;       // [cslot][4]  sum, min, max, sum of squares
    double* p_vol;        // [cslot][NB]
    // counters (device)
    int* ctr;             // CTR_COUNT ints: [0]=numRanges [1]=numActive [2]=maxActiveN [3]=cslots [4]=notDone [5]=numSplit [6]=statCount
                          // [7]=maxSplitN [8..13]=nodes per cluster class [14]=nodes for the multi-launch path
                          // [16]=eigensolver nodes that stopped unconverged (whole call, never reset between levels)
                          // [17]=nodes of the level whose cut was decided inside the cluster kernel (cl_fused_cut)
                          // [18]=nodes of the level the cluster kernels ran but left to the cut kernels (Eng::unfused)
                          // [19]=cluster-exchange waits that gave up (ANCUTS_EXCHANGE_GUARD builds only; an error)
    unsigned long long* acct;   // [SG_COUNT] algorithmic bytes
    ancuts_node_stat* stats; int stats_cap;
    int w_own;            // 1 = W holds the library's own affinities (0 or [2^-126, 2)): the matvec may widen on the integer pipe
    unsigned long long* dbg;   // optional [4 cluster sizes][8] phase cycle sums of the cluster kernel (thread 0 of rank 0), or NULL
    int w_guard;          // 1 = entries next to a block may be non-finite (caller-provided W without a gather)
    const double* pts;    // [P][3] input coordinates (chunk c at c_base[c], input order) for the Lanczos start vector, or NULL
    // node form (ANCUTS_OPT_NODE_FORM): node_csr = 1 keeps every active node as CSR rows over global positions (columns local
    // to the node, ascending; the unit diagonal and the non-zero float32 affinities only): rows of position g at
    // [csr_ptr[g], csr_ptr[g + 1]).  The dense blocks then hold only the nodes k_ncsr_densify wrote this level.
    int node_csr;
    const int* csr_ptr; const int* csr_col; const float* csr_val;
    int* dn_list; int* dn_count;          // slots k_ncsr_need lists for k_ncsr_densify
};

}  // namespace ancuts
