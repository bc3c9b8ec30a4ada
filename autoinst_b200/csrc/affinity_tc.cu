// affinity_tc.cu — stage 1 with the TARL feature Gram matrix on the tcgen05 tensor cores.
//   Replaces cdist(tarl, tarl) (ncuts_utils.py:144) by  td^2 = |f_i|^2 + |f_j|^2 - 2 f_i.f_j  with the
//   dot products computed by tcgen05.mma (kind::tf32, fp32 accumulators in TMEM), operands staged in
//   shared memory by TMA (cp.async.bulk.tensor, 128-byte swizzle).  The spatial float64 test, the zero-row
//   rule, the DINOv2 term and the exp are fused in the epilogue of the same tile (ncuts_utils.py:60-66,
//   125-133,145-156).
// Accuracy (north_star: 1e-5 relative): each feature is split f = hi + lo with hi = round-to-tf32(f),
//   lo = f - hi, and the tile needs hi.hi + hi.lo + lo.hi (3 x TF32, error ~2^-21 |f_i||f_j|).  Measured on
//   B200: accumulating all 36 MMAs into one TMEM accumulator loses ~0.5 ulp(|acc|) per MMA (1.7e-5 relative
//   error of W).  So every K = 8 slice of hi.hi gets its OWN accumulator (one MMA, no accumulation, 12 x 32
//   TMEM columns) and the small cross terms share a 13th; the epilogue adds the 13 partials in float64.
//   Pairs whose squared distance cancels below 1 % of |f_i|^2 + |f_j|^2 are re-evaluated by direct differences, and so
//   are pairs whose distance is small against theta (|f_i|^2 + |f_j|^2): the error of d^2 is relative to the norms
//   (measured on B200: up to ~8e-8 (|f_i|^2 + |f_j|^2)), W's relative error is theta err(d^2) / (2 td), and at TARL rows
//   ten times the synthetic norm it reached 3e-5 with the 1 % rule alone (tests/test_gpu_affinity_edges.py).
// One CTA (128 threads) per 128 x 32 output tile:
//   thread 0: mbarrier init, TMA loads of the four operand tiles, 36 MMAs (K = 96 = 3 swizzle atoms x 4),
//             tcgen05.commit;   warp 0: TMEM alloc/dealloc (512 columns);
//   all 4 warps: tcgen05.ld of their 32 TMEM lanes (one output row per thread), epilogue, staging in shared
//             memory, coalesced 128-bit stores of W.
#include <cuda.h>
#include "common.cuh"

namespace ancuts {

constexpr int TC_M = 128;            // rows per tile (UMMA M)
constexpr int TC_N = 32;             // columns per tile (UMMA N)
constexpr int TC_TMEM_COLS = 512;    // 12 hi.hi partial accumulators + 1 cross-term accumulator, 32 columns each
constexpr int TC_KB = 32;            // fp32 elements per 128-byte swizzle atom
constexpr int TC_UK = 8;             // K of one tf32 MMA
constexpr int TC_MAXKB = 3;          // up to 96 feature dimensions resident (TARL); shared memory bound

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a barrier that never completes traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t it = 0; it < (1u << 28); ++it)
        if (mbar_try_wait(bar, parity)) return;
    __trap();
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ uint64_t umma_desc_sw128(const void* smem_ptr) {
    // K-major, 128-byte swizzle: LBO = 1 (unused), SBO = 1024 B between 8-row groups, version 1 (sm_100)
    uint64_t a = (uint64_t)((smem_u32(smem_ptr) >> 4) & 0x3FFF);
    return a | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

// ---- operand preparation: hi/lo split, zero padding to (n_pad x kp), squared norms in float64 ------
__global__ void __launch_bounds__(256)
k_tc_prepare(int n, int n_pad, int dim, int kp, const float* __restrict__ f, float* __restrict__ hi,
             float* __restrict__ lo, double* __restrict__ nrm) {
    int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= n_pad) return;
    double s = 0.0;
    for (int k = lane; k < kp; k += 32) {
        float v = (row < n && k < dim) ? f[(size_t)row * dim + k] : 0.0f;
        uint32_t hb;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(v));
        float h = __uint_as_float(hb);
        hi[(size_t)row * kp + k] = h;
        lo[(size_t)row * kp + k] = v - h;
        s += (double)v * (double)v;
    }
    s = warp_sum(s);
    if (lane == 0 && row < n) nrm[row] = s;
}

struct TcParams {
    int n, tdim, ddim, kb_count;
    double alpha, theta, gamma, prox;
    const double* pts;
    const float* tarl;
    const float* dino;
    const uint8_t* tarl_zero;
    const double* nrm;
    float* W;
    long long ld;
};

__global__ void __launch_bounds__(128, 1)
k_affinity_tc(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, TcParams P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte aligned operand tiles (swizzle-128B requirement)
    uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int KB = P.kb_count;
    float* a_hi = (float*)base;                                   // KB x [128 rows x 128 B]
    float* a_lo = a_hi + (size_t)KB * TC_M * TC_KB;
    float* b_hi = a_lo + (size_t)KB * TC_M * TC_KB;               // KB x [64 rows x 128 B]
    float* b_lo = b_hi + (size_t)KB * TC_N * TC_KB;
    float* stage = b_lo + (size_t)KB * TC_N * TC_KB;              // 128 x 65 floats output staging
    double* prow = (double*)(stage + TC_M * (TC_N + 1) + 1);      // 128 x 3
    prow = (double*)(((uintptr_t)prow + 15) & ~(uintptr_t)15);
    double* pcol = prow + TC_M * 3;                               // TC_N x 3
    double* ncol = pcol + TC_N * 3;                               // TC_N squared norms
    double* gsum = ncol + TC_N;                                   // 128 x (TC_N + 1) dot products in float64
    __shared__ __align__(8) uint64_t bar_tma, bar_mma;
    __shared__ uint32_t tmem_base_slot;
    __shared__ uint8_t zcol[TC_N];

    const int tid = threadIdx.x, warp = tid >> 5;
    const int row0 = blockIdx.y * TC_M, col0 = blockIdx.x * TC_N;
    const int n = P.n;

    if (tid == 0) {
        mbar_init(&bar_tma, 1);
        mbar_init(&bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "n"(TC_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    // points / norms / zero flags of the tile (overlaps with the TMA loads issued below)
    for (int i = tid; i < TC_M * 3; i += 128) {
        int gr = row0 + i / 3;
        prow[i] = gr < n ? P.pts[(size_t)gr * 3 + i % 3] : 1e30;
    }
    for (int i = tid; i < TC_N * 3; i += 128) {
        int gc = col0 + i / 3;
        pcol[i] = gc < n ? P.pts[(size_t)gc * 3 + i % 3] : -1e30;
    }
    if (tid < TC_N) {
        int gc = col0 + tid;
        ncol[tid] = gc < n ? P.nrm[gc] : 0.0;
        zcol[tid] = (gc < n && P.tarl_zero) ? P.tarl_zero[gc] : 0;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_acc = tmem_base_slot;

    if (tid == 0) {
        const uint32_t bytes = (uint32_t)KB * (2 * TC_M + 2 * TC_N) * TC_KB * 4;
        mbar_expect_tx(&bar_tma, bytes);
        for (int kb = 0; kb < KB; ++kb) {
            // A tiles: four 32-row boxes each (the tensor maps carry a 32 x 32 box)
            for (int q = 0; q < TC_M / 32; ++q) {
                tma_load_2d(a_hi + (size_t)kb * TC_M * TC_KB + q * 32 * TC_KB, &map_hi, &bar_tma, kb * TC_KB, row0 + q * 32);
                tma_load_2d(a_lo + (size_t)kb * TC_M * TC_KB + q * 32 * TC_KB, &map_lo, &bar_tma, kb * TC_KB, row0 + q * 32);
            }
            tma_load_2d(b_hi + (size_t)kb * TC_N * TC_KB, &map_hi, &bar_tma, kb * TC_KB, col0);
            tma_load_2d(b_lo + (size_t)kb * TC_N * TC_KB, &map_lo, &bar_tma, kb * TC_KB, col0);
        }
        mbar_wait(&bar_tma, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // instruction descriptor: D = F32, A = B = TF32, both K-major, N = 64, M = 128
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TC_N >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
        uint32_t acc = 0;
        for (int kb = 0; kb < KB; ++kb) {
#pragma unroll
            for (int k = 0; k < TC_KB / TC_UK; ++k) {
                const size_t ko = (size_t)k * TC_UK;      // floats inside the 128-byte atom
                uint64_t dah = umma_desc_sw128(a_hi + (size_t)kb * TC_M * TC_KB + ko);
                uint64_t dal = umma_desc_sw128(a_lo + (size_t)kb * TC_M * TC_KB + ko);
                uint64_t dbh = umma_desc_sw128(b_hi + (size_t)kb * TC_N * TC_KB + ko);
                uint64_t dbl = umma_desc_sw128(b_lo + (size_t)kb * TC_N * TC_KB + ko);
                umma_tf32(tmem_acc + (uint32_t)(kb * 4 + k) * TC_N, dah, dbh, idesc, 0);     // own accumulator
                umma_tf32(tmem_acc + 12 * TC_N, dah, dbl, idesc, acc);                         // cross terms
                acc = 1;
                umma_tf32(tmem_acc + 12 * TC_N, dal, dbh, idesc, 1);
            }
        }
        umma_commit(&bar_mma);
    }
    __syncwarp();
    mbar_wait(&bar_mma, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue: thread = one row of the tile (TMEM lane), 64 columns ----
    const int r = tid;
    const int gi = row0 + r;
    float* srow = stage + (size_t)r * (TC_N + 1);
    double* grow = gsum + (size_t)r * (TC_N + 1);
    {
        double gs[TC_N];
#pragma unroll
        for (int c = 0; c < TC_N; ++c) gs[c] = 0.0;
        const uint32_t taddr = tmem_acc + ((uint32_t)(warp * 32) << 16);
        const int parts = KB * 4;
        for (int part = 0; part <= 12; ++part) {
            if (part < 12 && part >= parts) continue;           // unused hi.hi slices (feature dimension < 96)
            uint32_t g32[32];
            tmem_ld32(taddr + (uint32_t)part * TC_N, g32);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < TC_N; ++c) gs[c] += (double)__uint_as_float(g32[c]);
        }
#pragma unroll
        for (int c = 0; c < TC_N; ++c) grow[c] = gs[c];
    }
    const double px = prow[r * 3], py = prow[r * 3 + 1], pz = prow[r * 3 + 2];
    const double ni = gi < n ? P.nrm[gi] : 0.0;
    const bool zi = (gi < n && P.tarl_zero) ? (P.tarl_zero[gi] != 0) : false;
    const float ox = (float)(px - prow[0]), oy = (float)(py - prow[1]), oz = (float)(pz - prow[2]);
    const float lim32 = (float)((P.prox + 1e-2) * (P.prox + 1e-2) * 1.001);
    // direct differences below td = 2e-2 theta (|f_i|^2 + |f_j|^2): W's relative error stays below 25 x the relative
    // error of d^2 (~2e-6) at any feature scale
    const double near_rel = 2e-2 * P.theta;
#pragma unroll 2
    for (int c = 0; c < TC_N; ++c) {
        float out = 0.0f;
        const int gj = col0 + c;
        // float32 pre-filter relative to the first row point; exact float64 test for the candidates
        float fx = ox - (float)(pcol[c * 3] - prow[0]), fy = oy - (float)(pcol[c * 3 + 1] - prow[1]), fz = oz - (float)(pcol[c * 3 + 2] - prow[2]);
        if (gi < n && gj < n && !(fx * fx + fy * fy + fz * fz > lim32)) {
            double dx = px - pcol[c * 3], dy = py - pcol[c * 3 + 1], dz = pz - pcol[c * 3 + 2];
            double s = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
            double sd = __dsqrt_rn(s);
            if (sd <= P.prox) {                                           // ncuts_utils.py:61
                double arg = P.alpha != 0.0 ? P.alpha * sd : 0.0;
                if (P.theta != 0.0) {
                    double td = 0.0;
                    if (!(zi || zcol[c])) {                               // :145-146
                        double nsum = ni + ncol[c];
                        double d2 = nsum - 2.0 * grow[c];
                        if (gi == gj) {
                            d2 = 0.0;
                        } else if (d2 < 1e-2 * nsum || d2 < (near_rel * nsum) * (near_rel * nsum)) {   // direct differences
                            const float* fa = P.tarl + (size_t)gi * P.tdim;
                            const float* fb = P.tarl + (size_t)gj * P.tdim;
                            double acc2 = 0.0;
                            for (int k = 0; k < P.tdim; ++k) { double d = (double)fa[k] - (double)fb[k]; acc2 += d * d; }
                            d2 = acc2;
                        }
                        td = sqrt(fmax(d2, 0.0));
                    }
                    arg += P.theta * td;
                }
                if (P.gamma != 0.0 && P.dino != nullptr) {                // :129-133 (direct, masked pairs only)
                    const float* fa = P.dino + (size_t)gi * P.ddim;
                    const float* fb = P.dino + (size_t)gj * P.ddim;
                    double acc2 = 0.0;
                    for (int k = 0; k < P.ddim; ++k) { double d = (double)fa[k] - (double)fb[k]; acc2 += d * d; }
                    arg += P.gamma * sqrt(acc2);
                }
                out = (float)exp(-arg);
            }
        }
        srow[c] = out;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    // coalesced stores: 8 threads per row (4 floats each), 16 rows per pass
    for (int rr = tid >> 3; rr < TC_M; rr += 16) {
        int gr = row0 + rr;
        int gc = col0 + (tid & 7) * 4;
        if (gr < n && gc < P.ld) {
            const float* s = stage + (size_t)rr * (TC_N + 1) + (tid & 7) * 4;
            *reinterpret_cast<float4*>(P.W + (size_t)gr * P.ld + gc) = make_float4(s[0], s[1], s[2], s[3]);
        }
    }
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "n"(TC_TMEM_COLS));
    }
}

static size_t tc_smem_bytes(int kb) {
    size_t operands = (size_t)kb * (2 * TC_M + 2 * TC_N) * TC_KB * 4;
    size_t stage = (size_t)TC_M * (TC_N + 1) * 4 + 16;
    size_t pts = (size_t)(TC_M * 3 + TC_N * 3 + TC_N + TC_M * (TC_N + 1)) * 8 + 16;
    return 1024 + operands + stage + pts;
}

size_t affinity_tc_scratch_bytes(int n, int tdim, int ddim) {
    (void)ddim;
    if (tdim <= 0) return 0;
    size_t n_pad = ((size_t)n + TC_M - 1) / TC_M * TC_M;
    size_t kp = ((size_t)tdim + TC_KB - 1) / TC_KB * TC_KB;
    return 2 * n_pad * kp * 4 + n_pad * 8 + 1024;
}

int launch_affinity_tc(int n, const double* pts, const float* tarl, int tdim, const float* dino, int ddim,
                       const uint8_t* tarl_zero, double alpha, double theta, double gamma, double prox,
                       float* W, long long ld, void* scratch, size_t scratch_bytes, cudaStream_t st) {
    if (!tarl || theta == 0.0) {
        set_error("affinity_impl=1 needs the TARL term (theta != 0): the tensor-core path computes the TARL Gram matrix");
        return ANCUTS_EUNSUPPORTED;
    }
    const int kb = (tdim + TC_KB - 1) / TC_KB;
    if (kb > TC_MAXKB) { set_error("affinity_impl=1 supports up to %d TARL dimensions", TC_MAXKB * TC_KB); return ANCUTS_EUNSUPPORTED; }
    if (scratch_bytes < affinity_tc_scratch_bytes(n, tdim, ddim) || !scratch) { set_error("tensor-core affinity: scratch too small"); return ANCUTS_EINVAL; }
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return ANCUTS_ECUDA; }
    const size_t n_pad = ((size_t)n + TC_M - 1) / TC_M * TC_M;
    const size_t kp = (size_t)kb * TC_KB;
    uintptr_t sb = ((uintptr_t)scratch + 255) & ~(uintptr_t)255;
    float* hi = (float*)sb;
    float* lo = hi + n_pad * kp;
    double* nrm = (double*)(lo + n_pad * kp);
    k_tc_prepare<<<(unsigned)((n_pad + 7) / 8), 256, 0, st>>>(n, (int)n_pad, tdim, (int)kp, tarl, hi, lo, nrm);
    CUtensorMap mh, ml;
    cuuint64_t dims[2] = {(cuuint64_t)kp, (cuuint64_t)n_pad};
    cuuint64_t strides[1] = {(cuuint64_t)kp * 4};
    cuuint32_t box[2] = {(cuuint32_t)TC_KB, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r1 = enc(&mh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, hi, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult r2 = enc(&ml, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, lo, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d, %d)", (int)r1, (int)r2); return ANCUTS_ECUDA; }
    const size_t smem = tc_smem_bytes(kb);
    static bool attr_set = false;
    if (!attr_set) {
        ANCUTS_CUDA(cudaFuncSetAttribute(k_affinity_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes(TC_MAXKB)));
        attr_set = true;
    }
    TcParams P;
    P.n = n; P.tdim = tdim; P.ddim = ddim; P.kb_count = kb;
    P.alpha = alpha; P.theta = theta; P.gamma = gamma; P.prox = prox;
    P.pts = pts; P.tarl = tarl; P.dino = (gamma != 0.0) ? dino : nullptr; P.tarl_zero = tarl_zero; P.nrm = nrm; P.W = W; P.ld = ld;
    dim3 grid((unsigned)((ld + TC_N - 1) / TC_N), (unsigned)(n_pad / TC_M));
    k_affinity_tc<<<grid, 128, smem, st>>>(mh, ml, P);
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

}  // namespace ancuts
