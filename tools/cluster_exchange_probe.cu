// cluster_exchange_probe.cu — cost of one cluster-wide exchange of a float64 partial, at the occupancy of
// k_lanczos_cluster (512 threads, one CTA per SM through ~194 KB of dynamic shared memory), for clusters of 2, 4 and 8.
//   form 0  pull:      tid 0 writes its partial to shared memory, cluster barrier, every thread reads the C partials
//                      through distributed shared memory (what the Lanczos step did twice per step)
//   form 1  pull + z:  as 0, and first every thread stores one float64 of z into every CTA (plain remote stores,
//                      published by the barriers)
//   form 2  push:      tid 0 posts expect_tx(8 C) on the local mbarrier and st.async's its partial into slot [rank] of
//                      every CTA (itself included); every thread waits on the local mbarrier and sums its slots.  Rounds
//                      alternate between two barriers and slot rows, as the Lanczos step alternates its alpha and norm
//                      exchanges: a peer's push of round r + 2 needs our push of round r + 1, which follows our wait of
//                      round r, so no push lands in a phase it does not belong to.
//   form 3  push + z:  as 2, and every thread st.async's one float64 of z into every CTA, counted as complete_tx bytes
// Every round ends with a block barrier, as every step of the Lanczos kernel does.  Prints cycles per exchange
// (thread 0 of rank 0, clock64) and ns per exchange (CUDA events over the whole grid).
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o probe tools/cluster_exchange_probe.cu
#include <cooperative_groups.h>
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
namespace cg = cooperative_groups;

constexpr int THREADS = 512;
constexpr int DYN = 194 * 1024;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s -> %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

__device__ __forceinline__ uint32_t sa(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa(uint32_t a, uint32_t r) {
    uint32_t o; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(o) : "r"(a), "r"(r)); return o;
}
__device__ __forceinline__ void st_async(uint32_t dst, double v, uint32_t bar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.f64 [%0], %1, [%2];" ::"r"(dst), "d"(v), "r"(bar) : "memory");
}
__device__ __forceinline__ bool try_wait(uint32_t bar, uint32_t ph) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(ph) : "memory");
    return ok != 0;
}

template <int C, int FORM>
__global__ void __launch_bounds__(THREADS, 1) k_probe(int rounds, long long* cyc, double* sink) {
    extern __shared__ __align__(16) double zs[];
    __shared__ double slot[2][8];
    __shared__ __align__(8) uint64_t bar[2];
    cg::cluster_group cl = cg::this_cluster();
    const int rank = (int)cl.block_rank(), tid = threadIdx.x;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(sa(&bar[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(sa(&bar[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    cl.sync();
    double val = 1.0 + rank, acc = 0.0;
    const long long t0 = clock64();
    for (int it = 0; it < rounds; ++it) {
        double s = 0.0;
        if (FORM <= 1) {
            if (FORM == 1) {
#pragma unroll
                for (int r = 0; r < C; ++r) cl.map_shared_rank(zs, r)[rank * THREADS + tid] = val;
            }
            if (tid == 0) slot[it & 1][0] = val;
            cl.sync();
#pragma unroll
            for (int r = 0; r < C; ++r) s += cl.map_shared_rank(&slot[it & 1][0], r)[0];
        } else {
            const int b = it & 1;
            const uint32_t ph = (uint32_t)(it >> 1) & 1u;
            if (tid == 0) {
                const uint32_t bytes = 8u * C + (FORM == 3 ? 8u * THREADS * C : 0u);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sa(&bar[b])), "r"(bytes) : "memory");
#pragma unroll
                for (int r = 0; r < C; ++r) st_async(mapa(sa(&slot[b][rank]), r), val, mapa(sa(&bar[b]), r));
            }
            if (FORM == 3) {
#pragma unroll
                for (int r = 0; r < C; ++r) st_async(mapa(sa(zs + rank * THREADS + tid), r), val, mapa(sa(&bar[b]), r));
            }
            while (!try_wait(sa(&bar[b]), ph)) {}
#pragma unroll
            for (int r = 0; r < C; ++r) s += slot[b][r];
        }
        __syncthreads();   // every thread has read the slots before the next round's pushes can land
        val = s * 0.5;
        acc += s;
    }
    const long long t1 = clock64();
    if (tid == 0 && rank == 0 && blockIdx.x == 0) *cyc = t1 - t0;
    if (tid == 0) sink[blockIdx.x] = acc + zs[tid];
    cl.sync();
}

template <int C, int FORM>
int run(int nsm, int rounds, long long* dcyc, double* dsink) {
    auto kern = k_probe<C, FORM>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, DYN));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((nsm / C) * C);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = DYN;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    for (int w = 0; w < 2; ++w) CK(cudaLaunchKernelEx(&cfg, kern, 100, dcyc, dsink));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    float best = 1e30f; long long bcyc = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CK(cudaEventRecord(e0));
        CK(cudaLaunchKernelEx(&cfg, kern, rounds, dcyc, dsink));
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
        long long cyc; CK(cudaMemcpy(&cyc, dcyc, sizeof(cyc), cudaMemcpyDeviceToHost));
        if (ms < best) { best = ms; bcyc = cyc; }
    }
    static const char* names[4] = {"pull", "pull+z", "push", "push+z"};
    printf("{\"C\": %d, \"form\": \"%s\", \"ctas\": %d, \"rounds\": %d, \"cycles_per_exchange\": %.1f, \"ns_per_exchange\": %.1f}\n",
           C, names[FORM], (nsm / C) * C, rounds, (double)bcyc / rounds, best * 1e6 / rounds);
    return 0;
}

template <int C>
int run_all(int nsm, int rounds, long long* dcyc, double* dsink) {
    int rc = 0;
    rc |= run<C, 0>(nsm, rounds, dcyc, dsink);
    rc |= run<C, 1>(nsm, rounds, dcyc, dsink);
    rc |= run<C, 2>(nsm, rounds, dcyc, dsink);
    rc |= run<C, 3>(nsm, rounds, dcyc, dsink);
    return rc;
}

int main() {
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, 0));
    printf("{\"device\": \"%s\", \"sms\": %d}\n", p.name, p.multiProcessorCount);
    long long* dcyc; double* dsink;
    CK(cudaMalloc(&dcyc, sizeof(long long)));
    CK(cudaMalloc(&dsink, 4096 * sizeof(double)));
    const int rounds = 20000;
    int rc = 0;
    rc |= run_all<2>(p.multiProcessorCount, rounds, dcyc, dsink);
    rc |= run_all<4>(p.multiProcessorCount, rounds, dcyc, dsink);
    rc |= run_all<8>(p.multiProcessorCount, rounds, dcyc, dsink);
    CK(cudaDeviceSynchronize());
    return rc;
}
