// engine.cu — host side of libautoinst_ncuts: workspace planning, the level loop that drives the
// recursion of normalized_cut.py:37-63 breadth-first on the device, and the C ABI of
// include/autoinst_ncuts.h.  All decisions (costs, mcut < T, stop rules, child tables) are taken
// by kernels; the host only reads back a few counters per level to size the next grids.
#include <cub/cub.cuh>
#include <stdarg.h>
#include <algorithm>

#include "common.cuh"
#include "kernels_graph.cuh"
#include "kernels_lanczos.cuh"
#include "kernels_ncut.cuh"
#include "kernels_cluster.cuh"
#include "kernels_pool.cuh"
#include "kernels_dino.cuh"
#include "kernels_csr.cuh"
#include "kernels_nodecsr.cuh"

namespace ancuts {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// affinity_tc.cu
int launch_affinity_tc(int n, const double* pts, const float* tarl, int tdim, const float* dino, int ddim,
                       const uint8_t* tarl_zero, double alpha, double theta, double gamma, double prox,
                       float* W, long long ld, void* scratch, size_t scratch_bytes, cudaStream_t st);
size_t affinity_tc_scratch_bytes(int n, int tdim, int ddim);

}  // namespace ancuts

#include "handle.cuh"

using namespace ancuts;

namespace ancuts {

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Arena {
    char* base;
    size_t off = 0;
    template <typename T> T* take(size_t count) {
        off = align_up(off, 256);
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += count * sizeof(T);
        return p;
    }
};

struct Plan {
    int B = 0;
    int P = 0;
    int kmax = KMAX_DEFAULT;
    int KS = KMAX_DEFAULT + 4;
    int active_cap = 0;
    int cslot_cap = 0;
    bool own_w0 = true, own_w1 = true;
    std::vector<int> n, ld, base, norig;
    size_t cub_bytes = 0;
    // device pointers handed out by the arena
    int *c_base, *c_n, *c_ld, *c_norig;
    float **c_W0, **c_W1;
    std::vector<float*> hW0, hW1;
    int* labels_scratch;
    int* nseg;
    uint8_t* tarl_zero;
    void* cub_tmp;
    void* tc_scratch; size_t tc_scratch_bytes = 0;
    PairQ* pairq = nullptr; int* qctr = nullptr;     // pair queue, [2c]=count [2c+1]=overflow
    int qcap = 0;                          // stage entry (ancuts_affinity_f32): capacity of its single queue
    bool deferred = false;                 // points input: per-chunk pair queues kept until the root split (deferred affinity)
    std::vector<long long> qoff;           // deferred: first queue entry of chunk c
    std::vector<int> qcap_c;               // deferred: queue capacity of chunk c
    int* pg_cells = nullptr; int* pg_sorted = nullptr; int* pg_tmp = nullptr; double* pg_spts = nullptr; PairGrid* pg_grid = nullptr;   // deferred: cell grids of the pair search
    int* c_tile0 = nullptr; double* tbox = nullptr; long long* d_qoff = nullptr; int* d_qcap = nullptr;          // cell-sorted sweep
    std::vector<int> tile0; int max_tiles = 0;
    bool grid_pairs = false;
    bool csr = false;                      // caller graphs in CSR form (ancuts_segment_csr_f32)
    unsigned long long* csr_err = nullptr; int* csr_out = nullptr;      // k_csr_validate: first violation per graph, range flag
    // CSR node form (deferred points input, ANCUTS_OPT_NODE_FORM = 0): two row sets (the level's and its children's), the
    // per-pair values of the feature pass, per-row counts / cursors, the list of slots k_ncsr_densify writes
    bool node_csr = false;
    int* ncsr_ptr[2] = {nullptr, nullptr}; int* ncsr_col[2] = {nullptr, nullptr}; float* ncsr_val[2] = {nullptr, nullptr};
    int ncsr_cur = 0;
    int* ncsr_cnt = nullptr; float* pslot = nullptr; int* ncsr_list = nullptr; int* ncsr_count = nullptr;
    ancuts_node_stat* stats;
    Eng e{};            // zero: optional pointers (sel, unfused, dbg, stats) are NULL unless a call sets them
};

static size_t cub_temp_bytes(int P) {
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                    (int*)nullptr, (int*)nullptr, P, 0, 64);
    cub::DeviceScan::InclusiveSum(nullptr, b, (int*)nullptr, (int*)nullptr, P);
    size_t c = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, c, (int*)nullptr, (int*)nullptr, P + 1);     // row pointers of the CSR node form
    return std::max(std::max(a, b), c) + 256;
}

// lay out every buffer; with base == nullptr only the size is computed
static size_t layout(Plan& pl, char* base, int stats_cap, int tdim, int ddim, bool need_tc) {
    Arena ar{base};
    const int B = pl.B, P = pl.P, KS = pl.KS;
    Eng& e = pl.e;
    pl.c_base = ar.take<int>(B); pl.c_n = ar.take<int>(B); pl.c_ld = ar.take<int>(B); pl.c_norig = ar.take<int>(B);
    pl.c_W0 = ar.take<float*>(B); pl.c_W1 = ar.take<float*>(B);
    e.r_start = ar.take<int>(P + 1); e.r_n = ar.take<int>(P + 1); e.r_chunk = ar.take<int>(P + 1);
    e.r_status = ar.take<int>(P + 1); e.r_level = ar.take<int>(P + 1);
    e.q_start = ar.take<int>(P + 1); e.q_n = ar.take<int>(P + 1); e.q_chunk = ar.take<int>(P + 1);
    e.q_status = ar.take<int>(P + 1); e.q_level = ar.take<int>(P + 1);
    e.r_pass = ar.take<int>(2 * (size_t)P + 2); e.r_slot = nullptr;
    e.rid = ar.take<int>(P); e.rid2 = ar.take<int>(P); e.perm = ar.take<int>(P); e.perm2 = ar.take<int>(P);
    e.deg = ar.take<double>(P); e.sinv = ar.take<double>(P); e.wbuf = ar.take<double>(P);
    e.ybuf = ar.take<double>(P); e.ev = ar.take<double>(P); e.zbuf = ar.take<double>(P + 4);
    e.bucket = ar.take<uint8_t>(P); e.side = ar.take<uint8_t>(P); e.rownnz = ar.take<int>(P);
    e.parent = ar.take<int>(P); e.croot = ar.take<int>(P);
    e.key = ar.take<unsigned long long>(P); e.key2 = ar.take<unsigned long long>(P);
    e.val = ar.take<int>(P); e.val2 = ar.take<int>(P); e.flag = ar.take<int>(P); e.incl = ar.take<int>(P);
    e.V = ar.take<double>((size_t)KS * P);
    const int A = pl.active_cap;
    e.split_ids = ar.take<int>(A);
    e.a_rid = ar.take<int>(A); e.a_k = ar.take<int>(A); e.a_kcap = ar.take<int>(A); e.a_done = ar.take<int>(A);
    e.a_conv = ar.take<int>(A); e.a_slot0 = ar.take<int>(A); e.a_nch = ar.take<int>(A);
    e.a_alpha = ar.take<double>((size_t)A * KS); e.a_beta = ar.take<double>((size_t)A * KS);
    e.a_y = ar.take<double>((size_t)A * KS);
    e.a_bprev = ar.take<double>(A); e.a_h1 = ar.take<double>(A); e.a_h2 = ar.take<double>(A); e.a_need2 = ar.take<int>(A);
    e.a_theta = ar.take<double>(2 * (size_t)A); e.a_thr = ar.take<double>((size_t)A * NCUT);
    e.a_sign = ar.take<double>(A); e.a_nocut = ar.take<int>(A);
    e.a_diff = ar.take<unsigned long long>((size_t)A * (NB + 1)); e.a_cnt = ar.take<int>((size_t)A * NB);
    e.a_bestk = ar.take<int>(A); e.a_mcut = ar.take<double>(A); e.a_costs = ar.take<double>((size_t)A * NCUT);
    const int C = pl.cslot_cap;
    e.p_dot = ar.take<double>((size_t)C * KS); e.p_dot2 = ar.take<double>((size_t)C * KS);
    e.p_norm = ar.take<double>(C); e.p_stat = ar.take<double>((size_t)C * 4); e.p_vol = ar.take<double>((size_t)C * NB);
    e.ctr = ar.take<int>(CTR_COUNT);
    e.a_path = ar.take<int>(A);
    e.a_fused = ar.take<int>(A);
    e.unfused = ar.take<int>(A);
    e.cl_ids = ar.take<int>((size_t)CL_CLASSES * A);
    e.active_cap = A;
    e.acct = ar.take<unsigned long long>(SG_ACCT);
    pl.stats = ar.take<ancuts_node_stat>(std::max(stats_cap, 1));
    pl.labels_scratch = ar.take<int>(P);
    pl.nseg = ar.take<int>(B);
    pl.tarl_zero = ar.take<uint8_t>(P);
    pl.cub_tmp = ar.take<char>(pl.cub_bytes);
    pl.tc_scratch_bytes = 0;
    pl.tc_scratch = nullptr;
    if (need_tc) {
        int nmax = 0;
        for (int c = 0; c < B; ++c) nmax = std::max(nmax, pl.n[c]);
        pl.tc_scratch_bytes = affinity_tc_scratch_bytes(nmax, tdim, ddim);
        pl.tc_scratch = ar.take<char>(pl.tc_scratch_bytes);
    }
    pl.pairq = nullptr; pl.qctr = nullptr;
    if (pl.deferred) {
        size_t total = 0;
        pl.qoff.assign(B, 0); pl.qcap_c.assign(B, 0);
        for (int c = 0; c < B; ++c) {
            const long long nc = pl.n[c];
            pl.qoff[c] = total;
            pl.qcap_c[c] = (int)std::min<long long>(96ll * nc, nc * (nc - 1) / 2 + 1);
            total += (size_t)pl.qcap_c[c];
        }
        pl.pairq = ar.take<PairQ>(total);
        pl.qctr = ar.take<int>(2 * (size_t)B);
        pl.pg_cells = ar.take<int>((size_t)B * PG_STRIDE);
        pl.pg_sorted = ar.take<int>((size_t)P);
        pl.pg_tmp = ar.take<int>((size_t)P);
        pl.pg_spts = ar.take<double>((size_t)P * 3);
        pl.pg_grid = ar.take<PairGrid>((size_t)B);
        pl.tile0.assign(B + 1, 0);
        pl.max_tiles = 0;
        for (int c = 0; c < B; ++c) {
            const int t = (pl.n[c] + PS_T - 1) / PS_T;
            pl.tile0[c + 1] = pl.tile0[c] + t;
            pl.max_tiles = std::max(pl.max_tiles, t);
        }
        pl.c_tile0 = ar.take<int>((size_t)B + 1);
        pl.tbox = ar.take<double>((size_t)pl.tile0[B] * 6);
        pl.d_qoff = ar.take<long long>((size_t)B);
        pl.d_qcap = ar.take<int>((size_t)B);
        // CSR node form: at most both directions of every queued pair plus the diagonal (int row pointers)
        const size_t ecap = 2 * total + (size_t)P;
        if (ecap > 0x7fffffffULL) pl.node_csr = false;
        if (pl.node_csr) {
            for (int k = 0; k < 2; ++k) {
                pl.ncsr_ptr[k] = ar.take<int>((size_t)P + 1);
                pl.ncsr_col[k] = ar.take<int>(ecap);
                pl.ncsr_val[k] = ar.take<float>(ecap);
            }
            pl.ncsr_cnt = ar.take<int>((size_t)P + 1);
            pl.pslot = ar.take<float>(total);
            pl.ncsr_list = ar.take<int>((size_t)pl.active_cap);
            pl.ncsr_count = ar.take<int>(1);
        }
    } else {
        pl.node_csr = false;
    }
    pl.csr_err = nullptr; pl.csr_out = nullptr;
    if (pl.csr) { pl.csr_err = ar.take<unsigned long long>(B); pl.csr_out = ar.take<int>(1); }
    pl.hW0.assign(B, nullptr); pl.hW1.assign(B, nullptr);
    if (pl.own_w0) for (int c = 0; c < B; ++c) pl.hW0[c] = ar.take<float>((size_t)pl.n[c] * pl.ld[c]);
    if (pl.own_w1) for (int c = 0; c < B; ++c) pl.hW1[c] = ar.take<float>((size_t)pl.n[c] * pl.ld[c]);
    return align_up(ar.off, 256);
}

static void make_plan(Plan& pl, int B, const int* n, const int* norig, const int64_t* ld_user, int kmax,
                      int extra_active) {
    pl.B = B;
    pl.n.assign(n, n + B);
    pl.norig.resize(B); pl.ld.resize(B); pl.base.resize(B);
    long long P = 0;
    for (int c = 0; c < B; ++c) {
        pl.base[c] = (int)P;
        pl.norig[c] = norig ? norig[c] : n[c];
        pl.ld[c] = ld_user ? (int)ld_user[c] : (int)align_up((size_t)n[c], 32);
        P += n[c];
    }
    pl.P = (int)P;
    pl.kmax = kmax;
    pl.KS = kmax + 4;
    pl.active_cap = std::max(101 * B + 1, extra_active + 1);
    pl.active_cap = std::min(pl.active_cap, pl.P + 1);
    pl.cslot_cap = pl.P / CH + pl.active_cap + 1;
    pl.cub_bytes = cub_temp_bytes(pl.P);
}

static int ensure_ws(ancuts_handle* h, size_t bytes) {
    if (bytes <= h->ws_bytes) return ANCUTS_OK;
    if (h->ws) cudaFree(h->ws);
    h->ws = nullptr;
    h->ws_bytes = 0;
    cudaError_t err = cudaMalloc((void**)&h->ws, bytes);
    if (err != cudaSuccess) {
        set_error("workspace cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(err));
        cudaGetLastError();
        return ANCUTS_ENOMEM;
    }
    h->ws_bytes = bytes;
    return ANCUTS_OK;
}

// --- launch bookkeeping ------------------------------------------------------------------------
static cudaEvent_t take_event(ancuts_handle* h) {
    if (h->pool_used == h->pool.size()) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        h->pool.push_back(ev);
    }
    return h->pool[h->pool_used++];
}

struct LaunchScope {
    ancuts_handle* h; int stage; cudaStream_t st; cudaEvent_t b = nullptr;
    LaunchScope(ancuts_handle* h_, int stage_, cudaStream_t st_) : h(h_), stage(stage_), st(st_) {
        h->launches_total++;
        h->stage_launches[stage]++;
        if (h->stage_timing == 1 || (h->stage_timing == 2 && stage == SG_MATVEC)) {
            cudaEvent_t a = take_event(h);
            b = take_event(h);
            cudaEventRecord(a, st);
            h->timed.push_back({stage, a, b});
        }
    }
    ~LaunchScope() { if (b) cudaEventRecord(b, st); }
};
#define LAUNCH(stage, ...) do { LaunchScope _ls(h, stage, st); __VA_ARGS__; } while (0)
#define LAUNCH_ON(stream, stage, ...) do { LaunchScope _ls(h, stage, stream); __VA_ARGS__; } while (0)

static void begin_accounting(ancuts_handle* h) {
    for (int i = 0; i < SG_COUNT; ++i) { h->stage_launches[i] = 0; h->stage_bytes[i] = 0; h->stage_ms[i] = 0; }
    h->timed.clear();
    h->levels.clear();
    h->pool_used = 0;
}

static int end_accounting(ancuts_handle* h, const Eng& e, cudaStream_t st) {
    ANCUTS_CUDA(cudaMemcpyAsync(h->h_acct, e.acct, SG_ACCT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < SG_COUNT; ++i) h->stage_bytes[i] += (double)h->h_acct[i];
    h->sparse_entry_steps = (double)h->h_acct[SG_SPARSE_STEPS];
    h->sparse_nnz = (double)h->h_acct[SG_SPARSE_NNZ];
    h->cl_steps = (double)h->h_acct[SG_CL_STEPS];
    h->cl_full = (double)h->h_acct[SG_CL_FULL];
    for (auto& t : h->timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) {
            h->stage_ms[t.stage] += ms;
            if (t.level >= 0 && t.level < (int)h->levels.size()) h->levels[t.level].ms = ms;
        }
    }
    h->timed.clear();
    return ANCUTS_OK;
}

static int set_attrs(ancuts_handle* h, int KS) {
    if (h->attrs_set) return ANCUTS_OK;
    ANCUTS_CUDA(cudaFuncSetAttribute(k_lanczos_check, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (KMAX_LIMIT + 4) * 68 + 64));
    (void)KS;
    const int cl_smem = CL_DYN_SMEM;
#define ANCUTS_CL_ATTR(C, M) ANCUTS_CUDA(cudaFuncSetAttribute(k_lanczos_cluster<C, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, cl_smem))
    ANCUTS_CL_ATTR(1, 0); ANCUTS_CL_ATTR(2, 0); ANCUTS_CL_ATTR(4, 0); ANCUTS_CL_ATTR(8, 0);
    ANCUTS_CL_ATTR(1, 4); ANCUTS_CL_ATTR(2, 4); ANCUTS_CL_ATTR(4, 4); ANCUTS_CL_ATTR(8, 4);
    ANCUTS_CL_ATTR(1, 6); ANCUTS_CL_ATTR(2, 6); ANCUTS_CL_ATTR(4, 6); ANCUTS_CL_ATTR(8, 6);
    ANCUTS_CL_ATTR(1, 7); ANCUTS_CL_ATTR(2, 7); ANCUTS_CL_ATTR(4, 7); ANCUTS_CL_ATTR(8, 7);
#undef ANCUTS_CL_ATTR
    h->attrs_set = true;
    return ANCUTS_OK;
}

static int read_ctr(ancuts_handle* h, const Eng& e, cudaStream_t st) {
    ANCUTS_CUDA(cudaMemcpyAsync(h->h_ctr, e.ctr, CTR_COUNT * sizeof(int), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaStreamSynchronize(st));
#ifdef ANCUTS_EXCHANGE_GUARD
    if (h->h_ctr[19]) {
        set_error("internal: %d cluster-exchange waits of the Lanczos kernel gave up", h->h_ctr[19]);
        return ANCUTS_EINVAL;
    }
#endif
    return ANCUTS_OK;
}

// --- engine pieces -------------------------------------------------------------------------------
__global__ void k_init_roots(Eng e, double split_lim, double T) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < e.B) {
        int c = g;
        int n = e.c_n[c];
        e.r_start[c] = e.c_base[c];
        e.r_n[c] = n;
        e.r_chunk[c] = c;
        e.r_level[c] = 0;
        double frac = (double)n / ((double)e.c_norig[c] + 1e-8);
        bool pass = (n > 2) && (frac > split_lim) && (T > 0.0);     // normalized_cut.py:39-40
        e.r_status[c] = pass ? ST_SPLIT : ST_LEAF;
        e.r_pass[2 * c] = 1;
        e.r_pass[2 * c + 1] = 1;
        if (pass) {
            int s = atomicAdd(&e.ctr[5], 1);
            e.split_ids[s] = c;
            atomicMax(&e.ctr[7], n);
        }
    }
    if (g < e.P) e.side[g] = 0;
}

// order != NULL: position g of a chunk holds the point order[g] (cell-sorted order of the batched pair search: neighbours in
// space are neighbours in every node, the stored entries of a row come in runs of consecutive columns)
__global__ void k_init_positions(Eng e, const int* __restrict__ order) {
    int c = blockIdx.y;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < e.c_n[c]) {
        int g = e.c_base[c] + i;
        e.rid[g] = c;
        e.perm[g] = order ? order[g] : i;
    }
}

static int upload_tables(Plan& pl, cudaStream_t st) {
    const int B = pl.B;
    ANCUTS_CUDA(cudaMemcpyAsync(pl.c_base, pl.base.data(), B * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(pl.c_n, pl.n.data(), B * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(pl.c_ld, pl.ld.data(), B * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(pl.c_norig, pl.norig.data(), B * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(pl.c_W0, pl.hW0.data(), B * sizeof(float*), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(pl.c_W1, pl.hW1.data(), B * sizeof(float*), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaStreamSynchronize(st));      // host vectors may go away
    Eng& e = pl.e;
    e.P = pl.P; e.B = B; e.KS = pl.KS; e.kmax = pl.kmax;
    e.c_base = pl.c_base; e.c_n = pl.c_n; e.c_ld = pl.c_ld; e.c_norig = pl.c_norig;
    e.c_W0 = pl.c_W0; e.c_W1 = pl.c_W1;
    return ANCUTS_OK;
}

static void fill_params(Eng& e, const ancuts_params* p, int kmax) {
    e.kmax = kmax;
    e.KS = kmax + 4;
    e.check_every = p->lanczos_check_every > 0 ? p->lanczos_check_every : CHECK_DEFAULT;
    e.check_adapt = p->lanczos_check_every <= 0;
    e.tol = p->lanczos_tol > 0 ? p->lanczos_tol : TOL_DEFAULT;
    e.T = p->T;
}

static int resolve_kmax(const ancuts_params* p) {
    int k = p->lanczos_max_steps > 0 ? p->lanczos_max_steps : KMAX_DEFAULT;
    return std::min(std::max(k, 2), KMAX_LIMIT);
}

// feature inputs of an affinity call (stage entry, points input of the segment path)
static int check_features(const ancuts_params* p, const float* tarl, const float* dino, int dcams) {
    const bool use_tarl = p->theta != 0.0 && tarl != nullptr;
    const bool use_dino = p->gamma != 0.0 && dino != nullptr;
    if (dcams < 1) { set_error("dino_cams must be at least 1 (got %d)", dcams); return ANCUTS_EINVAL; }
    if (p->theta != 0.0 && tarl == nullptr) { set_error("theta != 0 but no TARL features"); return ANCUTS_EINVAL; }
    if (p->gamma != 0.0 && dino == nullptr) {
        set_error("The length should be longer than 0!");      // ncuts_utils.py:126-127
        return ANCUTS_EINVAL;
    }
    if ((use_tarl && (p->tarl_dim <= 0 || p->tarl_dim % 4)) || (use_dino && (p->dino_dim <= 0 || p->dino_dim % 4))) {
        set_error("feature dimensions must be positive multiples of 4 (got %d, %d)", p->tarl_dim, p->dino_dim);
        return ANCUTS_EUNSUPPORTED;
    }
    if (use_dino && dcams > 1 && p->affinity_impl == 1) {
        set_error("the tensor-core affinity form (affinity_impl = 1) takes one DINOv2 camera (got %d)", dcams);
        return ANCUTS_EUNSUPPORTED;
    }
    return ANCUTS_OK;
}

// W of one chunk written whole (inputs checked by check_features).  qctr != NULL selects the two-pass form of the stage
// entry (feature terms only): pairs into the single queue pl.pairq, then the feature pass.
static int run_affinity(ancuts_handle* h, Plan& pl, int n, const double* pts, const float* tarl, const float* dino,
                        int dcams, const ancuts_params* p, float* W, long long ld, uint8_t* tarl_zero, cudaStream_t st,
                        int* qctr = nullptr) {
    const bool use_tarl = p->theta != 0.0 && tarl != nullptr;
    const bool use_dino = p->gamma != 0.0 && dino != nullptr;
    if (use_tarl)
        LAUNCH(SG_AFFINITY, k_zero_rows<<<(n + 7) / 8, 256, 0, st>>>(n, tarl, p->tarl_dim, tarl_zero));
    if (p->affinity_impl == 1 && (use_tarl || use_dino)) {
        h->launches_total++; h->stage_launches[SG_AFFINITY]++;
        int rc = launch_affinity_tc(n, pts, use_tarl ? tarl : nullptr, p->tarl_dim, use_dino ? dino : nullptr,
                                    p->dino_dim, tarl_zero, p->alpha, p->theta, p->gamma, p->proximity, W, ld,
                                    pl.tc_scratch, pl.tc_scratch_bytes, st);
        if (rc != ANCUTS_OK) return rc;
    } else if (qctr) {
        // two-pass form: distances + zero fill + pair queue, then the queued pairs spread over the whole grid
        dim3 grid((unsigned)((ld + AT - 1) / AT), (n + AT - 1) / AT);
        LAUNCH(SG_AFFINITY, k_affinity_pairs<<<grid, 256, 0, st>>>(n, pts, p->alpha, p->proximity, W, ld, pl.pairq, pl.qcap, qctr,
                                                                   nullptr, 0));
        LAUNCH(SG_AFFINITY, k_affinity_feats<<<148 * 4, 256, 0, st>>>(pl.pairq, qctr, pl.qcap, use_tarl ? tarl : nullptr, p->tarl_dim,
                                                                        use_dino ? dino : nullptr, p->dino_dim, dcams, tarl_zero, p->theta,
                                                                        p->gamma, W, ld));
    } else {
        dim3 grid((unsigned)((ld + AT - 1) / AT), (n + AT - 1) / AT);
        LAUNCH(SG_AFFINITY, k_affinity_exact<<<grid, 256, 0, st>>>(n, pts, use_tarl ? tarl : nullptr, p->tarl_dim,
                                                                   use_dino ? dino : nullptr, p->dino_dim, dcams, tarl_zero,
                                                                   p->alpha, p->theta, p->gamma, p->proximity, W, ld));
    }
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

// CSR node form: dense blocks of the level's nodes that read dense W (all != 0: every node, for the grid-wide Lanczos
// path and the cut kernels after it; otherwise nodes above CL_NMAX points and slices that would not fit the cluster kernel)
static int densify_nodes(ancuts_handle* h, Eng& e, int cur, int num_active, bool all, unsigned cmap, cudaStream_t st) {
    ANCUTS_CUDA(cudaMemsetAsync(e.dn_count, 0, sizeof(int), st));
    LAUNCH(SG_PARTITION, k_ncsr_need<<<num_active, 256, 0, st>>>(e, all ? 1 : 0, cmap, e.dn_list, e.dn_count));
    LAUNCH(SG_PARTITION, k_ncsr_densify<<<dim3(ZB_BLOCKS, num_active), 256, 0, st>>>(e, cur, e.dn_list, e.dn_count));
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

// Lanczos for all active nodes of the current table (degrees must be set)
static int run_lanczos(ancuts_handle* h, Eng& e, int cur, int num_active, int max_n, cudaStream_t st) {
    const int KS = e.KS;
    if (e.node_csr) {                 // k_matvec, and after it the cut kernels, read every node's dense block
        int rc = densify_nodes(h, e, cur, num_active, true, 0u, st);
        if (rc) return rc;
    }
    LAUNCH(SG_REORTH, k_lanczos_init<<<num_active, 256, 0, st>>>(e));
    const int nch_max = (max_n + CH - 1) / CH;
    const size_t up_smem = (size_t)(KS + CH + 8) * 8;
    const size_t ck_smem = (size_t)KS * 8 * 8 + (size_t)KS * 4 + 64;
    const int kcap_max = std::min(e.kmax, std::max(max_n - 1, 1));
    int step = 0;
    while (true) {
        int burst = std::min(e.check_every, kcap_max - step);
        for (int s = 0; s < burst; ++s, ++step) {
            // rows per warp: with 4 a single 8-16 k node has only 256-512 CTAs of 8 warps for 148 SMs (58 / 62 % of the HBM peak
            // measured at 8 / 16 k); 2 rows per warp gave 84 % at 16 k, 1 row per warp only 47 % at 8 k
            const long long rows_total = (long long)max_n * num_active;
            if (rows_total >= 49152) {
                dim3 gmv((max_n + 31) / 32, num_active);
                LAUNCH(SG_MATVEC, k_matvec<4><<<gmv, 256, 0, st>>>(e, cur));
            } else {
                dim3 gmv((max_n + 15) / 16, num_active);
                LAUNCH(SG_MATVEC, k_matvec<2><<<gmv, 256, 0, st>>>(e, cur));
            }
            dim3 gd(nch_max, (step + 2 + 31) / 32, num_active);
            LAUNCH(SG_REORTH, k_dots<<<gd, 256, 0, st>>>(e));
            dim3 gu(nch_max, num_active);
            LAUNCH(SG_REORTH, k_update<1><<<gu, 256, up_smem, st>>>(e));
            LAUNCH(SG_REORTH, k_update<2><<<gu, 256, up_smem, st>>>(e));
            LAUNCH(SG_REORTH, k_lanczos_finalize<<<(num_active + 127) / 128, 128, 0, st>>>(e, num_active));
        }
        bool last = step >= kcap_max;
        ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 4, 0, sizeof(int), st));
        LAUNCH(SG_REORTH, k_lanczos_check<<<num_active, 128, ck_smem, st>>>(e, last ? 1 : 0));
        ANCUTS_CUDA(cudaGetLastError());
        int rc = read_ctr(h, e, st);
        if (rc) return rc;
        if (h->h_ctr[4] == 0 || last) break;
    }
    return ANCUTS_OK;
}

template <int C, int MODE>
static cudaError_t launch_cluster_m(const Eng& e, int cur, const int* ids, int count, cudaStream_t s) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)count * C, 1, 1);
    cfg.blockDim = dim3(CL_THREADS, 1, 1);
    cfg.dynamicSmemBytes = CL_DYN_SMEM;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = (C > 1) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, k_lanczos_cluster<C, MODE>, e, cur, ids, (int)(CL_DYN_SMEM / 8));
}

// matvec variant: 0 = guarded (out-of-block entries selected away: the caller's W is read in place and may hold anything next
// to a block), 4 = TMA ring (blocks written by k_gather_blocks_cur / k_zero_blocks: fringe zeroed, no selects),
// 6 = TMA ring + integer widening of every second element (the library's own affinities: 0 or [2^-126, 2))
static inline int cluster_mode(const Eng& e) {
    if (e.w_guard) return 0;
    return e.w_own ? 6 : 4;
}

template <int C>
static cudaError_t launch_cluster(const Eng& e, int cur, const int* ids, int count, cudaStream_t s, bool sparse = false) {
    if (sparse && cluster_mode(e) == 6) return launch_cluster_m<C, 7>(e, cur, ids, count, s);
    switch (cluster_mode(e)) {
        case 6: return launch_cluster_m<C, 6>(e, cur, ids, count, s);
        case 4: return launch_cluster_m<C, 4>(e, cur, ids, count, s);
        default: return launch_cluster_m<C, 0>(e, cur, ids, count, s);
    }
}

// Lanczos for every active node: persistent cluster kernels (one stream per cluster size, running
// concurrently) for nodes up to CL_NMAX points, then the grid-wide multi-launch path for larger
// nodes and for nodes the cluster kernel could not finish in CL_KMAX steps.
static int run_lanczos_all(ancuts_handle* h, Eng& e, int cur, int num_active, int max_n, const int* class_cnt,
                           int big_cnt, cudaStream_t st) {
    ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 4, 0, sizeof(int), st));
    bool any = false, launch_failed = false;
    // bins <=320, <=512, <=640, <=1024, <=2048, <=4096 points.  Latency mapping (short critical path) when all
    // clusters of the level are resident at once; otherwise the level is bound by SM time and fewer CTAs per
    // node do the same work with fewer cluster barriers.
    static const int c_latency[CL_CLASSES] = {1, 2, 2, 4, 8, 8};
    static const int c_throughput[CL_CLASSES] = {1, 1, 2, 2, 4, 8};
    // Shared-memory sparse form (ANCUTS_OPT_MATVEC = 0, the default): the same two mappings.  Its steps are short, the fixed
    // costs per CTA (cluster barriers, the redundant convergence checks) count, and a level is bound by SM time: the mapping
    // with the fewest CTAs per node measured 2858 chunks/s against 2351 with {1,2,2,4,8,8} (profiles/r2e_cmap_*.json); with
    // 512-row slices most of the basis then sits behind the CSR slice in L2.
    const bool sparse_on = h->opt[ANCUTS_OPT_MATVEC] == 0 && cluster_mode(e) == 6;
    int ctas = 0;
    for (int b = 0; b < CL_CLASSES; ++b) ctas += class_cnt[b] * c_latency[b];
    const int* cmap = (ctas <= 148) ? c_latency : c_throughput;
    int c_user[CL_CLASSES];
    if (h->opt[ANCUTS_OPT_CLUSTER_MAP] > 0) {                   // tuning: six decimal digits, CTAs per node for the six size bins
        int d = h->opt[ANCUTS_OPT_CLUSTER_MAP];
        bool ok = true;
        for (int b = CL_CLASSES - 1; b >= 0; --b) { c_user[b] = d % 10; d /= 10; ok &= (c_user[b] == 1 || c_user[b] == 2 || c_user[b] == 4 || c_user[b] == 8); }
        // a slice has at most CL_RPMAX rows
        static const int nmax[CL_CLASSES] = {320, 512, 640, 1024, 2048, 4096};
        for (int b = 0; b < CL_CLASSES; ++b) ok &= ((nmax[b] + c_user[b] - 1) / c_user[b] <= CL_RPMAX);
        if (ok && d == 0) cmap = c_user;
    }
    if (e.node_csr && sparse_on) {    // nodes whose slices would not fit read their dense block inside the cluster kernel
        unsigned packed = 0;
        for (int b = 0; b < CL_CLASSES; ++b) packed |= (unsigned)cmap[b] << (4 * b);
        int rc = densify_nodes(h, e, cur, num_active, false, packed, st);
        if (rc) return rc;
    }
    // one timed "launch" per level: the concurrent cluster kernels from fork to join on the launching stream (the fork
    // follows the dense blocks the cluster kernels read)
    cudaEvent_t t_a = nullptr, t_b = nullptr;
    if (h->stage_timing) { t_a = take_event(h); t_b = take_event(h); cudaEventRecord(t_a, st); }
    ANCUTS_CUDA(cudaEventRecord(h->ev_fork, st));
    for (int cls = CL_CLASSES - 1; cls >= 0; --cls) {          // largest nodes first
        int cnt = class_cnt[cls];
        if (cnt <= 0) continue;
        cudaStream_t s = h->side[cls];
        ANCUTS_CUDA(cudaStreamWaitEvent(s, h->ev_fork, 0));
        const int* ids = e.cl_ids + (size_t)cls * e.active_cap;
        cudaError_t err = cudaSuccess;
        {
            h->launches_total++;
            const bool sp = sparse_on;       // every bin: a slice that does not fit streams W inside the same kernel
            switch (cmap[cls]) {
                case 1: err = launch_cluster<1>(e, cur, ids, cnt, s, sp); break;
                case 2: err = launch_cluster<2>(e, cur, ids, cnt, s, sp); break;
                case 4: err = launch_cluster<4>(e, cur, ids, cnt, s, sp); break;
                default: err = launch_cluster<8>(e, cur, ids, cnt, s, sp); break;
            }
        }
        if (err != cudaSuccess) {                               // e.g. cluster size not schedulable: multi-launch path
            cudaGetLastError();
            launch_failed = true;
        }
        ANCUTS_CUDA(cudaEventRecord(h->ev_join[cls], s));
        ANCUTS_CUDA(cudaStreamWaitEvent(st, h->ev_join[cls], 0));
        any = true;
    }
    if (any) {
        h->stage_launches[SG_MATVEC]++;
        if (t_b) {
            cudaEventRecord(t_b, st);
            LevelRec lr;
            lr.num_active = num_active; lr.big = big_cnt; lr.ms = 0.0;
            for (int b = 0; b < CL_CLASSES; ++b) { lr.cls[b] = class_cnt[b]; lr.cmap[b] = cmap[b]; }
            h->levels.push_back(lr);
            h->timed.push_back({SG_MATVEC, t_a, t_b, (int)h->levels.size() - 1});
        }
    }
    int rest = big_cnt;
    if (any || launch_failed) {
        int rc = read_ctr(h, e, st);
        if (rc) return rc;
        rest += h->h_ctr[4];
    }
    if (rest > 0 || launch_failed) return run_lanczos(h, e, cur, num_active, max_n, st);
    return ANCUTS_OK;
}

// Ritz vector, sign, thresholds, buckets, cut scan, decision, side flags
static int run_cut(ancuts_handle* h, Eng& e, int cur, int num_active, int max_n, bool ritz, cudaStream_t st,
                   bool reset_split_list = true) {
    const int nch_max = (max_n + CH - 1) / CH;
    dim3 gc(nch_max, num_active);
    if (ritz) {
        LAUNCH(SG_REORTH, k_ritz<<<gc, 256, (size_t)(e.KS + 32) * 8, st>>>(e));
    }
    LAUNCH(SG_SCAN, k_ev_final<<<(num_active + 127) / 128, 128, 0, st>>>(e, num_active));
    LAUNCH(SG_SCAN, k_bucket<<<gc, 256, 0, st>>>(e));
    if (reset_split_list) {
        ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 5, 0, sizeof(int), st));
        ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 7, 0, sizeof(int), st));
    }
    dim3 gs((max_n + 7) / 8, num_active);
    LAUNCH(SG_SCAN, k_scan<<<gs, 256, 0, st>>>(e, cur));
    LAUNCH(SG_SCAN, k_decide<<<(num_active + 127) / 128, 128, 0, st>>>(e, num_active));
    LAUNCH(SG_SCAN, k_sides<<<gc, 256, 0, st>>>(e));
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

__global__ void k_add_scalar(int n, double* x, double v) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] += v;
}

// ABI side flags (1 = the reference's mask, ev > t) <-> internal side (0 = mask side, sorted first)
__global__ void k_mask_from_side(Eng e, uint8_t* __restrict__ out) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= e.P) return;
    int r = e.rid[g];
    out[g] = (e.r_status[r] == ST_SPLIT && e.side[g] == 0) ? 1 : 0;
}
__global__ void k_side_from_mask(Eng e, const uint8_t* __restrict__ mask) {
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < e.P) e.side[g] = mask[g] ? 0 : 1;
}

// chunk-level statistics for stand-alone ev input (stage 4a entry point): sum/min/max/sumsq partials
__global__ void __launch_bounds__(256)
k_ev_stats(Eng e) {
    __shared__ double red[32];
    int a = blockIdx.y;
    int nch = e.a_nch[a];
    int ch = blockIdx.x;
    if (ch >= nch) return;
    int r = e.a_rid[a];
    int start = e.r_start[r], n = e.r_n[r];
    int c0 = ch * CH + threadIdx.x, c1 = c0 + 256;
    double x0 = c0 < n ? e.ev[start + c0] : 0.0, x1 = c1 < n ? e.ev[start + c1] : 0.0;
    double s = x0 + x1;
    double mn = fmin(c0 < n ? x0 : 1e300, c1 < n ? x1 : 1e300);
    double mx = fmax(c0 < n ? x0 : -1e300, c1 < n ? x1 : -1e300);
    double q = x0 * x0 + x1 * x1;
    s = warp_sum(s); mn = warp_min(mn); mx = warp_max(mx); q = warp_sum(q);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { red[w] = s; red[8 + w] = mn; red[16 + w] = mx; red[24 + w] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0.0, tmn = 1e300, tmx = -1e300, tq = 0.0;
        for (int i = 0; i < 8; ++i) { ts += red[i]; tmn = fmin(tmn, red[8 + i]); tmx = fmax(tmx, red[16 + i]); tq += red[24 + i]; }
        double* o = e.p_stat + (size_t)(e.a_slot0[a] + ch) * 4;
        o[0] = ts; o[1] = tmn; o[2] = tmx; o[3] = tq;
    }
}

// split phase: components, sort, new table, gather.  Returns new counts through h->h_ctr.
// inputs of the deferred second affinity pass (run_rebuild of the root split)
struct DeferredAffinity {
    const ancuts_params* p;
    const float* tarl;      // all chunks, input order
    const float* dino;      // point-major, dcams * dino_dim values per point
    int dcams;
    const cudaEvent_t* feats;      // host entry: chunk c's features have arrived at feats[c], else NULL
    const int* order;              // batched pair stage: the queue holds cell-sorted ranks, order[base + rank] = input index
    // caller graphs (ancuts_segment_csr_f32): the stored entries take the place of the queued pairs
    const int64_t* row_ptr = nullptr;
    const int32_t* col = nullptr;
    const float* val = nullptr;
};

static void set_node_csr(Plan& pl, int s) {
    pl.ncsr_cur = s;
    pl.e.csr_ptr = pl.ncsr_ptr[s]; pl.e.csr_col = pl.ncsr_col[s]; pl.e.csr_val = pl.ncsr_val[s];
}

// CSR node form, root level (after the root split and the feature pass, which counted the entries per row on top of the
// diagonal k_ncsr_diag set; inv = e.val): scan, fill (diagonal first, then the pairs through atomic cursors), sort each
// row by column into the other row set and take its degree.
static int build_root_csr(ancuts_handle* h, Plan& pl, cudaStream_t st) {
    Eng& e = pl.e;
    const int P = e.P, g1 = (P + 1 + 255) / 256;
    const dim3 gq(148 * 4, e.B);
    size_t tmp = pl.cub_bytes;
    h->launches_total++; h->stage_launches[SG_AFFINITY]++;
    ANCUTS_CUDA(cub::DeviceScan::ExclusiveSum(pl.cub_tmp, tmp, pl.ncsr_cnt, pl.ncsr_ptr[0], P + 1, st));
    LAUNCH(SG_AFFINITY, k_ncsr_fill_diag<<<g1, 256, 0, st>>>(e, pl.ncsr_ptr[0], pl.ncsr_cnt, pl.ncsr_col[0], pl.ncsr_val[0]));
    LAUNCH(SG_AFFINITY, k_ncsr_pairs<<<gq, 256, 0, st>>>(pl.pairq, pl.d_qoff, pl.d_qcap, pl.qctr, pl.c_base, pl.pslot,
                                                                 e, e.val, pl.ncsr_cnt, pl.ncsr_col[0], pl.ncsr_val[0]));
    ANCUTS_CUDA(cudaMemcpyAsync(pl.ncsr_ptr[1], pl.ncsr_ptr[0], (size_t)(P + 1) * sizeof(int), cudaMemcpyDeviceToDevice, st));
    LAUNCH(SG_DEGREE, k_ncsr_sort_rows<<<(P + 7) / 8, 256, 0, st>>>(e, pl.ncsr_ptr[0], pl.ncsr_col[0], pl.ncsr_val[0],
                                                                       pl.ncsr_col[1], pl.ncsr_val[1]));
    ANCUTS_CUDA(cudaGetLastError());
    set_node_csr(pl, 1);
    return ANCUTS_OK;
}

static int run_rebuild(ancuts_handle* h, Plan& pl, int& cur, int num_split, int max_split_n, bool components,
                       cudaStream_t st, int* class_cnt = nullptr, int* big_cnt = nullptr,
                       const DeferredAffinity* df = nullptr, bool forest_inited = false) {
    Eng& e = pl.e;
    const int P = e.P;
    const int tb = 256, gP = (P + tb - 1) / tb;
    // forest_ready (deferred affinity): the input stage already joined every in-mask pair of the root ranges in e.parent
    // forest_inited: the level loop reset the forest before the Lanczos launch (the fused cut joins components into it)
    const bool forest_ready = df != nullptr;
    if (!forest_ready && !forest_inited) LAUNCH(SG_PARTITION, k_cc_init<<<gP, tb, 0, st>>>(e));
    if (!forest_ready && components && num_split > 0) {
        dim3 g((max_split_n + 7) / 8, num_split);
        LAUNCH(SG_PARTITION, k_cc_union<<<g, 256, 0, st>>>(e, cur, e.split_ids));
    }
    LAUNCH(SG_PARTITION, k_cc_flatten<<<gP, tb, 0, st>>>(e));
    LAUNCH(SG_PARTITION, k_build_keys<<<gP, tb, 0, st>>>(e));
    int pbits = 1;
    while ((1ll << pbits) < (long long)P + 1) ++pbits;
    size_t tmp = pl.cub_bytes;
    h->launches_total += 2; h->stage_launches[SG_PARTITION] += 2;
    ANCUTS_CUDA(cub::DeviceRadixSort::SortPairs(pl.cub_tmp, tmp, e.key, e.key2, e.val, e.val2, P, 0, 32 + pbits, st));
    LAUNCH(SG_PARTITION, k_boundaries<<<gP, tb, 0, st>>>(e));
    tmp = pl.cub_bytes;
    ANCUTS_CUDA(cub::DeviceScan::InclusiveSum(pl.cub_tmp, tmp, e.flag, e.incl, P, st));
    ANCUTS_CUDA(cudaMemsetAsync(e.ctr, 0, 4 * sizeof(int), st));
    ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 8, 0, 8 * sizeof(int), st));
    LAUNCH(SG_PARTITION, k_new_ranges<<<gP, tb, 0, st>>>(e));
    ANCUTS_CUDA(cudaGetLastError());
    int rc = read_ctr(h, e, st);
    if (rc) return rc;
    int num_ranges = h->h_ctr[0];
    LAUNCH(SG_PARTITION, k_finish_ranges<<<(num_ranges + tb - 1) / tb, tb, 0, st>>>(e, num_ranges));
    ANCUTS_CUDA(cudaGetLastError());
    rc = read_ctr(h, e, st);
    if (rc) return rc;
    int num_active = h->h_ctr[1], max_n = h->h_ctr[2];
    if (class_cnt) for (int i = 0; i < CL_CLASSES; ++i) class_cnt[i] = h->h_ctr[8 + i];
    if (big_cnt) *big_cnt = h->h_ctr[14];
    if (num_active > pl.active_cap || h->h_ctr[3] > pl.cslot_cap) {
        set_error("internal: active table overflow (%d nodes, %d chunk slots)", num_active, h->h_ctr[3]);
        return ANCUTS_EINVAL;
    }
    // the rebuilt table becomes current
    std::swap(e.r_start, e.q_start); std::swap(e.r_n, e.q_n); std::swap(e.r_chunk, e.q_chunk);
    std::swap(e.r_status, e.q_status); std::swap(e.r_level, e.q_level);
    std::swap(e.rid, e.rid2); std::swap(e.perm, e.perm2);
    if (num_active > 0 && df) {
        // deferred affinity: there is no matrix to gather from.  Dense node form: zero the blocks of the active ranges (unit
        // diagonal) and scatter the queued pairs of every chunk to the positions their points have now.  CSR node form: the
        // feature pass writes one value per queued pair and build_root_csr places them.
        if (!pl.node_csr) LAUNCH(SG_AFFINITY, k_zero_blocks<<<dim3(ZB_BLOCKS, num_active), 256, 0, st>>>(e, cur));
        LAUNCH(SG_PARTITION, k_inverse_positions<<<gP, tb, 0, st>>>(e, e.val));
        if (pl.node_csr) LAUNCH(SG_AFFINITY, k_ncsr_diag<<<(P + 1 + 255) / 256, 256, 0, st>>>(e, pl.ncsr_cnt));
        if (df->row_ptr) {
            // caller graphs: one pass over every graph's rows in input order
            int nmax = 0;
            for (int c = 0; c < e.B; ++c) nmax = std::max(nmax, pl.n[c]);
            dim3 g((nmax + 256 / CSR_LANES - 1) / (256 / CSR_LANES), e.B);
            LAUNCH(SG_AFFINITY, k_csr_scatter<<<g, 256, 0, st>>>(e, cur, df->row_ptr, df->col, df->val, e.val));
            ANCUTS_CUDA(cudaGetLastError());
            cur ^= 1;
            return ANCUTS_OK;
        }
        const ancuts_params* p = df->p;
        const bool use_tarl = p->theta != 0.0 && df->tarl, use_dino = p->gamma != 0.0 && df->dino;
        // the feature arrays hold every chunk from its first point on (chunk offsets start at 0): chunk c at row base[c]
        if (!df->feats) {
            // resident inputs: every chunk's pass in one launch
            LAUNCH(SG_AFFINITY, k_affinity_feats_b<<<dim3(148 * 4, e.B), 256, 0, st>>>(
                pl.pairq, pl.d_qoff, pl.d_qcap, pl.qctr, pl.c_base, use_tarl ? df->tarl : nullptr, p->tarl_dim,
                use_dino ? df->dino : nullptr, p->dino_dim, df->dcams, pl.tarl_zero, p->theta, p->gamma, cur ? pl.c_W0 : pl.c_W1,
                pl.c_ld, e.val, e.rid, e.r_status, df->order, pl.node_csr ? pl.pslot : nullptr, pl.ncsr_cnt));
        } else {
            // host entry: each chunk's pass waits for its features
            for (int c = 0; c < e.B; ++c) {
                const size_t o = (size_t)pl.base[c];
                ANCUTS_CUDA(cudaStreamWaitEvent(st, df->feats[c], 0));
                if (use_tarl)
                    LAUNCH(SG_AFFINITY, k_zero_rows<<<(pl.n[c] + 7) / 8, 256, 0, st>>>(pl.n[c], df->tarl + o * p->tarl_dim, p->tarl_dim,
                                                                                      pl.tarl_zero + o));
                LAUNCH(SG_AFFINITY, k_affinity_feats<<<148 * 4, 256, 0, st>>>(
                    pl.pairq + pl.qoff[c], pl.qctr + 2 * c, pl.qcap_c[c], use_tarl ? df->tarl : nullptr, p->tarl_dim,
                    use_dino ? df->dino : nullptr, p->dino_dim, df->dcams, pl.tarl_zero, p->theta, p->gamma,
                    pl.node_csr ? nullptr : (cur ? pl.hW0[c] : pl.hW1[c]), pl.ld[c], e.val, pl.base[c], e.rid, e.r_status,
                    df->order, pl.node_csr ? pl.pslot + pl.qoff[c] : nullptr, pl.ncsr_cnt));
            }
        }
        ANCUTS_CUDA(cudaGetLastError());
        if (pl.node_csr) {
            int rc2 = build_root_csr(h, pl, st);
            if (rc2) return rc2;
        }
        cur ^= 1;
    } else if (num_active > 0 && pl.node_csr) {
        // children's rows from their parents' rows (no dense block is gathered)
        LAUNCH(SG_PARTITION, k_inverse_positions<<<gP, tb, 0, st>>>(e, e.val));
        const int s = pl.ncsr_cur, gr = (P + 1 + 7) / 8;
        LAUNCH(SG_PARTITION, k_ncsr_children<false><<<gr, 256, 0, st>>>(e, e.val, pl.ncsr_ptr[s], pl.ncsr_col[s],
                                                                          pl.ncsr_val[s], pl.ncsr_cnt, nullptr, nullptr));
        tmp = pl.cub_bytes;
        h->launches_total++; h->stage_launches[SG_PARTITION]++;
        ANCUTS_CUDA(cub::DeviceScan::ExclusiveSum(pl.cub_tmp, tmp, pl.ncsr_cnt, pl.ncsr_ptr[s ^ 1], P + 1, st));
        LAUNCH(SG_DEGREE, k_ncsr_children<true><<<gr, 256, 0, st>>>(e, e.val, pl.ncsr_ptr[s], pl.ncsr_col[s],
                                                                         pl.ncsr_val[s], pl.ncsr_ptr[s ^ 1], pl.ncsr_col[s ^ 1],
                                                                         pl.ncsr_val[s ^ 1]));
        ANCUTS_CUDA(cudaGetLastError());
        set_node_csr(pl, s ^ 1);
        cur ^= 1;          // the level's on-demand dense blocks go to the other buffer (k_cc_union reads the previous one)
    } else if (num_active > 0) {
        dim3 g((max_n + 255) / 256, (max_n + 15) / 16, num_active);
        LAUNCH(SG_PARTITION, k_gather_blocks_cur<<<g, 256, 0, st>>>(e, cur));
        ANCUTS_CUDA(cudaGetLastError());
        cur ^= 1;
    }
    return ANCUTS_OK;
}

// the whole recursion for the chunks described by the plan; W of every chunk is in buffer `cur`, or, with df, written
// after the root split from the root-level forest the input stage built
static int run_levels(ancuts_handle* h, Plan& pl, const ancuts_params* p, int cur, int32_t* d_labels,
                      int32_t* h_num_segments, cudaStream_t st, const DeferredAffinity* df = nullptr) {
    Eng& e = pl.e;
    const int P = e.P, B = e.B;
    ANCUTS_CUDA(cudaMemsetAsync(e.ctr, 0, CTR_COUNT * sizeof(int), st));
    {
        int nmax = 0;
        for (int c = 0; c < B; ++c) nmax = std::max(nmax, pl.n[c]);
        dim3 g((nmax + 255) / 256, B);
        LAUNCH(SG_PARTITION, k_init_positions<<<g, 256, 0, st>>>(e, df ? df->order : nullptr));
        int m = std::max(P, B);
        LAUNCH(SG_PARTITION, k_init_roots<<<(m + 255) / 256, 256, 0, st>>>(e, p->split_lim, p->T));
    }
    int rc = read_ctr(h, e, st);
    if (rc) return rc;
    int num_split = h->h_ctr[5], max_split_n = h->h_ctr[7];
    int guard = 0;
    bool all_fused = false;            // previous level: every node joined its components inside the cluster kernel
    while (num_split > 0) {
        int class_cnt[CL_CLASSES] = {0}, big_cnt = 0;
        rc = run_rebuild(h, pl, cur, num_split, max_split_n, !all_fused, st, class_cnt, &big_cnt, guard == 0 ? df : nullptr,
                         guard > 0);
        if (rc) return rc;
        int num_active = h->h_ctr[1], max_n = h->h_ctr[2];
        if (num_active == 0) break;
        dim3 gdeg((max_n + 7) / 8, num_active);
        if (!e.node_csr) LAUNCH(SG_DEGREE, k_degree<<<gdeg, 256, 0, st>>>(e, cur));   // CSR rows: taken as they were written
        // the split list and the component forest of this level start empty BEFORE the Lanczos launch: cluster kernels that
        // hold their node as CSR slices decide the cut and join the components themselves (cl_fused_cut)
        ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 5, 0, sizeof(int), st));
        ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 7, 0, sizeof(int), st));
        ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 17, 0, 2 * sizeof(int), st));   // nodes decided inside / left over by the cluster kernels
        LAUNCH(SG_PARTITION, k_cc_init<<<(P + 255) / 256, 256, 0, st>>>(e));
        e.fuse_cut = (h->opt[ANCUTS_OPT_FUSED_CUT] == 0) ? 1 : 0;
        h->h_ctr[17] = 0; h->h_ctr[18] = 0;
        if (p->lanczos_impl == 1) rc = run_lanczos(h, e, cur, num_active, max_n, st);
        else rc = run_lanczos_all(h, e, cur, num_active, max_n, class_cnt, big_cnt, st);
        if (rc) return rc;
        // every node of the level decided by cl_fused_cut (the usual case): the counters read back after the cluster kernels
        // already hold the split list, no cut kernel and no second read-back
        all_fused = (h->h_ctr[17] == num_active);
        if (!all_fused) {
            // the few nodes the cluster kernels left over (slices that did not fit, more steps needed) are on a list: the cut
            // kernels run over those only; levels with nodes the cluster kernels never saw (> 4096 points) take every slot
            const int left = num_active - h->h_ctr[17];
            const bool listed = p->lanczos_impl != 1 && big_cnt == 0 && h->h_ctr[18] == left;
            e.sel = listed ? e.unfused : nullptr;
            rc = run_cut(h, e, cur, listed ? left : num_active, max_n, true, st, false);
            e.sel = nullptr;
            if (rc) return rc;
            rc = read_ctr(h, e, st);
            if (rc) return rc;
        }
        num_split = h->h_ctr[5];
        max_split_n = h->h_ctr[7];
        if (++guard > 100000) { set_error("internal: recursion did not terminate"); return ANCUTS_EINVAL; }
    }
    LAUNCH(SG_PARTITION, k_emit_labels<<<(P + 255) / 256, 256, 0, st>>>(e, d_labels, pl.nseg));
    ANCUTS_CUDA(cudaGetLastError());
    if (h_num_segments) {
        ANCUTS_CUDA(cudaMemcpyAsync(h_num_segments, pl.nseg, B * sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    ANCUTS_CUDA(cudaStreamSynchronize(st));
    return ANCUTS_OK;
}

static int copy_stats(ancuts_handle* h, Plan& pl, ancuts_node_stat* h_stats, int stats_cap, int32_t* h_num_stats,
                      cudaStream_t st) {
    int rc = read_ctr(h, pl.e, st);
    if (rc) return rc;
    int cnt = std::min(h->h_ctr[6], stats_cap);
    if (h_num_stats) *h_num_stats = cnt;
    if (h_stats && cnt > 0) {
        ANCUTS_CUDA(cudaMemcpyAsync(h_stats, pl.stats, (size_t)cnt * sizeof(ancuts_node_stat), cudaMemcpyDeviceToHost, st));
        ANCUTS_CUDA(cudaStreamSynchronize(st));
    }
    return ANCUTS_OK;
}

static int check_params(const ancuts_params* p) {
    if (!p) { set_error("params is NULL"); return ANCUTS_EINVAL; }
    if (!(p->proximity >= 0.0)) { set_error("proximity must be >= 0"); return ANCUTS_EINVAL; }
    return ANCUTS_OK;
}

}  // namespace ancuts

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int ancuts_version(void) { return 100; }

const char* ancuts_last_error(void) { return g_err; }

int ancuts_create(int device, ancuts_handle** out) {
    if (!out) { set_error("out is NULL"); return ANCUTS_EINVAL; }
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0) {
        set_error("no CUDA device available (%s); libautoinst_ncuts has no CPU fallback",
                  err != cudaSuccess ? cudaGetErrorString(err) : "device count is 0");
        cudaGetLastError();
        return ANCUTS_ECUDA;
    }
    if (device < 0 || device >= count) { set_error("device %d out of range (0..%d)", device, count - 1); return ANCUTS_EINVAL; }
    ANCUTS_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    ANCUTS_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        return ANCUTS_EUNSUPPORTED;
    }
    ancuts_handle* h = new ancuts_handle();
    h->device = device;
    if (const char* x = getenv("ANCUTS_PHASES")) {
        if (atoi(x)) { ANCUTS_CUDA(cudaMalloc((void**)&h->dbg, 32 * sizeof(unsigned long long))); ANCUTS_CUDA(cudaMemset(h->dbg, 0, 32 * sizeof(unsigned long long))); }
    }
    ANCUTS_CUDA(cudaMallocHost((void**)&h->h_ctr, CTR_COUNT * sizeof(int)));
    for (int i = 0; i < 6; ++i) {
        ANCUTS_CUDA(cudaStreamCreateWithFlags(&h->side[i], cudaStreamNonBlocking));
        ANCUTS_CUDA(cudaEventCreateWithFlags(&h->ev_join[i], cudaEventDisableTiming));
    }
    ANCUTS_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    ANCUTS_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    ANCUTS_CUDA(cudaEventCreateWithFlags(&h->points_ev, cudaEventDisableTiming));
    ANCUTS_CUDA(cudaMallocHost((void**)&h->h_acct, SG_ACCT * sizeof(unsigned long long)));
    *out = h;
    return ANCUTS_OK;
}

int ancuts_destroy(ancuts_handle* h) {
    if (!h) return ANCUTS_OK;
    cudaSetDevice(h->device);
    if (h->ws) cudaFree(h->ws);
    if (h->stage) cudaFree(h->stage);
    if (h->dbg) cudaFree(h->dbg);
    if (h->post_ws) cudaFree(h->post_ws);
    if (h->h_post) cudaFreeHost(h->h_post);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->points_ev) cudaEventDestroy(h->points_ev);
    for (auto ev : h->copy_ev) cudaEventDestroy(ev);
    if (h->h_ctr) cudaFreeHost(h->h_ctr);
    if (h->h_acct) cudaFreeHost(h->h_acct);
    for (auto ev : h->pool) cudaEventDestroy(ev);
    for (int i = 0; i < 6; ++i) { if (h->side[i]) cudaStreamDestroy(h->side[i]); if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]); }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    delete h;
    return ANCUTS_OK;
}

int64_t ancuts_segment_workspace_bytes(int num_chunks, const int32_t* h_chunk_n, int lanczos_max_steps) {
    if (num_chunks <= 0 || !h_chunk_n) return -1;
    Plan pl;
    int kmax = lanczos_max_steps > 0 ? lanczos_max_steps : KMAX_DEFAULT;
    make_plan(pl, num_chunks, h_chunk_n, nullptr, nullptr, kmax, 0);
    pl.deferred = true;                                // upper bound: tensor-core scratch and pair queues both counted
    pl.node_csr = true;                                // and the CSR node form's rows
    return (int64_t)layout(pl, nullptr, 1 << 16, 96, 384, true);
}

int64_t ancuts_launch_count(ancuts_handle* h, int reset) {
    if (!h) return -1;
    int64_t v = h->launches_total;
    if (reset) h->launches_total = 0;
    return v;
}

int ancuts_last_levels(ancuts_handle* h, double* out, int cap_rows) {
    if (!h) return ANCUTS_EINVAL;
    int n = std::min((int)h->levels.size(), cap_rows);
    for (int i = 0; i < n && out; ++i) {
        const LevelRec& l = h->levels[i];
        double* o = out + (size_t)i * 16;
        o[0] = l.num_active; o[1] = l.big; o[2] = l.ms;
        for (int b = 0; b < 6; ++b) { o[3 + b] = l.cls[b]; o[9 + b] = l.cmap[b]; }
        o[15] = 0.0;
    }
    return (int)h->levels.size();
}

int ancuts_debug_phases(ancuts_handle* h, double* out32, int reset) {
    if (!h || !h->dbg) return ANCUTS_EINVAL;
    unsigned long long tmp[32];
    ANCUTS_CUDA(cudaMemcpy(tmp, h->dbg, sizeof(tmp), cudaMemcpyDeviceToHost));
    if (out32) for (int i = 0; i < 32; ++i) out32[i] = (double)tmp[i];
    if (reset) ANCUTS_CUDA(cudaMemset(h->dbg, 0, sizeof(tmp)));
    return ANCUTS_OK;
}

int ancuts_set_option(ancuts_handle* h, int option, int value) {
    if (!h || option < 0 || option >= ANCUTS_OPT_COUNT) { set_error("unknown option %d", option); return ANCUTS_EINVAL; }
    if (option == 0) {
        set_error("option 0 is retired (it selected a dense affinity form of the segment path)");
        return ANCUTS_EINVAL;
    }
    h->opt[option] = value;
    return ANCUTS_OK;
}

int ancuts_last_unconverged(ancuts_handle* h) { return h ? h->last_unconverged : ANCUTS_EINVAL; }

int ancuts_last_sparse_accounting(ancuts_handle* h, double* out2) {
    if (!h || !out2) return ANCUTS_EINVAL;
    out2[0] = h->sparse_entry_steps;
    out2[1] = h->sparse_nnz;
    return ANCUTS_OK;
}

int ancuts_last_reorth_accounting(ancuts_handle* h, double* out2) {
    if (!h || !out2) return ANCUTS_EINVAL;
    out2[0] = h->cl_steps;
    out2[1] = h->cl_full;
    return ANCUTS_OK;
}

int ancuts_set_stage_timing(ancuts_handle* h, int on) {
    if (!h) return ANCUTS_EINVAL;
    h->stage_timing = on;
    return ANCUTS_OK;
}

int ancuts_last_accounting(ancuts_handle* h, double* bytes6, double* ms6, int64_t* launches6) {
    if (!h) return ANCUTS_EINVAL;
    for (int i = 0; i < SG_COUNT; ++i) {
        if (bytes6) bytes6[i] = h->stage_bytes[i];
        if (ms6) ms6[i] = h->stage_ms[i];
        if (launches6) launches6[i] = h->stage_launches[i];
    }
    return ANCUTS_OK;
}

int ancuts_affinity_f32(ancuts_handle* h, int n, const double* d_points, const float* d_tarl, const float* d_dino,
                        const ancuts_params* p, float* d_W, int64_t ld, double* d_rowsum, void* stream) {
    return ancuts_affinity_cams_f32(h, n, d_points, d_tarl, d_dino, 1, p, d_W, ld, d_rowsum, stream);
}

int ancuts_affinity_cams_f32(ancuts_handle* h, int n, const double* d_points, const float* d_tarl, const float* d_dino,
                             int dino_cams, const ancuts_params* p, float* d_W, int64_t ld, double* d_rowsum, void* stream) {
    if (!h || n <= 0 || !d_points || !d_W || ld < n || (ld % 4)) { set_error("bad argument to ancuts_affinity_f32"); return ANCUTS_EINVAL; }
    int rc = check_params(p);
    if (!rc) rc = check_features(p, d_tarl, d_dino, dino_cams);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    ANCUTS_CUDA(cudaSetDevice(h->device));
    Plan pl;
    size_t tcb = (p->affinity_impl == 1) ? affinity_tc_scratch_bytes(n, p->tarl_dim, p->dino_dim) : 0;
    const bool feats = (p->theta != 0.0 && d_tarl) || (p->gamma != 0.0 && d_dino);
    const bool two_pass = p->affinity_impl == 0 && feats;       // spatial only: the one-kernel form
    const int qcap = two_pass ? (int)std::min<long long>(96ll * n, (long long)n * (n - 1) / 2 + 1) : 0;
    const size_t o_tc = align_up((size_t)n, 256) + 256;
    const size_t o_q = o_tc + align_up(tcb, 256) + 256;
    const size_t o_ctr = o_q + align_up((size_t)qcap * sizeof(PairQ), 256);
    size_t need = o_ctr + 256;
    rc = ensure_ws(h, need);
    if (rc) return rc;
    uint8_t* tz = (uint8_t*)h->ws;
    pl.tc_scratch = h->ws + o_tc;
    pl.tc_scratch_bytes = tcb;
    pl.pairq = (PairQ*)(h->ws + o_q);
    pl.qcap = qcap;
    int* qctr = two_pass ? (int*)(h->ws + o_ctr) : nullptr;
    begin_accounting(h);
    if (qctr) ANCUTS_CUDA(cudaMemsetAsync(qctr, 0, 2 * sizeof(int), st));
    rc = run_affinity(h, pl, n, d_points, d_tarl, d_dino, dino_cams, p, d_W, ld, tz, st, qctr);
    if (rc) return rc;
    if (qctr) {
        // queue overflow (flag set by pass 1): the one-kernel form runs, otherwise its CTAs exit at once; no host sync
        const bool use_tarl = p->theta != 0.0 && d_tarl != nullptr, use_dino = p->gamma != 0.0 && d_dino != nullptr;
        dim3 grid((unsigned)((ld + AT - 1) / AT), (n + AT - 1) / AT);
        LAUNCH(SG_AFFINITY, k_affinity_exact<<<grid, 256, 0, st>>>(n, d_points, use_tarl ? d_tarl : nullptr, p->tarl_dim,
                                                                   use_dino ? d_dino : nullptr, p->dino_dim, dino_cams, tz, p->alpha,
                                                                   p->theta, p->gamma, p->proximity, d_W, ld, qctr + 1));
    }
    if (d_rowsum) {
        LAUNCH(SG_DEGREE, k_degree_dense<<<(n + 7) / 8, 256, 0, st>>>(n, d_W, ld, d_rowsum));
        LAUNCH(SG_DEGREE, k_add_scalar<<<(n + 255) / 256, 256, 0, st>>>(n, d_rowsum, -1.0));
    }
    ANCUTS_CUDA(cudaGetLastError());
    if (h->stage_timing) {
        ANCUTS_CUDA(cudaStreamSynchronize(st));
        for (auto& t : h->timed) { float ms = 0.f; if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) h->stage_ms[t.stage] += ms; }
        h->timed.clear();
        h->stage_bytes[SG_AFFINITY] = 4.0 * n * (double)n +
                                      4.0 * n * (3 + (p->theta != 0 ? p->tarl_dim : 0) + (p->gamma != 0 ? dino_cams * p->dino_dim : 0));
    }
    return ANCUTS_OK;
}

int ancuts_degree_normalize_f32(ancuts_handle* h, int n, const float* d_W, int64_t ld, double* d_deg, float* d_M,
                                int64_t ldm, void* stream) {
    if (!h || n <= 0 || !d_W || !d_deg || ld < n || (ld % 4) || (d_M && (ldm < n || (ldm % 4)))) {
        set_error("bad argument to ancuts_degree_normalize_f32");
        return ANCUTS_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ANCUTS_CUDA(cudaSetDevice(h->device));
    begin_accounting(h);
    LAUNCH(SG_DEGREE, k_degree_dense<<<(n + 7) / 8, 256, 0, st>>>(n, d_W, ld, d_deg));
    if (d_M) {
        dim3 g((n + 1023) / 1024, (n + NRM_ROWS - 1) / NRM_ROWS);
        LAUNCH(SG_DEGREE, k_normalize_dense<<<g, 256, 0, st>>>(n, d_W, ld, d_deg, d_M, ldm));
    }
    ANCUTS_CUDA(cudaGetLastError());
    if (h->stage_timing) {
        ANCUTS_CUDA(cudaStreamSynchronize(st));
        for (auto& t : h->timed) { float ms = 0.f; if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) h->stage_ms[t.stage] += ms; }
        h->timed.clear();
        h->stage_bytes[SG_DEGREE] = (d_M ? 12.0 : 4.0) * n * (double)n;
    }
    return ANCUTS_OK;
}

// common set-up for the stage entry points that take explicit node lists on one dense matrix
static int setup_nodes(ancuts_handle* h, Plan& pl, int n_total, float* W0, float* W1, int64_t ld, int num_nodes,
                       const int32_t* h_off, const int32_t* h_n, const ancuts_params* p, int status,
                       cudaStream_t st, int* max_n_out) {
    if (!h || n_total <= 0 || !W0 || ld < n_total || (ld % 4) || num_nodes <= 0 || !h_off || !h_n) {
        set_error("bad argument (n_total=%d ld=%lld num_nodes=%d)", n_total, (long long)ld, num_nodes);
        return ANCUTS_EINVAL;
    }
    ANCUTS_CUDA(cudaSetDevice(h->device));
    int kmax = resolve_kmax(p);
    int nn = n_total;
    int64_t ldu = ld;
    make_plan(pl, 1, &nn, nullptr, &ldu, kmax, num_nodes + 2 * n_total / 3 + 8);
    pl.own_w0 = false; pl.own_w1 = false;
    size_t bytes = layout(pl, nullptr, 1, 0, 0, false);
    int rc = ensure_ws(h, bytes);
    if (rc) return rc;
    layout(pl, h->ws, 1, 0, 0, false);
    pl.hW0[0] = W0; pl.hW1[0] = W1 ? W1 : W0;
    rc = upload_tables(pl, st);
    if (rc) return rc;
    fill_params(pl.e, p, kmax);
    pl.e.w_own = 0; pl.e.w_guard = 1; pl.e.dbg = nullptr; pl.e.pts = nullptr;           // caller's W is read in place: anything may sit next to a block
    pl.e.stats = nullptr; pl.e.stats_cap = 0;
    rc = set_attrs(h, pl.KS);
    if (rc) return rc;
    // host-built range table: the given nodes plus filler leaves so that ranges tile [0, n_total)
    std::vector<int> rs, rn, rst, aid, anch, aslot;
    std::vector<std::pair<int, int>> nodes;
    for (int i = 0; i < num_nodes; ++i) {
        if (h_n[i] <= 0 || h_off[i] < 0 || h_off[i] + h_n[i] > n_total) { set_error("node %d out of range", i); return ANCUTS_EINVAL; }
        nodes.push_back({h_off[i], i});
    }
    std::sort(nodes.begin(), nodes.end());
    int pos = 0, maxn = 0, cslots = 0;
    for (auto& pr : nodes) {
        int i = pr.second;
        if (h_off[i] < pos) { set_error("nodes overlap"); return ANCUTS_EINVAL; }
        if (h_off[i] > pos) { rs.push_back(pos); rn.push_back(h_off[i] - pos); rst.push_back(ST_LEAF); }
        rs.push_back(h_off[i]); rn.push_back(h_n[i]); rst.push_back(status);
        pos = h_off[i] + h_n[i];
        maxn = std::max(maxn, h_n[i]);
    }
    if (pos < n_total) { rs.push_back(pos); rn.push_back(n_total - pos); rst.push_back(ST_LEAF); }
    int R = (int)rs.size();
    std::vector<int> rid(n_total), chunk(R, 0), level(R, 0), pass(2 * R, 1), perm(n_total);
    // active slots in the caller's node order
    aid.resize(num_nodes); anch.resize(num_nodes); aslot.resize(num_nodes);
    for (int r = 0; r < R; ++r) for (int i = 0; i < rn[r]; ++i) rid[rs[r] + i] = r;
    for (int i = 0; i < num_nodes; ++i) {
        aid[i] = rid[h_off[i]];
        anch[i] = (h_n[i] + CH - 1) / CH;
        aslot[i] = cslots;
        cslots += anch[i];
    }
    for (int i = 0; i < n_total; ++i) perm[i] = i;
    Eng& e = pl.e;
    {   // Lanczos bookkeeping the rebuild kernels would have written
        std::vector<int> zeros(num_nodes, DONE_NO), ones(num_nodes, 1);
        std::vector<int> cl((size_t)CL_CLASSES * pl.active_cap, 0);
        int cnt[16] = {0};
        for (int i = 0; i < num_nodes; ++i) {
            int cls = (p->lanczos_impl == 1) ? -1 : cluster_class(h_n[i]);
            if (cls >= 0) cl[(size_t)cls * pl.active_cap + cnt[8 + cls]++] = i; else cnt[14]++;
        }
        ANCUTS_CUDA(cudaMemcpyAsync(e.a_done, zeros.data(), num_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
        ANCUTS_CUDA(cudaMemcpyAsync(e.a_path, ones.data(), num_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
        ANCUTS_CUDA(cudaMemsetAsync(e.a_fused, 0, num_nodes * sizeof(int), st));
        e.fuse_cut = 0;                        // stage entries return the eigenvectors; the cut is its own stage
        ANCUTS_CUDA(cudaMemcpyAsync(e.cl_ids, cl.data(), cl.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        ANCUTS_CUDA(cudaStreamSynchronize(st));
        for (int i = 0; i < CL_CLASSES; ++i) h->h_ctr[8 + i] = cnt[8 + i];
        h->h_ctr[14] = cnt[14];
    }
    ANCUTS_CUDA(cudaMemcpyAsync(e.r_start, rs.data(), R * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.r_n, rn.data(), R * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.r_status, rst.data(), R * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.r_chunk, chunk.data(), R * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.r_level, level.data(), R * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.r_pass, pass.data(), 2 * R * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.rid, rid.data(), n_total * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.perm, perm.data(), n_total * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.a_rid, aid.data(), num_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.split_ids, aid.data(), num_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.a_nch, anch.data(), num_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemcpyAsync(e.a_slot0, aslot.data(), num_nodes * sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaMemsetAsync(e.ctr, 0, 8 * sizeof(int), st));
    ANCUTS_CUDA(cudaMemsetAsync(e.ctr + 16, 0, (CTR_COUNT - 16) * sizeof(int), st));
    ANCUTS_CUDA(cudaMemsetAsync(e.acct, 0, SG_ACCT * sizeof(unsigned long long), st));
    ANCUTS_CUDA(cudaStreamSynchronize(st));
    *max_n_out = maxn;
    return ANCUTS_OK;
}

int ancuts_lanczos_fiedler_batched(ancuts_handle* h, int n_total, const float* d_W, int64_t ld, int num_nodes,
                                   const int32_t* h_node_off, const int32_t* h_node_n, const ancuts_params* p,
                                   double* d_ev, double* h_lambda2, int32_t* h_steps, int32_t* h_converged,
                                   void* stream) {
    int rc = check_params(p);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    for (int i = 0; i < num_nodes; ++i)
        if (h_node_n && h_node_n[i] < 3) { set_error("node %d has %d points; the eigensolver needs n >= 3", i, h_node_n[i]); return ANCUTS_EINVAL; }
    Plan pl;
    int max_n = 0;
    begin_accounting(h);
    rc = setup_nodes(h, pl, n_total, const_cast<float*>(d_W), nullptr, ld, num_nodes, h_node_off, h_node_n, p,
                     ST_ACTIVE, st, &max_n);
    if (rc) return rc;
    Eng& e = pl.e;
    dim3 gdeg((max_n + 7) / 8, num_nodes);
    LAUNCH(SG_DEGREE, k_degree<<<gdeg, 256, 0, st>>>(e, 0));
    {
        int class_cnt[CL_CLASSES], big_cnt = h->h_ctr[14];
        for (int i = 0; i < CL_CLASSES; ++i) class_cnt[i] = h->h_ctr[8 + i];
        rc = run_lanczos_all(h, e, 0, num_nodes, max_n, class_cnt, big_cnt, st);
        if (rc) return rc;
    }
    dim3 gc((max_n + CH - 1) / CH, num_nodes);
    LAUNCH(SG_REORTH, k_ritz<<<gc, 256, (size_t)(e.KS + 32) * 8, st>>>(e));
    LAUNCH(SG_SCAN, k_ev_final<<<(num_nodes + 127) / 128, 128, 0, st>>>(e, num_nodes));
    LAUNCH(SG_SCAN, k_bucket<<<gc, 256, 0, st>>>(e));          // applies sign and unit norm to ev
    ANCUTS_CUDA(cudaGetLastError());
    if (d_ev) ANCUTS_CUDA(cudaMemcpyAsync(d_ev, e.ev, (size_t)n_total * sizeof(double), cudaMemcpyDeviceToDevice, st));
    std::vector<double> th(2 * (size_t)num_nodes);
    std::vector<int> kk(num_nodes), cv(num_nodes);
    ANCUTS_CUDA(cudaMemcpyAsync(th.data(), e.a_theta, th.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaMemcpyAsync(kk.data(), e.a_k, num_nodes * sizeof(int), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaMemcpyAsync(cv.data(), e.a_conv, num_nodes * sizeof(int), cudaMemcpyDeviceToHost, st));
    rc = end_accounting(h, e, st);
    if (rc) return rc;
    for (int i = 0; i < num_nodes; ++i) {
        if (h_lambda2) h_lambda2[i] = 1.0 - th[2 * i];
        if (h_steps) h_steps[i] = kk[i];
        if (h_converged) h_converged[i] = cv[i];
    }
    return ANCUTS_OK;
}

int ancuts_ncut_scan_batched(ancuts_handle* h, int n_total, const float* d_W, int64_t ld, int num_nodes,
                             const int32_t* h_node_off, const int32_t* h_node_n, const double* d_ev,
                             int32_t* h_best_k, double* h_mcut, double* h_costs, uint8_t* d_side, void* stream) {
    if (!d_ev) { set_error("d_ev is NULL"); return ANCUTS_EINVAL; }
    cudaStream_t st = (cudaStream_t)stream;
    ancuts_params p;
    memset(&p, 0, sizeof(p));
    p.T = 1e300;                // every node "splits": the caller wants the best cut and its side flags
    p.proximity = 1.0;
    Plan pl;
    int max_n = 0;
    begin_accounting(h);
    int rc = setup_nodes(h, pl, n_total, const_cast<float*>(d_W), nullptr, ld, num_nodes, h_node_off, h_node_n, &p,
                         ST_ACTIVE, st, &max_n);
    if (rc) return rc;
    Eng& e = pl.e;
    ANCUTS_CUDA(cudaMemcpyAsync(e.ev, d_ev, (size_t)n_total * sizeof(double), cudaMemcpyDeviceToDevice, st));
    ANCUTS_CUDA(cudaMemsetAsync(e.side, 0, n_total, st));
    dim3 gdeg((max_n + 7) / 8, num_nodes);
    LAUNCH(SG_DEGREE, k_degree<<<gdeg, 256, 0, st>>>(e, 0));
    dim3 gc((max_n + CH - 1) / CH, num_nodes);
    LAUNCH(SG_SCAN, k_ev_stats<<<gc, 256, 0, st>>>(e));
    ANCUTS_CUDA(cudaMemsetAsync(e.a_k, 0, num_nodes * sizeof(int), st));
    ANCUTS_CUDA(cudaMemsetAsync(e.a_conv, 0, num_nodes * sizeof(int), st));
    ANCUTS_CUDA(cudaMemsetAsync(e.a_theta, 0, 2 * num_nodes * sizeof(double), st));
    rc = run_cut(h, e, 0, num_nodes, max_n, false, st);
    if (rc) return rc;
    // the reference's mask is ev > t: side kernel stores 0 for the mask side; the ABI returns 1 there
    std::vector<int> bk(num_nodes);
    std::vector<double> mc(num_nodes), cs((size_t)num_nodes * NCUT);
    ANCUTS_CUDA(cudaMemcpyAsync(bk.data(), e.a_bestk, num_nodes * sizeof(int), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaMemcpyAsync(mc.data(), e.a_mcut, num_nodes * sizeof(double), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaMemcpyAsync(cs.data(), e.a_costs, cs.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (d_side) {
        LAUNCH(SG_SCAN, k_mask_from_side<<<(n_total + 255) / 256, 256, 0, st>>>(e, d_side));
    }
    rc = end_accounting(h, e, st);
    if (rc) return rc;
    for (int i = 0; i < num_nodes; ++i) {
        if (h_best_k) h_best_k[i] = bk[i];
        if (h_mcut) h_mcut[i] = mc[i];
    }
    if (h_costs) memcpy(h_costs, cs.data(), cs.size() * sizeof(double));
    return ANCUTS_OK;
}

int ancuts_partition_batched(ancuts_handle* h, int n_total, const float* d_W_in, float* d_W_out, int64_t ld,
                             int num_nodes, const int32_t* h_node_off, const int32_t* h_node_n,
                             const uint8_t* d_side, int split_components, int32_t* d_perm_out,
                             int32_t* h_num_children, int32_t* h_child_off, int32_t* h_child_n, void* stream) {
    if (!d_W_out || !d_side) { set_error("d_W_out / d_side is NULL"); return ANCUTS_EINVAL; }
    cudaStream_t st = (cudaStream_t)stream;
    ancuts_params p;
    memset(&p, 0, sizeof(p));
    p.T = 1.0;
    Plan pl;
    int max_n = 0;
    begin_accounting(h);
    int rc = setup_nodes(h, pl, n_total, const_cast<float*>(d_W_in), d_W_out, ld, num_nodes, h_node_off, h_node_n, &p,
                         ST_SPLIT, st, &max_n);
    if (rc) return rc;
    Eng& e = pl.e;
    // ABI: side 1 = mask (goes first); internal: 0 = mask side
    LAUNCH(SG_PARTITION, k_side_from_mask<<<(n_total + 255) / 256, 256, 0, st>>>(e, d_side));
    // stop rule off for this entry point: every child is kept as an ACTIVE range so it gets gathered
    std::vector<int> big(1, 1);
    ANCUTS_CUDA(cudaMemcpyAsync(const_cast<int*>(e.c_norig), big.data(), sizeof(int), cudaMemcpyHostToDevice, st));
    ANCUTS_CUDA(cudaStreamSynchronize(st));
    if (!split_components)       // sides stay whole: no component roots in the sort key
        ANCUTS_CUDA(cudaMemsetAsync(e.r_pass, 0, 2 * (size_t)(n_total + 1) * sizeof(int), st));
    int cur = 0;
    rc = run_rebuild(h, pl, cur, num_nodes, max_n, split_components != 0, st);
    if (rc) return rc;
    int num_ranges = h->h_ctr[0];
    std::vector<int> rs(num_ranges), rn(num_ranges), rst(num_ranges);
    ANCUTS_CUDA(cudaMemcpyAsync(rs.data(), e.r_start, num_ranges * sizeof(int), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaMemcpyAsync(rn.data(), e.r_n, num_ranges * sizeof(int), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaMemcpyAsync(rst.data(), e.r_status, num_ranges * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (d_perm_out) {
        // perm2 holds the previous (identity) permutation after the swap; val2 = old position per new position
        ANCUTS_CUDA(cudaMemcpyAsync(d_perm_out, e.val2, (size_t)n_total * sizeof(int), cudaMemcpyDeviceToDevice, st));
    }
    rc = end_accounting(h, e, st);
    if (rc) return rc;
    int cnt = 0;
    for (int r = 0; r < num_ranges; ++r) {
        // children of the given nodes only (filler leaves are skipped)
        bool inside = false;
        for (int i = 0; i < num_nodes && !inside; ++i)
            inside = rs[r] >= h_node_off[i] && rs[r] < h_node_off[i] + h_node_n[i];
        if (!inside) continue;
        if (h_child_off) h_child_off[cnt] = rs[r];
        if (h_child_n) h_child_n[cnt] = rn[r];
        ++cnt;
    }
    if (h_num_children) *h_num_children = cnt;
    return ANCUTS_OK;
}

int ancuts_nn_reproject(ancuts_handle* h, int num_query, const double* d_query, int num_source,
                        const double* d_source, const int32_t* d_source_label, double max_radius, int32_t no_label,
                        int32_t* d_out_label, int32_t* d_out_index, void* stream) {
    if (!h || num_query <= 0 || num_source <= 0 || !d_query || !d_source || !d_out_label) {
        set_error("bad argument to ancuts_nn_reproject");
        return ANCUTS_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ANCUTS_CUDA(cudaSetDevice(h->device));
    LAUNCH(SG_PARTITION, k_nn_reproject<<<(num_query + 255) / 256, 256, 0, st>>>(
        num_query, d_query, num_source, d_source, d_source_label, max_radius, no_label, d_out_label, d_out_index));
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

// ---- next row N3 (TARL half): radius-mean pooling of scan-point features onto the major points ----
static size_t pool_sort_tmp_bytes(int m) {
    size_t a = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (unsigned*)nullptr, (unsigned*)nullptr, (int*)nullptr, (int*)nullptr, m, 0, 32);
    return align_up(a, 256);
}

int64_t ancuts_feature_pool_workspace_bytes(int num_scan) {
    if (num_scan < 0) return -1;
    const size_t m = (size_t)std::max(num_scan, 1);
    return (int64_t)(4 * align_up(m * 4, 256) + pool_sort_tmp_bytes((int)m) + 256);
}

int ancuts_feature_pool(ancuts_handle* h, int num_major, const double* d_major, int num_scan, const double* d_scan_points,
                        const float* d_scan_feat, int feat_dim, double radius, const double* h_box_min,
                        const double* h_box_max, int normalise, double* d_out, int32_t* d_out_count, void* d_workspace,
                        int64_t workspace_bytes, void* stream) {
    if (!h || num_major <= 0 || num_scan < 0 || !d_major || !d_out || feat_dim <= 0 || feat_dim > 384 || !(radius > 0.0) ||
        !h_box_min || !h_box_max || (num_scan > 0 && (!d_scan_points || !d_scan_feat))) {
        set_error("bad argument to ancuts_feature_pool");
        return ANCUTS_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ANCUTS_CUDA(cudaSetDevice(h->device));
    if (num_scan == 0) {                         // no scan point at all: every row stays zero (chunk_generation.py:247,255-256)
        ANCUTS_CUDA(cudaMemsetAsync(d_out, 0, (size_t)num_major * feat_dim * sizeof(double), st));
        if (d_out_count) ANCUTS_CUDA(cudaMemsetAsync(d_out_count, 0, (size_t)num_major * sizeof(int32_t), st));
        return ANCUTS_OK;
    }
    if (!d_workspace || workspace_bytes < ancuts_feature_pool_workspace_bytes(num_scan)) {
        set_error("ancuts_feature_pool: workspace of %lld bytes needed", (long long)ancuts_feature_pool_workspace_bytes(num_scan));
        return ANCUTS_EINVAL;
    }
    PoolGrid g;
    double ext = 0.0;
    for (int a = 0; a < 3; ++a) {
        g.lo[a] = h_box_min[a]; g.hi[a] = h_box_max[a];
        if (!(g.hi[a] > g.lo[a])) { set_error("ancuts_feature_pool: empty box"); return ANCUTS_EINVAL; }
        ext = std::max(ext, g.hi[a] - g.lo[a]);
    }
    const double pitch = std::max(radius, ext / 1024.0);       // <= 1024 cells per axis: keys fit 30 bits
    g.inv_h = 1.0 / pitch;
    for (int a = 0; a < 3; ++a) g.n[a] = std::min(1025, (int)std::floor((g.hi[a] - g.lo[a]) * g.inv_h) + 1);
    char* w = (char*)d_workspace;
    const size_t seg = align_up((size_t)num_scan * 4, 256);
    unsigned* keys = (unsigned*)w;  unsigned* keys2 = (unsigned*)(w + seg);
    int* idx = (int*)(w + 2 * seg); int* idx2 = (int*)(w + 3 * seg);
    int* inside = (int*)(w + 4 * seg);
    void* tmp = w + 4 * seg + 256;
    size_t tmp_bytes = pool_sort_tmp_bytes(num_scan);
    ANCUTS_CUDA(cudaMemsetAsync(inside, 0, sizeof(int), st));
    LAUNCH(SG_PARTITION, k_pool_keys<<<(num_scan + 255) / 256, 256, 0, st>>>(num_scan, d_scan_points, g, keys, idx, inside));
    h->launches_total += 1;
    // all 32 key bits: the UINT_MAX keys of the cropped points must end up behind every cell
    ANCUTS_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys, keys2, idx, idx2, num_scan, 0, 32, st));
    const int blocks = (num_major + 7) / 8;
    const double r2 = radius * radius;
    const int fpl = (feat_dim + 31) / 32;
#define POOL_CASE(F) LAUNCH(SG_PARTITION, k_pool_gather<F><<<blocks, 256, 0, st>>>(num_major, d_major, num_scan, d_scan_points, \
        d_scan_feat, feat_dim, g, r2, normalise, keys2, idx2, inside, d_out, d_out_count))
    if (fpl <= 1) POOL_CASE(1); else if (fpl <= 3) POOL_CASE(3); else if (fpl <= 4) POOL_CASE(4); else POOL_CASE(12);
#undef POOL_CASE
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

// Pair stage of the deferred affinity for ALL chunks of the call in four launches (ANCUTS_OPT_PAIR_SEARCH = 0, the default):
// cell sort, tile boxes, tile-pair sweep, root-level unions.  Needs the points only; points_ev (host entry): they have arrived.
static int run_pairs_batched(ancuts_handle* h, Plan& pl, const double* d_points, const ancuts_params* p, cudaEvent_t points_ev,
                             cudaStream_t st) {
    const int B = pl.B;
    ANCUTS_CUDA(cudaMemcpyAsync(pl.c_tile0, pl.tile0.data(), (B + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
    if (points_ev) ANCUTS_CUDA(cudaStreamWaitEvent(st, points_ev, 0));
    LAUNCH(SG_AFFINITY, k_pair_grid_b<<<B, 1024, PG_CELLS * sizeof(int), st>>>(pl.c_n, pl.c_base, d_points, p->proximity,
                                                                              pl.pg_cells, pl.pg_sorted, pl.pg_tmp, pl.pg_spts, pl.pg_grid));
    LAUNCH(SG_AFFINITY, k_tile_boxes<<<dim3(pl.max_tiles, B), PS_T, 0, st>>>(pl.c_n, pl.c_base, pl.c_tile0, pl.pg_spts, pl.tbox));
    const int npair = pl.max_tiles * (pl.max_tiles + 1) / 2;
    LAUNCH(SG_AFFINITY, k_pair_sweep<<<dim3(npair, B), 256, 0, st>>>(pl.c_n, pl.c_base, pl.c_tile0, pl.pg_spts, pl.tbox,
                                                                     p->alpha, p->proximity, pl.pairq, pl.d_qoff, pl.d_qcap, pl.qctr));
    LAUNCH(SG_AFFINITY, k_pair_unions<<<dim3(32, B), 256, 0, st>>>(pl.pairq, pl.d_qoff, pl.d_qcap, pl.qctr, pl.c_base, pl.e.parent));
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

// The same stage with the shuffled 64 x 64 tile sweep over each chunk's whole upper triangle (ANCUTS_OPT_PAIR_SEARCH = 1),
// one launch per chunk that also joins the root-level components while the pairs are at hand.  Needs the points only.
static int run_pairs_shuffled(ancuts_handle* h, Plan& pl, const double* d_points, const ancuts_params* p, cudaStream_t st) {
    for (int c = 0; c < pl.B; ++c) {
        const int n = pl.n[c];
        dim3 grid((unsigned)((pl.ld[c] + AT - 1) / AT), (n + AT - 1) / AT);
        LAUNCH(SG_AFFINITY, k_affinity_pairs<<<grid, 256, 0, st>>>(n, d_points + (size_t)pl.base[c] * 3, p->alpha, p->proximity,
                                                                   nullptr, pl.ld[c], pl.pairq + pl.qoff[c], pl.qcap_c[c],
                                                                   pl.qctr + 2 * c, pl.e.parent, pl.base[c]));
    }
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

// ---- next row N3 (DINOv2 half): per-view feature-map pixel of every major point, then the mean over views ----
int ancuts_dino_view_pixels(ancuts_handle* h, int num_major, const double* d_major_cam, int num_visible,
                            const double* d_visible_cam, double max_dist, const double* h_K, int img_h, int img_w,
                            int map_h, int map_w, int32_t* d_out_pixel, void* stream) {
    if (!h || num_major <= 0 || !d_major_cam || num_visible < 0 || (num_visible > 0 && !d_visible_cam) || !h_K ||
        img_h <= 0 || img_w <= 0 || map_h <= 0 || map_w <= 0 || !d_out_pixel) {
        set_error("bad argument to ancuts_dino_view_pixels");
        return ANCUTS_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ANCUTS_CUDA(cudaSetDevice(h->device));
    LAUNCH(SG_AFFINITY, k_dino_view_pixels<<<(num_major + 255) / 256, 256, 0, st>>>(
        num_major, d_major_cam, num_visible, d_visible_cam, max_dist, h_K[0], h_K[1], h_K[2], h_K[3], h_K[4], h_K[5], h_K[6],
        h_K[7], h_K[8], img_h, img_w, map_h, map_w, d_out_pixel));
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

int ancuts_dino_mean(ancuts_handle* h, int num_major, int num_views, const int32_t* d_view_pixel,
                     const float* const* h_feature_maps, int feat_dim, double* d_out, int32_t* d_out_count, void* stream) {
    if (!h || num_major <= 0 || num_views < 0 || (num_views > 0 && (!d_view_pixel || !h_feature_maps)) || feat_dim <= 0 ||
        feat_dim > 384 || !d_out) {
        set_error("bad argument to ancuts_dino_mean (feat_dim 1 .. 384)");
        return ANCUTS_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ANCUTS_CUDA(cudaSetDevice(h->device));
    const float** d_maps = nullptr;
    if (num_views > 0) {
        int rc = ensure_ws(h, (size_t)num_views * sizeof(float*) + 256);      // the table of map pointers lives in the workspace
        if (rc) return rc;
        d_maps = reinterpret_cast<const float**>(h->ws);
        ANCUTS_CUDA(cudaMemcpyAsync(d_maps, h_feature_maps, (size_t)num_views * sizeof(float*), cudaMemcpyHostToDevice, st));
        ANCUTS_CUDA(cudaStreamSynchronize(st));                              // h_feature_maps is the caller's
    }
    const int blocks = (num_major + 7) / 8;
    const int fpl = (feat_dim + 31) / 32;
#define DINO_CASE(F) LAUNCH(SG_AFFINITY, k_dino_mean<F><<<blocks, 256, 0, st>>>(num_major, num_views, d_view_pixel, d_maps, feat_dim, \
                                                                           d_out, d_out_count))
    if (fpl <= 1) DINO_CASE(1); else if (fpl <= 3) DINO_CASE(3); else if (fpl <= 4) DINO_CASE(4); else DINO_CASE(12);
#undef DINO_CASE
    ANCUTS_CUDA(cudaGetLastError());
    return ANCUTS_OK;
}

// caller graphs of ancuts_segment_csr_f32 (one concatenated CSR, columns local to the row's graph)
struct CsrInput {
    const int64_t* row_ptr;
    const int32_t* col;
    const float* val;
    int64_t nnz;
    const int32_t* norig;      // per graph, or NULL
};

static const char* csr_rule(int kind) {
    switch (kind) {
        case CSR_ROWPTR: return "row_ptr decreases or leaves [0, nnz]";
        case CSR_ROWPTR_ENDS: return "row_ptr[0] != 0 or row_ptr[P] != nnz";
        case CSR_COLUMN: return "column outside [0, n)";
        case CSR_UNSORTED: return "columns not in increasing order";
        case CSR_DUPLICATE: return "duplicate column";
        case CSR_NONFINITE: return "non-finite value";
        case CSR_DIAGONAL: return "stored diagonal entry is not 1";
        case CSR_NO_MIRROR: return "not symmetric: entry (i, j) without entry (j, i)";
        case CSR_ASYMMETRIC: return "not symmetric: value of (i, j) differs from (j, i)";
        default: return "unknown";
    }
}

// Input stage of a CSR call: validation, the w_own rule, root-level components.  The points path's pair stage ends at
// the same state (forest in e.parent, W written after the root split by run_rebuild's deferred branch).
static int run_csr_front(ancuts_handle* h, Plan& pl, const CsrInput& csr, cudaStream_t st) {
    const int B = pl.B;
    int nmax = 0;
    for (int c = 0; c < B; ++c) nmax = std::max(nmax, pl.n[c]);
    const dim3 g((nmax + 256 / CSR_LANES - 1) / (256 / CSR_LANES), B);
    ANCUTS_CUDA(cudaMemsetAsync(pl.csr_err, 0xff, (size_t)B * sizeof(unsigned long long), st));
    ANCUTS_CUDA(cudaMemsetAsync(pl.csr_out, 0, sizeof(int), st));
    LAUNCH(SG_AFFINITY, k_csr_validate<<<g, 256, 0, st>>>(pl.c_base, pl.c_n, pl.P, csr.row_ptr, csr.col, csr.val,
                                                          (long long)csr.nnz, pl.csr_err, pl.csr_out));
    ANCUTS_CUDA(cudaGetLastError());
    std::vector<unsigned long long> herr(B);
    int outside = 0;
    ANCUTS_CUDA(cudaMemcpyAsync(herr.data(), pl.csr_err, (size_t)B * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaMemcpyAsync(&outside, pl.csr_out, sizeof(int), cudaMemcpyDeviceToHost, st));
    ANCUTS_CUDA(cudaStreamSynchronize(st));
    for (int c = 0; c < B; ++c) {
        if (herr[c] == ~0ull) continue;
        const int kind = (int)(herr[c] & 0xff), row = (int)((herr[c] >> 8) & 0x3fffffffu);
        set_error("graph %d, row %d: %s", c, row, csr_rule(kind));
        return ANCUTS_EINVAL;
    }
    // Every stored value in {0} U [2^-126, 2), the range of the library's own affinities: the default forms of the points
    // path apply (shared-memory CSR slices, fused cut, integer widening).  The widening is exact for +0 and positive
    // normal floats; the fixed-point cut sums need non-negative weights (a node's volume bounds its cut weights).
    // Otherwise the plain widening and separate cut kernels, as segment_dense.
    pl.e.w_own = outside ? 0 : 1;
    LAUNCH(SG_PARTITION, k_cc_init<<<(pl.P + 255) / 256, 256, 0, st>>>(pl.e));
    LAUNCH(SG_AFFINITY, k_csr_unions<<<g, 256, 0, st>>>(pl.c_base, pl.c_n, csr.row_ptr, csr.col, csr.val, pl.e.parent));
    ANCUTS_CUDA(cudaGetLastError());
    // algorithmic bytes of validation, unions and scatter: row pointers 8 B per row three times; per stored entry its column
    // and value (8 B) in each of the three passes, the mirror entry's (8 B) in the validation, the position of the column's
    // point (4 B) and the store (4 B) in the scatter
    h->stage_bytes[SG_AFFINITY] = 24.0 * pl.P + 40.0 * (double)csr.nnz;
    return ANCUTS_OK;
}

// Host entry: the inputs of the call arrive on a copy stream, the coordinates of every chunk first (points), then the
// features chunk by chunk (feats[c]).
struct Arrival {
    cudaEvent_t points;
    const cudaEvent_t* feats;
};

static int segment_common(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off, const double* d_points,
                          const float* d_tarl, const float* d_dino, int dcams, const float* d_W_dense, int64_t ld_dense,
                          int num_points_orig, const ancuts_params* p, int32_t* d_labels, int32_t* h_num_segments,
                          ancuts_node_stat* h_stats, int32_t stats_cap, int32_t* h_num_stats, cudaStream_t st,
                          const CsrInput* csr = nullptr, const Arrival* arrival = nullptr) {
    int rc = check_params(p);
    if (!rc && !d_W_dense && !csr) rc = check_features(p, d_tarl, d_dino, dcams);
    if (rc) return rc;
    if (!h || num_chunks <= 0 || !h_chunk_off || !d_labels) { set_error("bad argument to segment"); return ANCUTS_EINVAL; }
    ANCUTS_CUDA(cudaSetDevice(h->device));
    std::vector<int> n(num_chunks), norig(num_chunks);
    for (int c = 0; c < num_chunks; ++c) {
        int64_t d = h_chunk_off[c + 1] - h_chunk_off[c];
        if (d <= 0 || d > (1 << 28)) { set_error("chunk %d has %lld points", c, (long long)d); return ANCUTS_EINVAL; }
        n[c] = (int)d;
        norig[c] = (d_W_dense && num_points_orig > 0) ? num_points_orig : (int)d;
        if (csr && csr->norig) {
            if (csr->norig[c] <= 0) { set_error("graph %d: num_points_orig %d must be positive", c, csr->norig[c]); return ANCUTS_EINVAL; }
            norig[c] = csr->norig[c];
        }
    }
    if (h_chunk_off[num_chunks] - h_chunk_off[0] > 0x7fffffffLL / 4) { set_error("batch too large"); return ANCUTS_EINVAL; }
    const int kmax = resolve_kmax(p);
    Plan pl;
    make_plan(pl, num_chunks, n.data(), norig.data(), nullptr, kmax, 0);
    if (stats_cap < 0) stats_cap = 0;
    const bool need_tc = (p->affinity_impl == 1) && !d_W_dense && !csr;
    pl.csr = csr != nullptr;
    // points input: the deferred form (spatial-only configs too: pass 2 = exp(-alpha d)) unless the tensor-core form writes W
    pl.deferred = !d_W_dense && !csr && p->affinity_impl == 0;
    pl.grid_pairs = pl.deferred && h->opt[ANCUTS_OPT_PAIR_SEARCH] == 0;     // cell-sorted, batched sweep (default) or the shuffled one
    if (pl.grid_pairs) ANCUTS_CUDA(cudaFuncSetAttribute(k_pair_grid_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(PG_CELLS * sizeof(int))));
    // CSR node form: the cell-sorted pair queue with the default eigensolver forms (shared-memory slices, fused cut, cluster
    // kernels).  A dense matvec, the separate cut kernels, the grid-wide Lanczos path and the shuffled pair search (its
    // queue holds input indices) read or build every node's dense block anyway: those calls keep the dense node form.
    pl.node_csr = pl.grid_pairs && h->opt[ANCUTS_OPT_NODE_FORM] == 0 && h->opt[ANCUTS_OPT_MATVEC] == 0 &&
                  h->opt[ANCUTS_OPT_FUSED_CUT] == 0 && p->lanczos_impl != 1;
    size_t bytes = layout(pl, nullptr, stats_cap, p->tarl_dim, p->dino_dim, need_tc);
    rc = ensure_ws(h, bytes);
    if (rc) return rc;
    layout(pl, h->ws, stats_cap, p->tarl_dim, p->dino_dim, need_tc);
    // deferred != NULL: the input stage builds the root-level forest and W is written after the root split (CSR: from the
    // stored entries); otherwise W is whole before the level loop
    DeferredAffinity df{p, d_tarl, d_dino, dcams, arrival ? arrival->feats : nullptr, pl.grid_pairs ? pl.pg_sorted : nullptr};
    if (csr) { df.row_ptr = csr->row_ptr; df.col = csr->col; df.val = csr->val; }
    const DeferredAffinity* deferred = (pl.deferred || pl.csr) ? &df : nullptr;
    rc = upload_tables(pl, st);
    if (rc) return rc;
    fill_params(pl.e, p, kmax);
    pl.e.dbg = h->dbg;
    pl.e.pts = (d_W_dense || csr) ? nullptr : d_points;      // caller weights: hash start vector
    pl.e.w_guard = 0;                         // every node block is written by k_gather_blocks_cur (fringe zeroed)
    pl.e.w_own = d_W_dense ? 0 : 1;           // caller-provided weights may be negative or denormal: plain widening (CSR: run_csr_front)
    pl.e.stats = (h_stats && stats_cap > 0) ? pl.stats : nullptr;
    pl.e.stats_cap = stats_cap;
    rc = set_attrs(h, pl.KS);
    if (rc) return rc;
    begin_accounting(h);
    ANCUTS_CUDA(cudaMemsetAsync(pl.e.acct, 0, SG_ACCT * sizeof(unsigned long long), st));
    const int64_t off0 = h_chunk_off[0];
    if (d_W_dense) {
        ANCUTS_CUDA(cudaMemcpy2DAsync(pl.hW0[0], (size_t)pl.ld[0] * 4, d_W_dense, (size_t)ld_dense * 4, (size_t)n[0] * 4,
                                      n[0], cudaMemcpyDeviceToDevice, st));
    } else if (csr) {
        rc = run_csr_front(h, pl, *csr, st);
        if (rc) return rc;
    } else {
        if (pl.deferred) {
            ANCUTS_CUDA(cudaMemsetAsync(pl.qctr, 0, 2 * (size_t)num_chunks * sizeof(int), st));
            // queue offsets and capacities for the kernels that take every chunk in one launch
            ANCUTS_CUDA(cudaMemcpyAsync(pl.d_qoff, pl.qoff.data(), num_chunks * sizeof(long long), cudaMemcpyHostToDevice, st));
            ANCUTS_CUDA(cudaMemcpyAsync(pl.d_qcap, pl.qcap_c.data(), num_chunks * sizeof(int), cudaMemcpyHostToDevice, st));
            const int gP = (pl.P + 255) / 256;
            LAUNCH(SG_PARTITION, k_cc_init<<<gP, 256, 0, st>>>(pl.e));          // forest of the root-level components
            if (pl.grid_pairs) {
                rc = run_pairs_batched(h, pl, d_points, p, arrival ? arrival->points : nullptr, st);
            } else {
                if (arrival) ANCUTS_CUDA(cudaStreamWaitEvent(st, arrival->points, 0));
                rc = run_pairs_shuffled(h, pl, d_points, p, st);
            }
            if (rc) return rc;
            // host entry: the features arrive chunk by chunk while the pair stage and the root split run; the zero-row flags
            // are then taken per chunk right before its feature pass (run_rebuild)
            if (!arrival && p->theta != 0.0 && d_tarl)
                LAUNCH(SG_AFFINITY, k_zero_rows<<<(pl.P + 7) / 8, 256, 0, st>>>(pl.P, d_tarl, p->tarl_dim, pl.tarl_zero));
            // a pair queue that overflowed (more than 96 in-mask pairs per point on average) leaves W incomplete:
            // redo the batch with the one-kernel form.  One small read-back per call.
            std::vector<int> hq(2 * (size_t)num_chunks);
            ANCUTS_CUDA(cudaMemcpyAsync(hq.data(), pl.qctr, hq.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
            ANCUTS_CUDA(cudaStreamSynchronize(st));
            for (int c = 0; c < num_chunks; ++c)
                if (hq[2 * c + 1] != 0) deferred = nullptr;
            if (!deferred) pl.node_csr = false;             // the one-kernel form writes dense W: dense node form
        } else if (arrival) {
            ANCUTS_CUDA(cudaStreamWaitEvent(st, arrival->points, 0));
        }
        if (!deferred) {
            // W of every chunk written whole: the tensor-core form, or the one-kernel form after an overflow
            for (int c = 0; c < num_chunks; ++c) {
                int64_t o = h_chunk_off[c] - off0;
                if (arrival) ANCUTS_CUDA(cudaStreamWaitEvent(st, arrival->feats[c], 0));
                const float* tz = d_tarl ? d_tarl + (size_t)(h_chunk_off[c]) * p->tarl_dim : nullptr;
                const float* dz = d_dino ? d_dino + (size_t)(h_chunk_off[c]) * dcams * p->dino_dim : nullptr;
                rc = run_affinity(h, pl, n[c], d_points + (size_t)h_chunk_off[c] * 3, tz, dz, dcams, p, pl.hW0[c], pl.ld[c],
                                  pl.tarl_zero + o, st);
                if (rc) return rc;
            }
        }
        double aff_bytes = 0.0;
        for (int c = 0; c < num_chunks; ++c)
            aff_bytes += 4.0 * n[c] * (double)n[c] +
                         4.0 * n[c] * (3 + (p->theta != 0 ? p->tarl_dim : 0) + (p->gamma != 0 ? dcams * p->dino_dim : 0));
        h->stage_bytes[SG_AFFINITY] = aff_bytes;
    }
    pl.e.node_csr = pl.node_csr ? 1 : 0;
    pl.e.dn_list = pl.ncsr_list; pl.e.dn_count = pl.ncsr_count;
    rc = run_levels(h, pl, p, 0, d_labels, h_num_segments, st, deferred);
    if (rc) return rc;
    rc = copy_stats(h, pl, h_stats, stats_cap, h_num_stats, st);
    if (rc) return rc;
    h->last_unconverged = h->h_ctr[16];        // counted by k_decide, read back by copy_stats
    return end_accounting(h, pl.e, st);
}

int ancuts_segment_chunks(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off, const double* d_points,
                          const float* d_tarl, const float* d_dino, const ancuts_params* p, int32_t* d_labels,
                          int32_t* h_num_segments, ancuts_node_stat* h_stats, int32_t stats_cap,
                          int32_t* h_num_stats, void* stream) {
    return ancuts_segment_chunks_cams(h, num_chunks, h_chunk_off, d_points, d_tarl, d_dino, 1, p, d_labels, h_num_segments,
                                      h_stats, stats_cap, h_num_stats, stream);
}

int ancuts_segment_chunks_cams(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off, const double* d_points,
                               const float* d_tarl, const float* d_dino, int dino_cams, const ancuts_params* p,
                               int32_t* d_labels, int32_t* h_num_segments, ancuts_node_stat* h_stats, int32_t stats_cap,
                               int32_t* h_num_stats, void* stream) {
    if (!d_points) { set_error("d_points is NULL"); return ANCUTS_EINVAL; }
    if (h_chunk_off && h_chunk_off[0] != 0) { set_error("h_chunk_off[0] must be 0"); return ANCUTS_EINVAL; }
    return segment_common(h, num_chunks, h_chunk_off, d_points, d_tarl, d_dino, dino_cams, nullptr, 0, 0, p, d_labels,
                          h_num_segments, h_stats, stats_cap, h_num_stats, (cudaStream_t)stream);
}

int ancuts_segment_dense_f32(ancuts_handle* h, int n, const float* d_W, int64_t ld, int num_points_orig,
                             const ancuts_params* p, int32_t* d_labels, int32_t* h_num_segments,
                             ancuts_node_stat* h_stats, int32_t stats_cap, int32_t* h_num_stats, void* stream) {
    if (!d_W || n <= 0 || ld < n) { set_error("bad argument to ancuts_segment_dense_f32"); return ANCUTS_EINVAL; }
    int64_t off[2] = {0, n};
    return segment_common(h, 1, off, nullptr, nullptr, nullptr, 1, d_W, ld, num_points_orig, p, d_labels,
                          h_num_segments, h_stats, stats_cap, h_num_stats, (cudaStream_t)stream);
}

int ancuts_segment_csr_f32(ancuts_handle* h, int num_graphs, const int64_t* h_graph_off, const int64_t* d_row_ptr,
                           const int32_t* d_col, const float* d_val, int64_t nnz, const int32_t* h_num_points_orig,
                           const ancuts_params* p, int32_t* d_labels, int32_t* h_num_segments, ancuts_node_stat* h_stats,
                           int32_t stats_cap, int32_t* h_num_stats, void* stream) {
    if (!d_row_ptr || nnz < 0 || (nnz > 0 && (!d_col || !d_val))) { set_error("bad argument to ancuts_segment_csr_f32"); return ANCUTS_EINVAL; }
    if (h_graph_off && h_graph_off[0] != 0) { set_error("h_graph_off[0] must be 0"); return ANCUTS_EINVAL; }
    CsrInput csr{d_row_ptr, d_col, d_val, nnz, h_num_points_orig};
    return segment_common(h, num_graphs, h_graph_off, nullptr, nullptr, nullptr, 1, nullptr, 0, 0, p, d_labels, h_num_segments,
                          h_stats, stats_cap, h_num_stats, (cudaStream_t)stream, &csr);
}

int ancuts_segment_chunks_host(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off, const double* h_points,
                               const float* h_tarl, const float* h_dino, const ancuts_params* p, int32_t* h_labels,
                               int32_t* h_num_segments, ancuts_node_stat* h_stats, int32_t stats_cap,
                               int32_t* h_num_stats, void* stream) {
    return ancuts_segment_chunks_cams_host(h, num_chunks, h_chunk_off, h_points, h_tarl, h_dino, 1, p, h_labels,
                                           h_num_segments, h_stats, stats_cap, h_num_stats, stream);
}

int ancuts_segment_chunks_cams_host(ancuts_handle* h, int num_chunks, const int64_t* h_chunk_off, const double* h_points,
                                    const float* h_tarl, const float* h_dino, int dino_cams, const ancuts_params* p,
                                    int32_t* h_labels, int32_t* h_num_segments, ancuts_node_stat* h_stats,
                                    int32_t stats_cap, int32_t* h_num_stats, void* stream) {
    if (!h || !h_points || !h_labels || !h_chunk_off || num_chunks <= 0 || !p) { set_error("bad argument to ancuts_segment_chunks_host"); return ANCUTS_EINVAL; }
    if (h_chunk_off[0] != 0) { set_error("h_chunk_off[0] must be 0"); return ANCUTS_EINVAL; }
    cudaStream_t st = (cudaStream_t)stream;
    ANCUTS_CUDA(cudaSetDevice(h->device));
    const size_t P = (size_t)h_chunk_off[num_chunks];
    const bool use_t = h_tarl && p->theta != 0.0, use_d = h_dino && p->gamma != 0.0;
    if (use_d && dino_cams < 1) { set_error("dino_cams must be at least 1 (got %d)", dino_cams); return ANCUTS_EINVAL; }
    const size_t drow = use_d ? (size_t)dino_cams * p->dino_dim : 0;        // floats per point, every camera
    size_t bp = P * 3 * sizeof(double), bt = use_t ? P * p->tarl_dim * sizeof(float) : 0,
           bd = P * drow * sizeof(float), bl = P * sizeof(int32_t);
    size_t total = align_up(bp, 256) + align_up(bt, 256) + align_up(bd, 256) + align_up(bl, 256);
    if (total > h->stage_cap) {
        if (h->stage) cudaFree(h->stage);
        h->stage = nullptr;
        h->stage_cap = 0;
        cudaError_t me = cudaMalloc((void**)&h->stage, total);
        if (me != cudaSuccess) { set_error("staging cudaMalloc(%zu) failed: %s", total, cudaGetErrorString(me)); cudaGetLastError(); return ANCUTS_ENOMEM; }
        h->stage_cap = total;
    }
    char* stage = h->stage;
    double* d_points = (double*)stage;
    float* d_tarl = use_t ? (float*)(stage + align_up(bp, 256)) : nullptr;
    float* d_dino = use_d ? (float*)(stage + align_up(bp, 256) + align_up(bt, 256)) : nullptr;
    int32_t* d_labels = (int32_t*)(stage + align_up(bp, 256) + align_up(bt, 256) + align_up(bd, 256));
    int rc = ANCUTS_OK;
    // copies on their own stream (pinned host memory): the coordinates of every chunk first in one copy, for the pair stage,
    // then the features chunk by chunk with one event each, which arrive while the pair stage and the root split run
    while ((int)h->copy_ev.size() < num_chunks + 1) {
        cudaEvent_t ev;
        ANCUTS_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        h->copy_ev.push_back(ev);
    }
    cudaError_t ce = cudaEventRecord(h->copy_ev[num_chunks], st);           // earlier work on st may still read the staging area
    if (ce == cudaSuccess) ce = cudaStreamWaitEvent(h->copy_stream, h->copy_ev[num_chunks], 0);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_points, h_points, bp, cudaMemcpyHostToDevice, h->copy_stream);
    if (ce == cudaSuccess) ce = cudaEventRecord(h->points_ev, h->copy_stream);
    for (int c = 0; c < num_chunks && ce == cudaSuccess; ++c) {
        const size_t o = (size_t)h_chunk_off[c], m = (size_t)(h_chunk_off[c + 1] - h_chunk_off[c]);
        if (use_t) ce = cudaMemcpyAsync(d_tarl + o * p->tarl_dim, h_tarl + o * p->tarl_dim, m * p->tarl_dim * sizeof(float), cudaMemcpyHostToDevice, h->copy_stream);
        if (ce == cudaSuccess && use_d)
            ce = cudaMemcpyAsync(d_dino + o * drow, h_dino + o * drow, m * drow * sizeof(float), cudaMemcpyHostToDevice, h->copy_stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(h->copy_ev[c], h->copy_stream);
    }
    if (ce != cudaSuccess) { set_error("H2D copy failed: %s", cudaGetErrorString(ce)); rc = ANCUTS_ECUDA; cudaStreamSynchronize(h->copy_stream); }
    const Arrival arrival{h->points_ev, h->copy_ev.data()};
    if (rc == ANCUTS_OK)
        rc = segment_common(h, num_chunks, h_chunk_off, d_points, d_tarl, d_dino, dino_cams, nullptr, 0, 0, p, d_labels,
                            h_num_segments, h_stats, stats_cap, h_num_stats, st, nullptr, &arrival);
    if (rc != ANCUTS_OK) cudaStreamSynchronize(h->copy_stream);        // the caller may release its buffers after an error
    if (rc == ANCUTS_OK) {
        ce = cudaMemcpyAsync(h_labels, d_labels, bl, cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) { set_error("D2H copy failed: %s", cudaGetErrorString(ce)); rc = ANCUTS_ECUDA; }
    }
    return rc;
}

}  // extern "C"
