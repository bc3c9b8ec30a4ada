// handle.cuh — the library handle shared by the translation units of libautoinst_ncuts (engine.cu, map_post.cu).
#pragma once
#include <vector>
#include "common.cuh"

namespace ancuts {

struct TimedLaunch { int stage; cudaEvent_t a, b; int level = -1; };
// one record per recursion level (timing mode 2): node counts per size bin and the time of the cluster phase
struct LevelRec { int num_active, big; int cls[6]; int cmap[6]; double ms; };

}  // namespace ancuts

struct ancuts_handle {
    int device = 0;
    char* ws = nullptr;
    size_t ws_bytes = 0;
    char* stage = nullptr;                   // device staging of host inputs / labels (host entry point)
    size_t stage_cap = 0;
    int* h_ctr = nullptr;                    // pinned, CTR_COUNT ints
    cudaStream_t side[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // one per node size bin
    cudaEvent_t ev_fork = nullptr;
    cudaEvent_t ev_join[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    unsigned long long* h_acct = nullptr;    // pinned, ancuts::SG_ACCT
    double sparse_entry_steps = 0, sparse_nnz = 0;   // shared-memory sparse matvec: sum of k * entries, entries (last call)
    double cl_steps = 0, cl_full = 0;                // cluster kernel: Lanczos steps, steps with the full pass (last call)
    int64_t launches_total = 0;
    int64_t stage_launches[ancuts::SG_COUNT] = {0};
    double stage_bytes[ancuts::SG_COUNT] = {0};
    double stage_ms[ancuts::SG_COUNT] = {0};
    int stage_timing = 0;                    // 0 off, 1 every launch, 2 matvec launches only
    std::vector<ancuts::TimedLaunch> timed;
    std::vector<ancuts::LevelRec> levels;
    std::vector<cudaEvent_t> pool;
    size_t pool_used = 0;
    bool attrs_set = false;
    // Code paths with more than one implementation behind the same results (ancuts_set_option; every one is parity-tested;
    // option 0 is retired):
    int opt[ANCUTS_OPT_COUNT] = {0, 0, 0, 0, 0, 0};
    int last_unconverged = 0;                // eigensolver nodes of the last segment call that stopped at lanczos_max_steps
    cudaStream_t copy_stream = nullptr;      // host entry point: H2D copies run ahead of the affinity kernels
    cudaEvent_t points_ev = nullptr;         // host entry point: the coordinates of every chunk have arrived
    std::vector<cudaEvent_t> copy_ev;        // host entry point: [c] chunk c's features have arrived, [num_chunks] copy fence
    unsigned long long* dbg = nullptr;       // device, 32 entries: phase cycles of the cluster kernel (ANCUTS_PHASES=1)
    char* post_ws = nullptr;                 // map_post.cu (merge / metrics): growable device workspace
    size_t post_ws_bytes = 0;
    long long* h_post = nullptr;             // pinned, 16 x int64: counters read back by the merge / metrics entry points
};
