// C ABI implementation (include/smplgpu.h) over the sm_100a kernels.
// Host side is plain CUDA runtime: device buffers, pinned staging, one stream.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <memory>
#include <mutex>
#include <thread>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/smplgpu.h"
#include "bfs.cuh"
#include "bfs_tiles.cuh"
#include "edt.cuh"
#include "voxelize.cuh"
#include "heuristic.cuh"
#include "model.cuh"
#include "validity.cuh"
#include "validity32.cuh"
#include "validity_warp.cuh"
#include "expand1.cuh"
#include "lattice.cuh"
#include "ik.cuh"
#include "euclid.cuh"

using namespace smplgpu;

static thread_local std::string g_create_error;

struct smplgpu_ctx
{
    int device = 0;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    std::string error;
    int64_t launches = 0;

    // robot
    bool has_robot = false;
    DevModel* h_model = nullptr; // host copy
    DevModel* d_model = nullptr;
    int validity_threads = VALIDITY_THREADS;

    // certified single-precision model (validity32.cuh)
    int precision_mode = SMPLGPU_PRECISION_CERTIFIED_F32;
    bool has_model32 = false;
    std::vector<float> h_blob;
    float* d_blob = nullptr; size_t blob_cap = 0;   // bytes
    int blob_words = 0;
    int v32_threads = V32_THREADS;
    int v32_edge_batch_blocks_per_sm = 0;   // 0: the batched edge kernel does not fit
    int v32_blocks_per_sm = 1;            // resident blocks of states_valid32_kernel per SM (persistent launch)
    int v32_slots = 0, v32_ptrees = 0;
    double e_pos = 0.0, eps_cells = 0.0;
    Grid32 grid32{};
    double fk32_origin[3] = { 0.0, 0.0, 0.0 };   // metres of the model's coordinate 0 (fk_centers32_kernel)
    int* d_prim = nullptr; size_t prim_cap = 0;     // bytes; primitive ids of two chunks in flight
    double* d_deltas = nullptr; size_t deltas_cap = 0;
    int* d_unc_list = nullptr; size_t unc_cap = 0;  // ints
    int* d_unc_mask = nullptr;                      // [unc_cap] per edge: which waypoints are undecided (edges_valid32_kernel)
    int* d_unc_count = nullptr;

    // distance field
    bool has_df = false;
    uint16_t* d_df = nullptr;
    size_t df_cells = 0;
    GridParams grid{};
    double res = 0.0, padding = 0.0;
    double origin[3] = { 0, 0, 0 };
    int dmax_sq = 0;

    // BFS
    bool has_bfs = false;
    BfsGrid bfs{};
    size_t bfs_words = 0, bfs_cells = 0;
    int bfs_levels = 0;
    BfsTiles bfs_tiles{}, bank_tiles{};
    int bfs_mode = SMPLGPU_BFS_AUTO;
    int* d_seed_count = nullptr;

    // bank of stacked BFS grids (one per concurrent planning query)
    bool has_bank = false;
    BfsGrid bank{};
    size_t bank_words = 0, bank_cells = 0;
    int bank_slots = 0, bank_slot_dz = 0, bank_kmax = -1;

    // scratch / staging
    double* d_q0 = nullptr; double* d_q1 = nullptr; size_t q_cap = 0;   // doubles
    uint8_t* d_verdict = nullptr; int* d_counts = nullptr; size_t v_cap = 0;
    void* d_misc = nullptr; size_t misc_cap = 0;
    void* d_vox = nullptr; size_t vox_cap = 0;      // voxeliser: vertices, triangles, per-triangle constants
    void* pinned[2] = { nullptr, nullptr }; size_t pinned_cap = 0;
    void* pinned_out[2] = { nullptr, nullptr }; size_t pinned_out_cap = 0;
    cudaEvent_t ev[2] = { nullptr, nullptr };      // chunk b: kernels + result copies done
    // two expansion batches may be in flight (smplgpu_expand_batch_submit / _wait)
    // expansion batches in flight (smplgpu_expand_batch_submit / _wait): SMPLGPU_EXPAND_BUFFERS of them
    void* exp_in[SMPLGPU_EXPAND_BUFFERS] = { }; size_t exp_in_cap[SMPLGPU_EXPAND_BUFFERS] = { };     // pinned
    void* exp_out[SMPLGPU_EXPAND_BUFFERS] = { }; size_t exp_out_cap[SMPLGPU_EXPAND_BUFFERS] = { };   // pinned
    void* d_exp[SMPLGPU_EXPAND_BUFFERS] = { }; size_t d_exp_cap[SMPLGPU_EXPAND_BUFFERS] = { };
    cudaEvent_t ev_exp[SMPLGPU_EXPAND_BUFFERS] = { };
    int exp_n[SMPLGPU_EXPAND_BUFFERS] = { -1, -1, -1, -1 };
    int64_t exp_resolved_total = 0;   // edges of expansion batches resolved in double, since creation
    cudaEvent_t ev_in[2] = { nullptr, nullptr };   // chunk b: inputs on the device
    cudaStream_t copy_stream = nullptr;
    // asynchronous bank runs (smplgpu_bfs_bank_run_slots_async): their own stream, staging and seed counter
    cudaStream_t bfs_stream = nullptr;
    cudaEvent_t ev_bfs = nullptr;
    void* d_bank_stage = nullptr; size_t bank_stage_cap = 0;
    void* h_bank_stage = nullptr; size_t h_bank_stage_cap = 0;
    int* d_bank_seed_count = nullptr;
    int bank_run_state = 0;               // 0 none, 1 staged on the host (waiting for the device's turn), 2 queued
    // asynchronous bank runs go level by level (bfs_level_step_kernel): launched in chunks, continued when a chunk
    // ends without the device having raised *bank_done (page-locked, mapped)
    volatile int* bank_done = nullptr;
    int bank_next_level = 0;              // first level / super-step of the next chunk; 0 = the run in flight is a cooperative one
    long long bank_level_cap = 0;
    int bank_step_tiles = 0;              // the stepwise run in flight: 0 = one level per launch, else the tile kernel's TILE_RPT
    int bank_step_blocks = 0;
    std::vector<int32_t> staged_slots, staged_seeds, staged_offsets;
    unsigned long long* d_stats = nullptr;
    unsigned long long h_stats[4] = { 0, 0, 0, 0 };
    // bumped whenever an answer of the validity / heuristic entry points may change (robot, field, walls, BFS run):
    // host-side caches of such answers (smplhost::ExpansionCache) compare it
    int64_t scene_epoch = 0;
    // lattice discretisation (smplgpu_set_lattice) and staging of 16-bit coordinates / 8-bit primitive ids
    bool has_lattice = false;
    LatticeParams lattice{};
    int lattice_vals[MAX_DOF] = { };
    int16_t* d_coord = nullptr; size_t coord_cap = 0;   // bytes, two chunks
    uint8_t* d_prim8 = nullptr; size_t prim8_cap = 0;
    // device-resident lattices (smplgpu_lattice_*): one per bank slot
    bool has_lat = false;
    LatticeBank lat{};
    LatticeParams lat_params{};
    LatticeVals lat_vals{};
    double lat_xyz_tol[3] = { 0, 0, 0 };    // smplgpu_lattice_params::xyz_tolerance (the goals of smplgpu_lattice_begin)
    void* d_lat_aux = nullptr;              // deltas | long list | short list
    void* lat_in[SMPLGPU_EXPAND_BUFFERS] = { };  size_t lat_in_cap[SMPLGPU_EXPAND_BUFFERS] = { };   // pinned, mapped: slot | parent
    void* lat_out[SMPLGPU_EXPAND_BUFFERS] = { }; size_t lat_out_cap[SMPLGPU_EXPAND_BUFFERS] = { };  // pinned, mapped: succ | h | count | resolved
    void* d_lat[SMPLGPU_EXPAND_BUFFERS] = { };   size_t d_lat_cap[SMPLGPU_EXPAND_BUFFERS] = { };    // q0 | q1 | active | verdict
    int lat_n[SMPLGPU_EXPAND_BUFFERS] = { -1, -1, -1, -1 };
    int lat_max_n = 0;
    int lat_dof = 0;                               // dof the lattice arrays were sized for
    unsigned long long* lat_resolved = nullptr;   // pinned, mapped: edges the rounds resolved in double (running total)
    bool lat_fused = false;                        // one kernel per round (lattice_round_kernel)
    int lat_prim_stride = 0;                       // successor words of the primitives (smplgpu_lattice_create)
    unsigned long long* d_snap_counters = nullptr; // IK solves of the snap actions: run, converged, per SMPLGPU_SNAP_* kind
    size_t lat_round_smem = 0;
    // smplgpu_expand_state: primitive table, page-locked record array + completion flag, arrival counter
    double* d_x1_deltas = nullptr; int x1_prims = -1; int x1_dof = 0;
    smplgpu_succ_info* x1_out = nullptr; size_t x1_out_cap = 0;   // records; the flag word follows them
    unsigned int* d_x1_done = nullptr;
    unsigned long long x1_seq = 0;
    size_t x1_smem_set = 0;
};

static int fail(smplgpu_ctx* ctx, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) {
        ctx->error = buf;
    } else {
        g_create_error = buf;
    }
    return code;
}

// SMPLGPU_V32_PERSISTENT=1 selects the lane-persistent kernels (A/B switch; measured 1.7x SLOWER than the warp-batched
// ones on B200, see DESIGN.md: kept for the record, off by default)
static bool v32_persistent()
{
    static const bool on = [] {
        const char* e = getenv("SMPLGPU_V32_PERSISTENT");
        return e != nullptr && atoi(e) != 0;
    }();
    return on;
}

// SMPLGPU_WARP_RESOLVE=0 selects the thread-per-item double-precision resolve kernels of round 1 (A/B switch)
static bool warp_resolve()
{
    static const bool on = [] {
        const char* e = getenv("SMPLGPU_WARP_RESOLVE");
        return e == nullptr || atoi(e) != 0;
    }();
    return on;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            return fail(ctx, SMPLGPU_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                       \
        }                                                                                          \
    } while (0)

// A kernel's dynamic shared memory cap (cudaFuncAttributeMaxDynamicSharedMemorySize) belongs to the process and the
// device, not to a context: contexts of different robots size the same kernels differently, so a context only ever
// raises the cap to what its own launches need.  Setting it to a smaller context's size would make every launch of a
// larger context in the same process fail with an invalid argument.
template <class K>
static cudaError_t raise_smem_cap(K* kernel, int smem)
{
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, kernel);
    if (e != cudaSuccess || a.maxDynamicSharedSizeBytes >= smem) {
        return e;
    }
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

static int grow(smplgpu_ctx* ctx, void** p, size_t* cap, size_t need)
{
    if (need <= *cap) {
        return 0;
    }
    if (*p) {
        CU(cudaFree(*p));
        *p = nullptr;
        *cap = 0;
    }
    size_t n = std::max(need, (size_t)1 << 16);
    CU(cudaMalloc(p, n));
    *cap = n;
    return 0;
}

static int grow_pinned(smplgpu_ctx* ctx, void** p, size_t* cap, size_t need)
{
    if (need <= *cap) {
        return 0;
    }
    for (int i = 0; i < 2; ++i) {
        if (p[i]) {
            CU(cudaFreeHost(p[i]));
            p[i] = nullptr;
        }
    }
    *cap = 0;
    for (int i = 0; i < 2; ++i) {
        CU(cudaMallocHost(&p[i], need));
    }
    *cap = need;
    return 0;
}

static int ensure_state_buffers(smplgpu_ctx* ctx, size_t n, int dof, bool edges)
{
    size_t need_q = n * (size_t)dof * sizeof(double);
    if (need_q > ctx->q_cap) {
        if (ctx->d_q0) { CU(cudaFree(ctx->d_q0)); ctx->d_q0 = nullptr; }
        if (ctx->d_q1) { CU(cudaFree(ctx->d_q1)); ctx->d_q1 = nullptr; }
        ctx->q_cap = 0;
        CU(cudaMalloc(&ctx->d_q0, need_q));
        CU(cudaMalloc(&ctx->d_q1, need_q));
        ctx->q_cap = need_q;
    }
    if (n > ctx->v_cap) {
        if (ctx->d_verdict) { CU(cudaFree(ctx->d_verdict)); ctx->d_verdict = nullptr; }
        if (ctx->d_counts) { CU(cudaFree(ctx->d_counts)); ctx->d_counts = nullptr; }
        ctx->v_cap = 0;
        CU(cudaMalloc(&ctx->d_verdict, n));
        CU(cudaMalloc(&ctx->d_counts, n * sizeof(int)));
        ctx->v_cap = n;
    }
    (void)edges;
    return 0;
}

extern "C" {

smplgpu_ctx* smplgpu_create(int device)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        fail(nullptr, SMPLGPU_ERR_NO_DEVICE, "no CUDA device: %s (there is no CPU fallback)",
             e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return nullptr;
    }
    if (device < 0 || device >= count) {
        fail(nullptr, SMPLGPU_ERR_INVALID, "device %d out of range (count %d)", device, count);
        return nullptr;
    }
    smplgpu_ctx* ctx = new smplgpu_ctx;
    ctx->device = device;
    auto bail = [&](const char* what, cudaError_t err) {
        fail(nullptr, SMPLGPU_ERR_CUDA, "%s: %s", what, cudaGetErrorString(err));
        delete ctx;
        return (smplgpu_ctx*)nullptr;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    ctx->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    ctx->stream = ctx->own_stream;
    if ((e = cudaMalloc(&ctx->d_model, sizeof(DevModel))) != cudaSuccess) return bail("cudaMalloc(model)", e);
    if ((e = cudaMalloc(&ctx->d_stats, 4 * sizeof(unsigned long long))) != cudaSuccess) return bail("cudaMalloc(stats)", e);
    if ((e = cudaMalloc(&ctx->d_seed_count, sizeof(int))) != cudaSuccess) return bail("cudaMalloc(seed)", e);
    if ((e = cudaMalloc(&ctx->d_unc_count, 2 * sizeof(int))) != cudaSuccess) return bail("cudaMalloc(unc)", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    {
        // the stream of the bank runs queued behind the caller's back: highest priority, so that the block scheduler
        // prefers a waiting wavefront kernel's blocks to the next expansion round's when an SM drains
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        if ((e = cudaStreamCreateWithPriority(&ctx->bfs_stream, cudaStreamNonBlocking, prio_hi)) != cudaSuccess) return bail("cudaStreamCreate", e);
    }
    if ((e = cudaEventCreateWithFlags(&ctx->ev_bfs, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaMalloc(&ctx->d_bank_seed_count, sizeof(int))) != cudaSuccess) return bail("cudaMalloc(seed)", e);
    for (int i = 0; i < 2; ++i) {
        if ((e = cudaEventCreateWithFlags(&ctx->ev[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
        if ((e = cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    }
    for (int i = 0; i < SMPLGPU_EXPAND_BUFFERS; ++i) {
        if ((e = cudaEventCreateWithFlags(&ctx->ev_exp[i], cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    }
    ctx->h_model = new DevModel;
    memset(ctx->h_model, 0, sizeof(DevModel));
    if (const char* e = getenv("SMPLGPU_BFS_MODE")) {   // experiments: 0 tiles, 1 levels, 2 auto (smplgpu_bfs_set_mode)
        const int m = atoi(e);
        if (m >= 0 && m <= 2) ctx->bfs_mode = m;
    }
    return ctx;
}

static void free_tiles(BfsTiles& t)
{
    cudaFree(t.tb[0]); cudaFree(t.ver);
    memset(&t, 0, sizeof(t));
}

static int alloc_tiles(smplgpu_ctx* ctx, const BfsGrid& g, BfsTiles& t, size_t words)
{
    free_tiles(t);
    t.ntx = (g.DX + 31) / 32;
    t.nty = (g.DY + TILE_Y - 1) / TILE_Y;
    t.ntz = (g.DZ + TILE_Y - 1) / TILE_Y;
    t.ntiles = t.ntx * t.nty * t.ntz;
    (void)words;
    {
        // the four tile-major bitmaps (two blocked copies, two frontiers) in one allocation
        const size_t tw = (size_t)t.ntiles * TILE_WORDS;
        CU(cudaMalloc(&t.tb[0], 4 * tw * sizeof(uint32_t)));
        t.tb[1] = t.tb[0] + tw;
        t.tf[0] = t.tb[0] + 2 * tw;
        t.tf[1] = t.tb[0] + 3 * tw;
    }
    // ver[ntiles] | flag[3][ntiles] | queue[3][ntiles] | qn[3] (+ pad), all 32-bit
    CU(cudaMalloc(&t.ver, ((size_t)7 * t.ntiles + 16) * sizeof(uint32_t)));
    t.flag = t.ver + t.ntiles;
    t.queue = reinterpret_cast<int*>(t.flag + (size_t)3 * t.ntiles);
    t.qn = t.queue + (size_t)3 * t.ntiles;
    return 0;
}

static void free_grid(BfsGrid& g)
{
    cudaFree(g.wall); cudaFree(g.blocked); cudaFree(g.front0); cudaFree(g.front1);
    cudaFree(g.cand0); cudaFree(g.cand1);
    cudaFree(g.dist); cudaFree(g.ctrl);
    memset(&g, 0, sizeof(g));
}

static void free_bfs(smplgpu_ctx* ctx)
{
    free_grid(ctx->bfs);
    free_tiles(ctx->bfs_tiles);
    ctx->has_bfs = false;
}

static int finish_bank_run(smplgpu_ctx* ctx);   // waits for an asynchronous bank run (defined with the bank)

static void free_lattice(smplgpu_ctx* ctx)
{
    cudaFree(ctx->lat.q); cudaFree(ctx->lat.coord); cudaFree(ctx->lat.gdist); cudaFree(ctx->lat.table);
    cudaFree(ctx->lat.count); cudaFree(ctx->lat.goal); cudaFree(ctx->lat.n_goals); cudaFree(ctx->d_lat_aux);
    if (ctx->lat_resolved) cudaFreeHost(ctx->lat_resolved);
    ctx->lat_resolved = nullptr;
    memset(&ctx->lat, 0, sizeof(ctx->lat));
    ctx->d_lat_aux = nullptr;
    for (int b = 0; b < SMPLGPU_EXPAND_BUFFERS; ++b) {
        if (ctx->lat_in[b]) cudaFreeHost(ctx->lat_in[b]);
        if (ctx->lat_out[b]) cudaFreeHost(ctx->lat_out[b]);
        cudaFree(ctx->d_lat[b]);
        ctx->lat_in[b] = ctx->lat_out[b] = ctx->d_lat[b] = nullptr;
        ctx->lat_in_cap[b] = ctx->lat_out_cap[b] = ctx->d_lat_cap[b] = 0;
        ctx->lat_n[b] = -1;
    }
    ctx->has_lat = false;
    ctx->lat_max_n = 0;
}

void smplgpu_destroy(smplgpu_ctx* ctx)
{
    if (!ctx) {
        return;
    }
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    finish_bank_run(ctx);
    if (ctx->bfs_stream) cudaStreamSynchronize(ctx->bfs_stream);
    free_bfs(ctx);
    free_grid(ctx->bank);
    free_tiles(ctx->bank_tiles);
    cudaFree(ctx->d_snap_counters);
    cudaFree(ctx->d_model); cudaFree(ctx->d_stats); cudaFree(ctx->d_seed_count); cudaFree(ctx->d_df);
    cudaFree(ctx->d_blob); cudaFree(ctx->d_unc_list); cudaFree(ctx->d_unc_mask); cudaFree(ctx->d_unc_count);
    cudaFree(ctx->d_prim); cudaFree(ctx->d_deltas);
    cudaFree(ctx->d_q0); cudaFree(ctx->d_q1); cudaFree(ctx->d_verdict); cudaFree(ctx->d_counts); cudaFree(ctx->d_misc); cudaFree(ctx->d_vox);
    for (int i = 0; i < 2; ++i) {
        if (ctx->pinned[i]) cudaFreeHost(ctx->pinned[i]);
        if (ctx->pinned_out[i]) cudaFreeHost(ctx->pinned_out[i]);
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
        if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
    }
    for (int i = 0; i < SMPLGPU_EXPAND_BUFFERS; ++i) {
        if (ctx->ev_exp[i]) cudaEventDestroy(ctx->ev_exp[i]);
        if (ctx->exp_in[i]) cudaFreeHost(ctx->exp_in[i]);
        if (ctx->exp_out[i]) cudaFreeHost(ctx->exp_out[i]);
        cudaFree(ctx->d_exp[i]);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->bfs_stream) cudaStreamDestroy(ctx->bfs_stream);
    if (ctx->ev_bfs) cudaEventDestroy(ctx->ev_bfs);
    cudaFree(ctx->d_bank_stage); cudaFree(ctx->d_bank_seed_count);
    if (ctx->bank_done) cudaFreeHost((void*)ctx->bank_done);
    cudaFree(ctx->d_x1_deltas); cudaFree(ctx->d_x1_done);
    cudaFree(ctx->d_coord); cudaFree(ctx->d_prim8);
    free_lattice(ctx);
    if (ctx->x1_out) cudaFreeHost(ctx->x1_out);
    if (ctx->h_bank_stage) cudaFreeHost(ctx->h_bank_stage);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx->h_model;
    delete ctx;
}

const char* smplgpu_last_error(const smplgpu_ctx* ctx)
{
    return ctx ? ctx->error.c_str() : g_create_error.c_str();
}

int smplgpu_device(const smplgpu_ctx* ctx) { return ctx ? ctx->device : -1; }

int smplgpu_bind_thread(smplgpu_ctx* ctx)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    CU(cudaSetDevice(ctx->device));
    return 0;
}

int smplgpu_set_stream(smplgpu_ctx* ctx, void* cuda_stream)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return 0;
}

int smplgpu_synchronize(smplgpu_ctx* ctx)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int64_t smplgpu_launch_count(const smplgpu_ctx* ctx) { return ctx ? ctx->launches : 0; }

int64_t smplgpu_scene_epoch(const smplgpu_ctx* ctx) { return ctx ? ctx->scene_epoch : -1; }

///////////////////////////////////////////////////////////////////////////////
// robot
///////////////////////////////////////////////////////////////////////////////

// ok  <=>  (res*sqrt(d2))^2 >= (r+pad)^2, evaluated exactly like
// collision_operations.h:74-76 over distance_map.hpp:142-146, 298-299
static int sphere_threshold(double res, int dmax_sq, double radius, double padding)
{
    const double eff = radius + padding;
    const double eff2 = eff * eff;
    for (int k = 0; k <= dmax_sq; ++k) {
        const double d = res * std::sqrt((double)k);
        if (d * d >= eff2) {
            return k;
        }
    }
    return dmax_sq + 1;
}

///////////////////////////////////////////////////////////////////////////////
// certified single-precision model
///////////////////////////////////////////////////////////////////////////////

static double norm3(const double* v) { return std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }

// origin * joint_fn(value) in double, for joints whose value is a constant of the scene
static void const_joint_transform(int fn, const double* o, const double* axis, double val, double* t)
{
    double R[12] = { 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0 };
    const double s = std::sin(val), c = std::cos(val);
    if (fn == 1) { R[5] = c; R[6] = -s; R[9] = s; R[10] = c; }
    else if (fn == 2) { R[0] = c; R[2] = s; R[8] = -s; R[10] = c; }
    else if (fn == 3) { R[0] = c; R[1] = -s; R[4] = s; R[5] = c; }
    else if (fn == 4) {
        const double k = 1.0 - c, x = axis[0], y = axis[1], z = axis[2];
        R[0] = k * x * x + c;     R[1] = k * x * y - s * z; R[2] = k * x * z + s * y;
        R[4] = k * x * y + s * z; R[5] = k * y * y + c;     R[6] = k * y * z - s * x;
        R[8] = k * x * z - s * y; R[9] = k * y * z + s * x; R[10] = k * z * z + c;
    } else if (fn == 5) { R[11] = val; }
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 4; ++j) {
            t[4 * i + j] = o[4 * i] * R[j] + o[4 * i + 1] * R[4 + j] + o[4 * i + 2] * R[8 + j] + (j == 3 ? o[4 * i + 3] : 0.0);
        }
    }
}

// a (3x4) * b (3x4), double
static void mul34(const double* a, const double* b, double* r)
{
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 4; ++j) {
            r[4 * i + j] = a[4 * i] * b[j] + a[4 * i + 1] * b[4 + j] + a[4 * i + 2] * b[8 + j] + (j == 3 ? a[4 * i + 3] : 0.0);
        }
    }
}

// The single-precision kernels walk a state's link chain once per state and pay a 3x4 product per link, so links
// whose joint is a CONSTANT of the scene (fixed joints, non-planning joints: half of the PR2 arm group's 14 links)
// are folded away here: a constant link's spheres are re-expressed in the frame of the nearest moving ancestor
// (c' = C c, C = the product of the constant joint transforms in between, in double), and a moving link below a
// constant one takes C into its joint origin (T = T_anchor (C O) R(q)).  World positions are the same up to
// rounding, which the error bounds below -- computed from THIS table -- cover; the double-precision kernels keep
// the reference's link-by-link operation order.  Constant links without a parent in the table keep their entry.
// SMPLGPU_V32_FOLD=0 disables the folding (A/B).
static void fold_constant_links(const DevModel& m, DevModel& F)
{
    F = m;
    static const bool enabled = [] {
        const char* e = getenv("SMPLGPU_V32_FOLD");
        return e == nullptr || atoi(e) != 0;
    }();
    if (!enabled) {
        return;
    }
    const int nl = m.n_links;
    std::vector<int> new_index(nl, -1), carrier(nl, -1);
    std::vector<std::array<double, 12>> C(nl);
    const double I12[12] = { 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0 };
    int n_new = 0;
    for (int l = 0; l < nl; ++l) {
        const int p = m.link_parent[l];
        const bool is_const = m.link_var[l] < 0;
        if (is_const && p >= 0) {
            // folded: its frame = carrier frame * C[l]
            double J[12];
            const_joint_transform(m.link_joint[l], m.link_origin[l], m.link_axis[l], m.link_const[l], J);
            const bool parent_kept = new_index[p] >= 0;
            carrier[l] = parent_kept ? new_index[p] : carrier[p];
            mul34(parent_kept ? I12 : C[p].data(), J, C[l].data());
            continue;
        }
        const int L = n_new++;
        new_index[l] = L;
        carrier[l] = L;
        memcpy(C[l].data(), I12, sizeof(I12));
        F.link_joint[L] = m.link_joint[l];
        F.link_var[L] = m.link_var[l];
        F.link_const[L] = m.link_const[l];
        memcpy(F.link_axis[L], m.link_axis[l], sizeof(m.link_axis[l]));
        memcpy(F.link_base[L], m.link_base[l], sizeof(m.link_base[l]));
        if (p >= 0 && new_index[p] < 0) {
            F.link_parent[L] = carrier[p];
            mul34(C[p].data(), m.link_origin[l], F.link_origin[L]);   // T = T_anchor * (C O) * R(q)
        } else {
            F.link_parent[L] = p < 0 ? -1 : new_index[p];
            memcpy(F.link_origin[L], m.link_origin[l], sizeof(m.link_origin[l]));
        }
    }
    F.n_links = n_new;
    // spheres ride on their link's carrier, centres in the carrier's frame
    for (int n = 0; n < m.n_nodes; ++n) {
        const int l = m.node_link[n];
        F.node_link[n] = carrier[l];
        if (new_index[l] < 0) {
            const double* c = m.node_center[n];
            const double* T = C[l].data();
            for (int i = 0; i < 3; ++i) {
                F.node_center[n][i] = T[4 * i] * c[0] + T[4 * i + 1] * c[1] + T[4 * i + 2] * c[2] + T[4 * i + 3];
            }
        }
    }
    // trees grouped by (new) link, in the order the double kernels visit them
    int k = 0;
    std::vector<int> order;
    for (int l = 0; l < nl; ++l) {
        for (int ti = m.link_tree_begin[l]; ti < m.link_tree_end[l]; ++ti) order.push_back(m.tree_by_link[ti]);
    }
    for (int L = 0; L < n_new; ++L) {
        F.link_tree_begin[L] = k;
        for (int t : order) {
            if (F.node_link[m.tree_root[t]] == L) F.tree_by_link[k++] = t;
        }
        F.link_tree_end[L] = k;
    }
    // slots: transforms the kernels keep per thread = branching parents + links that carry a paired tree
    std::vector<char> keep(n_new, 0);
    for (int L = 0; L < n_new; ++L) {
        const int p = F.link_parent[L];
        if (p >= 0 && p != L - 1) keep[p] = 1;
    }
    for (int pi = 0; pi < m.n_pairs; ++pi) {
        keep[F.node_link[m.tree_root[m.pair_a[pi]]]] = 1;
        keep[F.node_link[m.tree_root[m.pair_b[pi]]]] = 1;
    }
    int slots = 0;
    for (int L = 0; L < n_new; ++L) F.link_slot[L] = keep[L] ? slots++ : -1;
    F.n_slots = slots;
}

// Builds the shared-memory blob of validity32.cuh and the error bounds that certify it.
//
// The blob is in GRID UNITS: with s = inv_res and o the grid's (ox, oy, oz), every link-origin translation, sphere
// centre and radius is scaled by s, the rotation blocks are left as they are, and the base transform of a root link
// (world <- root, [R_b | t_b]) becomes [R_b | s (t_b - o) - 1 - K], K the whole cell of the first root link's origin.
// The chain then yields c - K, where c = s (x - o) - 1 for a centre x in metres is the grid coordinate whose
// round-to-nearest is the reference's cell; the lookup adds K back in its integer index step (validity32.cuh:
// lookup32).  With K taken out, the chain's translations are lengths along the robot, not distances from the grid
// origin, which keeps the rounding terms 7u tn below small.  A
// moving prismatic joint keeps q in joint units: its axis slot holds s times the third origin column.
//
// Error model (u = 2^-24, all norms Euclidean, all lengths in cells; R = rotation part, t = translation part of a
// link transform):
//   joint transform J(q):  ||dR_J||_F <= 3.5u (constant), 40u (axis-aligned revolute: sincosf <= 2 ulp, hi/lo
//                          angle split, 2 roundings per entry), 80u (general axis); ||dt_J|| <= u ||t_J|| (+ 4u s |q|max
//                          for a prismatic joint, whose low part of q is dropped)
//   base transform:        ||dR_B||_F <= 3.5u, ||dt_B|| <= u ||t_B||, t_B = s (t_b - o) - 1 - K (formed in double, rounded
//                          once to float): the world -> grid map's own rounding is this one term
//   product T = P J:       ||dR_T||_F <= ||dR_P||_F + ||dR_J||_F + 12u                  (||R|| = 1)
//                          ||dt_T||   <= ||dt_P|| + ||dR_P||_F ||t_J|| + ||dt_J|| + 7u tn,   tn >= ||t_T||
//   centre  c = T y:       ||dc||     <= ||dt_T|| + ||dR_T||_F ||y|| + 7u (tn + ||y||) + u ||y||
// E = 1.5 * max over nodes bounds |c_f32 - c_f64| (the factor covers the double chain's own rounding).  The lookup
// forms its cell and remainder exactly (lookup32) and compares the remainder against 1/2 - eps in float, which rounds
// by at most 2^-26; the reference rounds its double grid coordinate by ~2^-53 |c|.  Both sit in the 1e-7 of
// eps_cells = E + 1e-7.  Since E >= 10.5u (tn + ||y||) >= 10.5u |c - K|, eps_cells < 0.125 also means |c - K| < 2^21
// for every centre the kernels evaluate (joints beyond V32_MAX_ANGLE or q_lin_max go to the double path first), where
// lookup32's rounding is exact; the check of that below only restates it.  |K| < 2^21 keeps the index in int range.  The pair tests compare squared
// distances in cells, which scale with s^2 on both sides, with the tolerance 2.5 E (d + r) + 2e-6 (d^2 + r^2).
static int build_model32(smplgpu_ctx* ctx)
{
    ctx->has_model32 = false;
    if (!ctx->has_robot || !ctx->has_df) {
        return 0;
    }
    std::unique_ptr<DevModel> folded(new DevModel);
    fold_constant_links(*ctx->h_model, *folded);
    const DevModel& m = *folded;
    if (m.n_nodes >= 65536) {
        return 0; // node ids are packed in 16 bits in the pair descent: fall back to the double path
    }
    const double u = std::ldexp(1.0, -24);
    const int nl = m.n_links, nn = m.n_nodes;

    // ---- pre-order renumbering, trees grouped by link ----
    std::vector<int> new_of(nn, -1), orig_of, skip, link_nbeg(nl), link_nend(nl);
    orig_of.reserve(nn);
    for (int l = 0; l < nl; ++l) {
        link_nbeg[l] = (int)orig_of.size();
        for (int ti = m.link_tree_begin[l]; ti < m.link_tree_end[l]; ++ti) {
            // iterative pre-order (left child first)
            std::vector<int> st(1, m.tree_root[m.tree_by_link[ti]]);
            while (!st.empty()) {
                const int node = st.back();
                st.pop_back();
                new_of[node] = (int)orig_of.size();
                orig_of.push_back(node);
                if (m.node_left[node] >= 0) {
                    st.push_back(m.node_right[node]);
                    st.push_back(m.node_left[node]);
                }
            }
        }
        link_nend[l] = (int)orig_of.size();
    }
    const int n32 = (int)orig_of.size();   // nodes reachable from a tree root
    skip.assign(n32, 0);
    {
        // subtree sizes: skip[i] = i + size(i)
        std::vector<int> size(nn, 0);
        for (int i = n32 - 1; i >= 0; --i) {
            const int node = orig_of[i];
            size[node] = 1;
            if (m.node_left[node] >= 0) {
                size[node] += size[m.node_left[node]] + size[m.node_right[node]];
            }
            skip[i] = i + size[node];
        }
    }

    // ---- error bounds (cells) ----
    const double sc = ctx->grid.inv_res;
    const double go[3] = { ctx->grid.ox, ctx->grid.oy, ctx->grid.oz };
    // whole-cell offset K: the grid cell of the first root link's origin (validity32.cuh: Grid32)
    double K[3] = { 0.0, 0.0, 0.0 };
    for (int l = 0; l < nl; ++l) {
        if (m.link_parent[l] < 0) {
            for (int i = 0; i < 3; ++i) K[i] = std::nearbyint(sc * (m.link_base[l][4 * i + 3] - go[i]) - 1.0);
            break;
        }
    }
    auto base_t = [&](int l, int i) { return sc * (m.link_base[l][4 * i + 3] - go[i]) - 1.0 - K[i]; };
    std::vector<double> EF(nl), Et(nl), tn(nl);
    double q_lin_max = 0.0;
    for (int v = 0; v < m.dof; ++v) {
        if (m.var_type[v] == 2) {
            double lim = std::max(std::fabs(m.var_min[v]), std::fabs(m.var_max[v]));
            if (!std::isfinite(lim)) lim = 4.0;
            q_lin_max = std::max(q_lin_max, lim + 1.0);
        }
    }
    const double q_lin_cells = sc * q_lin_max;
    double e_max = 0.0, c_max = 0.0;
    for (int l = 0; l < nl; ++l) {
        const int fn = m.link_joint[l];
        const bool moving = m.link_var[l] >= 0;
        const double* o = m.link_origin[l];
        const double to[3] = { sc * o[3], sc * o[7], sc * o[11] };
        double EF_J, Et_J, tJ;
        if (!moving || fn == 0) {
            EF_J = 3.5 * u;
            tJ = norm3(to) + ((fn == 5) ? sc * std::fabs(m.link_const[l]) : 0.0);
            Et_J = u * tJ;
        } else if (fn <= 3) {
            EF_J = 40.0 * u; tJ = norm3(to); Et_J = u * tJ;
        } else if (fn == 4) {
            EF_J = 80.0 * u; tJ = norm3(to); Et_J = u * tJ;
        } else {
            EF_J = 3.5 * u; tJ = norm3(to) + q_lin_cells; Et_J = u * tJ + 4.0 * u * q_lin_cells;
        }
        double EF_P, Et_P, tn_P;
        const int p = m.link_parent[l];
        if (p < 0) {
            const double tb[3] = { base_t(l, 0), base_t(l, 1), base_t(l, 2) };
            EF_P = 3.5 * u; tn_P = norm3(tb); Et_P = u * tn_P;
        } else {
            EF_P = EF[p]; Et_P = Et[p]; tn_P = tn[p];
        }
        EF[l] = EF_P + EF_J + 12.0 * u;
        tn[l] = tn_P + tJ;
        Et[l] = Et_P + EF_P * tJ + Et_J + 7.0 * u * tn[l];
        for (int i = link_nbeg[l]; i < link_nend[l]; ++i) {
            const double cn = sc * norm3(m.node_center[orig_of[i]]);
            e_max = std::max(e_max, Et[l] + EF[l] * cn + 7.0 * u * (tn[l] + cn) + u * cn);
            c_max = std::max(c_max, tn[l] + cn);
        }
    }
    const double e_cells = 1.5 * e_max;
    const double eps_cells = e_cells + 1e-7;
    ctx->e_pos = e_cells / sc;   // metres
    ctx->eps_cells = eps_cells;
    const double k_max = std::max(std::fabs(K[0]), std::max(std::fabs(K[1]), std::fabs(K[2])));
    if (!(eps_cells < 0.125) || !(c_max < 0x1p21) || !(k_max < 0x1p21)) {
        return 0; // bound too loose for this resolution: the double path handles everything
    }

    // ---- per-thread shared-memory state: transforms of branching parents, root centres of pair trees ----
    std::vector<int> slot32(nl, -1), ptree_of_tree(m.n_trees, -1);
    int n_slots32 = 0, n_ptrees = 0;
    for (int l = 0; l < nl; ++l) {
        const int p = m.link_parent[l];
        if (p >= 0 && p != l - 1 && slot32[p] < 0) {
            slot32[p] = 0;   // marked; numbered below in link order
        }
    }
    for (int l = 0; l < nl; ++l) {
        if (slot32[l] == 0) slot32[l] = n_slots32++;
    }
    // Pair tests: with few checked pairs (one arm) the root spheres almost never overlap, so the kernel keeps
    // only the root centres and sends an overlap to the double kernel; with many pairs (two arms + torso: root
    // overlaps in every sixth state) it keeps the transforms of all paired links and descends itself.
    const bool roots_only = m.n_pairs <= 24;
    if (roots_only) {
        for (int p = 0; p < m.n_pairs; ++p) {
            if (ptree_of_tree[m.pair_a[p]] < 0) ptree_of_tree[m.pair_a[p]] = n_ptrees++;
            if (ptree_of_tree[m.pair_b[p]] < 0) ptree_of_tree[m.pair_b[p]] = n_ptrees++;
        }
    } else {
        n_slots32 = 0;
        for (int l = 0; l < nl; ++l) {
            slot32[l] = m.link_slot[l];     // the double kernels' slot set: branching parents + paired links
            n_slots32 = std::max(n_slots32, slot32[l] + 1);
        }
    }
    // ranks of the double radii (the full pair descent splits the larger sphere)
    std::vector<double> radii;
    for (int i = 0; i < n32; ++i) radii.push_back(m.node_radius[orig_of[i]]);
    std::sort(radii.begin(), radii.end());
    radii.erase(std::unique(radii.begin(), radii.end()), radii.end());
    std::vector<int> ptree_of_root(nn, -1);
    for (int t = 0; t < m.n_trees; ++t) {
        if (ptree_of_tree[t] >= 0) ptree_of_root[m.tree_root[t]] = ptree_of_tree[t];
    }

    // ---- blob ----
    auto align4 = [](int w) { return (w + 3) / 4 * 4; };
    Model32Header h;
    memset(&h, 0, sizeof(h));
    int w = (int)(sizeof(Model32Header) / 4);
    h.n_links = nl; h.n_nodes = n32; h.n_pairs = m.n_pairs; h.n_allowed = m.n_allowed; h.n_slots = n_slots32; h.dof = m.dof;
    h.n_ptrees = n_ptrees;
    h.off_link_i = w; w += 4 * nl;
    h.off_link_n = w; w = align4(w + 2 * nl);
    h.off_origin = w; w += 12 * nl;
    h.off_axis = w; w += 4 * nl;
    h.off_base = w; w += 12 * nl;
    h.off_node_c = w; w += 4 * n32;
    h.off_node_i = w; w += 4 * n32;
    h.off_node_orig = w; w = align4(w + n32);
    h.off_pair = w; w = align4(w + 4 * m.n_pairs);
    h.off_allowed = w; w = align4(w + 2 * m.n_allowed);
    h.words = w;
    h.e_cells = (float)e_cells;
    h.eps_cells = (float)(eps_cells * 1.0000002);
    h.pair_k = (float)(2.5 * e_cells);
    h.q_lin_max = (float)q_lin_max;
    std::vector<float>& B = ctx->h_blob;
    B.assign(w, 0.0f);
    memcpy(B.data(), &h, sizeof(h));
    int* BI = reinterpret_cast<int*>(B.data());
    for (int l = 0; l < nl; ++l) {
        int fn = m.link_joint[l];
        double J[12];
        if (m.link_var[l] < 0 && fn != 0) {
            const_joint_transform(fn, m.link_origin[l], m.link_axis[l], m.link_const[l], J);
            fn = 0;
        } else {
            memcpy(J, m.link_origin[l], sizeof(J));
        }
        BI[h.off_link_i + 4 * l] = m.link_parent[l];
        BI[h.off_link_i + 4 * l + 1] = fn;
        BI[h.off_link_i + 4 * l + 2] = m.link_var[l];
        BI[h.off_link_i + 4 * l + 3] = slot32[l];
        BI[h.off_link_n + 2 * l] = link_nbeg[l];
        BI[h.off_link_n + 2 * l + 1] = link_nend[l];
        for (int k = 0; k < 12; ++k) {
            // row-major k = 4 i + j; the kernels keep rows 0 and 1 as (m[0][j], m[1][j]) pairs, then row 2 (Xf32)
            const int i = k / 4, j = k % 4, word = i < 2 ? 2 * j + i : 8 + j;
            const bool t = j == 3;
            B[h.off_origin + 12 * l + word] = (float)(t ? sc * J[k] : J[k]);
            B[h.off_base + 12 * l + word] = (float)(t ? base_t(l, i) : m.link_base[l][k]);
        }
        for (int k = 0; k < 3; ++k) {
            B[h.off_axis + 4 * l + k] = (float)(fn == 5 ? sc * J[4 * k + 2] : m.link_axis[l][k]);
        }
    }
    for (int i = 0; i < n32; ++i) {
        const int node = orig_of[i];
        for (int k = 0; k < 3; ++k) B[h.off_node_c + 4 * i + k] = (float)(sc * m.node_center[node][k]);
        B[h.off_node_c + 4 * i + 3] = (float)(sc * m.node_radius[node]);
        BI[h.off_node_i + 4 * i] = skip[i];
        BI[h.off_node_i + 4 * i + 1] = m.node_thresh[node];
        BI[h.off_node_i + 4 * i + 2] = roots_only ? ptree_of_root[node] : m.link_slot[m.node_link[node]];
        BI[h.off_node_i + 4 * i + 3] = (int)(std::lower_bound(radii.begin(), radii.end(), m.node_radius[node]) - radii.begin());
        BI[h.off_node_orig + i] = node;
    }
    for (int p = 0; p < m.n_pairs; ++p) {
        BI[h.off_pair + 4 * p] = ptree_of_tree[m.pair_a[p]];
        BI[h.off_pair + 4 * p + 1] = ptree_of_tree[m.pair_b[p]];
        BI[h.off_pair + 4 * p + 2] = new_of[m.tree_root[m.pair_a[p]]];
        BI[h.off_pair + 4 * p + 3] = new_of[m.tree_root[m.pair_b[p]]];
    }
    for (int k = 0; k < m.n_allowed; ++k) {
        BI[h.off_allowed + 2 * k] = new_of[m.allowed_a[k]];
        BI[h.off_allowed + 2 * k + 1] = new_of[m.allowed_b[k]];
    }

    // ---- launch geometry + upload ----
    const size_t per_thread = ((size_t)n_slots32 * 12 + (size_t)n_ptrees * 3) * sizeof(float) +
                              4 * (v32_persistent() ? V32P_EDGES_PER_THREAD : 1) * sizeof(int);
    const size_t fixed = (size_t)w * 4 + 64;
    ctx->v32_slots = n_slots32;
    ctx->v32_ptrees = n_ptrees;
    const size_t smem_max = 227 * 1024;
    int threads = V32_THREADS;
    while (threads > 32 && fixed + per_thread * threads > smem_max) threads -= 32;
    if (fixed + per_thread * threads > smem_max) {
        return 0;
    }
    ctx->v32_threads = threads;
    const int smem = (int)std::max(fixed + per_thread * threads, (size_t)1024);
    // the two hot kernels are compiled per pair mode (validity32.cuh: PairMode)
    const auto states_k = roots_only ? states_valid32_kernel<PAIRS_ROOTS> : states_valid32_kernel<PAIRS_DESCENT>;
    const auto edges_k = roots_only ? edges_valid32_kernel<PAIRS_ROOTS> : edges_valid32_kernel<PAIRS_DESCENT>;
    CU(raise_smem_cap(states_k, smem));
    CU(raise_smem_cap(edges_k, smem));
    ctx->v32_edge_batch_blocks_per_sm = 0;
    {
        const size_t smem_b = (size_t)w * 4 + ((size_t)n_slots32 * 12 + (size_t)n_ptrees * 3) * sizeof(float) * threads +
                              (2 * (size_t)V32_EDGE_EPT * threads + 4) * sizeof(int);   // == v32_smem_edge_batch once blob_words is set
        if (smem_b <= smem_max) {
            CU(raise_smem_cap(edges_valid32b_kernel, (int)smem_b));
            int per_sm = 0;
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, edges_valid32b_kernel, threads, smem_b));
            ctx->v32_edge_batch_blocks_per_sm = per_sm;
            if (getenv("SMPLGPU_V32_VERBOSE")) {
                int per_sm_old = 0;
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_old, edges_k, threads, (size_t)smem);
                fprintf(stderr, "[smplgpu] edge kernels: %d threads, shared memory %d B (block form, %d blocks/SM) / %zu B (batched, %d blocks/SM)\n",
                        threads, smem, per_sm_old, smem_b, per_sm);
            }
        }
    }
    CU(raise_smem_cap(fk_centers32_kernel, smem));
    CU(raise_smem_cap(states_valid32p_kernel, smem));
    CU(raise_smem_cap(edges_valid32p_kernel, smem));
    {
        int per_sm = 0;
        if (v32_persistent()) {
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, states_valid32p_kernel, threads, (size_t)smem));
        } else
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, states_k, threads, (size_t)smem));
        ctx->v32_blocks_per_sm = std::max(1, per_sm);
    }
    int r = grow(ctx, (void**)&ctx->d_blob, &ctx->blob_cap, (size_t)w * 4);
    if (r) return r;
    CU(cudaMemcpyAsync(ctx->d_blob, B.data(), (size_t)w * 4, cudaMemcpyHostToDevice, ctx->stream));
    ctx->blob_words = w;
    ctx->grid32.nx = ctx->grid.nx; ctx->grid32.ny = ctx->grid.ny; ctx->grid32.nz = ctx->grid.nz;
    {
        int magic;
        memcpy(&magic, &ROUND_MAGIC, sizeof(magic));
        ctx->grid32.kx = magic - (int)K[0]; ctx->grid32.ky = magic - (int)K[1]; ctx->grid32.kz = magic - (int)K[2];
        for (int i = 0; i < 3; ++i) ctx->fk32_origin[i] = (&ctx->grid.ox)[i] + (K[i] + 1.0) * ctx->res;
    }
    ctx->has_model32 = true;
    return 0;
}

// SMPLGPU_V32_EDGE_BATCH=1: the batched persistent form of the edge kernel (edges_valid32b_kernel) instead of a block per
// blockDim edges.  Measured equal within noise (0.480 vs 0.476 ms per 2^20 edges; 72 registers and 7 blocks per SM
// against 64 and 8), so the simpler kernel stays the default (DESIGN.md section 7).
static bool v32_edge_batch()
{
    static const bool on = [] {
        const char* e = getenv("SMPLGPU_V32_EDGE_BATCH");
        return e != nullptr && atoi(e) != 0;
    }();
    return on;
}

// the batched edge kernel keeps V32_EDGE_EPT edges per thread in shared memory: offsets, ok, unc, counts
static size_t v32_smem_edge_batch(const smplgpu_ctx* ctx)
{
    return (size_t)ctx->blob_words * 4
           + ((size_t)ctx->v32_slots * 12 + (size_t)ctx->v32_ptrees * 3) * sizeof(float) * ctx->v32_threads
           + (2 * (size_t)V32_EDGE_EPT * ctx->v32_threads + 4) * sizeof(int);
}

static size_t v32_smem(const smplgpu_ctx* ctx)
{
    // blob | per-thread slots and root centres | the edge kernels' per-edge block state (the lane-persistent form
    // keeps V32P_EDGES_PER_THREAD edges per thread: offsets, ok, unc, counts)
    return (size_t)ctx->blob_words * 4
           + ((size_t)ctx->v32_slots * 12 + (size_t)ctx->v32_ptrees * 3) * sizeof(float) * ctx->v32_threads
           + (4 * (size_t)(v32_persistent() ? V32P_EDGES_PER_THREAD : 1) * ctx->v32_threads + 4) * sizeof(int);
}


static int upload_model(smplgpu_ctx* ctx)
{
    DevModel& m = *ctx->h_model;
    if (ctx->has_df) {
        for (int i = 0; i < m.n_nodes; ++i) {
            m.node_thresh[i] = sphere_threshold(ctx->res, ctx->dmax_sq, m.node_radius[i], ctx->padding);
        }
    }
    CU(cudaMemcpyAsync(ctx->d_model, &m, sizeof(DevModel), cudaMemcpyHostToDevice, ctx->stream));
    int r = build_model32(ctx);
    if (r) return r;
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int tree_depth(const DevModel& m, int node)
{
    if (m.node_left[node] < 0) {
        return 1;
    }
    return 1 + std::max(tree_depth(m, m.node_left[node]), tree_depth(m, m.node_right[node]));
}

int smplgpu_set_robot(smplgpu_ctx* ctx, const smplgpu_robot_desc* d)
{
    if (!ctx || !d) return SMPLGPU_ERR_INVALID;
    if (d->dof <= 0 || d->dof > MAX_DOF) return fail(ctx, SMPLGPU_ERR_LIMIT, "dof %d outside [1,%d]", d->dof, MAX_DOF);
    if (d->n_links < 0 || d->n_links > MAX_LINKS) return fail(ctx, SMPLGPU_ERR_LIMIT, "n_links %d > %d", d->n_links, MAX_LINKS);
    if (d->n_nodes < 0 || d->n_nodes > MAX_NODES) return fail(ctx, SMPLGPU_ERR_LIMIT, "n_nodes %d > %d", d->n_nodes, MAX_NODES);
    if (d->n_trees < 0 || d->n_trees > MAX_TREES) return fail(ctx, SMPLGPU_ERR_LIMIT, "n_trees %d > %d", d->n_trees, MAX_TREES);
    if (d->n_pairs < 0 || d->n_pairs > MAX_PAIRS) return fail(ctx, SMPLGPU_ERR_LIMIT, "n_pairs %d > %d", d->n_pairs, MAX_PAIRS);
    if (d->n_allowed_leaf_pairs < 0 || d->n_allowed_leaf_pairs > MAX_ALLOWED) return fail(ctx, SMPLGPU_ERR_LIMIT, "allowed leaf pairs %d > %d", d->n_allowed_leaf_pairs, MAX_ALLOWED);
    if (d->n_segments < 0 || d->n_segments > MAX_SEGMENTS) return fail(ctx, SMPLGPU_ERR_LIMIT, "n_segments %d > %d", d->n_segments, MAX_SEGMENTS);

    DevModel& m = *ctx->h_model;
    memset(&m, 0, sizeof(m));
    m.dof = d->dof;
    m.n_links = d->n_links;
    m.n_nodes = d->n_nodes;
    m.n_trees = d->n_trees;
    m.n_pairs = d->n_pairs;
    m.n_robot_trees = (d->n_robot_trees > 0 && d->n_robot_trees <= d->n_trees) ? d->n_robot_trees : d->n_trees;
    m.n_robot_pairs = 0;
    for (int k = 0; k < d->n_pairs; ++k) {
        if (d->pair_a[k] < m.n_robot_trees && d->pair_b[k] < m.n_robot_trees) ++m.n_robot_pairs;
    }
    m.n_allowed = d->n_allowed_leaf_pairs;
    m.n_segments = d->n_segments;

    for (int l = 0; l < m.n_links; ++l) {
        const int p = d->link_parent[l];
        if (p >= l) return fail(ctx, SMPLGPU_ERR_INVALID, "link %d: parent %d is not earlier in the table", l, p);
        const int fn = d->link_joint[l];
        if (fn < 0 || fn > SMPLGPU_JOINT_PRISMATIC) return fail(ctx, SMPLGPU_ERR_INVALID, "link %d: joint fn %d", l, fn);
        const int v = d->link_var[l];
        if (v >= m.dof) return fail(ctx, SMPLGPU_ERR_INVALID, "link %d: variable %d >= dof", l, v);
        m.link_parent[l] = p < 0 ? -1 : p;
        m.link_joint[l] = fn;
        m.link_var[l] = v < 0 ? -1 : v;
        m.link_const[l] = d->link_const[l];
        memcpy(m.link_origin[l], d->link_origin + 12 * l, 12 * sizeof(double));
        memcpy(m.link_axis[l], d->link_axis + 3 * l, 3 * sizeof(double));
        memcpy(m.link_base[l], d->link_base + 12 * l, 12 * sizeof(double));
        m.link_slot[l] = -1;
    }
    for (int i = 0; i < m.n_nodes; ++i) {
        const int l = d->node_link[i];
        if (l < 0 || l >= m.n_links) return fail(ctx, SMPLGPU_ERR_INVALID, "node %d: link %d", i, l);
        const int a = d->node_left[i], b = d->node_right[i];
        if ((a < 0) != (b < 0) || a >= m.n_nodes || b >= m.n_nodes) return fail(ctx, SMPLGPU_ERR_INVALID, "node %d: children %d %d", i, a, b);
        if (a >= 0 && (d->node_link[a] != l || d->node_link[b] != l)) return fail(ctx, SMPLGPU_ERR_INVALID, "node %d: child on another link", i);
        m.node_link[i] = l;
        m.node_left[i] = a < 0 ? -1 : a;
        m.node_right[i] = b < 0 ? -1 : b;
        m.node_radius[i] = d->node_radius[i];
        memcpy(m.node_center[i], d->node_center + 3 * i, 3 * sizeof(double));
        m.node_thresh[i] = 0x7FFFFFFF; // until a distance field is set
    }
    int max_depth = 0;
    for (int t = 0; t < m.n_trees; ++t) {
        const int r = d->tree_root[t];
        if (r < 0 || r >= m.n_nodes) return fail(ctx, SMPLGPU_ERR_INVALID, "tree %d: root %d", t, r);
        m.tree_root[t] = r;
        max_depth = std::max(max_depth, tree_depth(m, r));
    }
    if (2 * max_depth + 2 > MAX_TREE_DEPTH) return fail(ctx, SMPLGPU_ERR_LIMIT, "sphere tree depth %d too deep", max_depth);
    for (int p = 0; p < m.n_pairs; ++p) {
        if (d->pair_a[p] < 0 || d->pair_a[p] >= m.n_trees || d->pair_b[p] < 0 || d->pair_b[p] >= m.n_trees)
            return fail(ctx, SMPLGPU_ERR_INVALID, "pair %d out of range", p);
        m.pair_a[p] = d->pair_a[p];
        m.pair_b[p] = d->pair_b[p];
    }
    for (int k = 0; k < m.n_allowed; ++k) {
        m.allowed_a[k] = d->allowed_leaf_a[k];
        m.allowed_b[k] = d->allowed_leaf_b[k];
    }
    for (int v = 0; v < m.dof; ++v) {
        m.var_type[v] = d->var_type[v];
        m.var_weight[v] = d->var_motion_weight[v];
        m.var_min[v] = d->var_min ? d->var_min[v] : -INFINITY;
        m.var_max[v] = d->var_max ? d->var_max[v] : INFINITY;
        // angles::normalize_angle(min)  (smpl/angles.h:45-62)
        double a = m.var_min[v];
        if (std::fabs(a) > 2.0 * M_PI) a = std::fmod(a, 2.0 * M_PI);
        if (a < -M_PI) a += 2.0 * M_PI;
        if (a > M_PI) a -= 2.0 * M_PI;
        m.var_min_norm[v] = a;
    }
    for (int s = 0; s < m.n_segments; ++s) {
        m.seg_kind[s] = d->seg_kind[s];
        m.seg_var[s] = d->seg_var[s] < 0 ? -1 : d->seg_var[s];
        if (m.seg_var[s] >= m.dof) return fail(ctx, SMPLGPU_ERR_INVALID, "segment %d: variable out of range", s);
        memcpy(m.seg_axis[s], d->seg_axis + 3 * s, 3 * sizeof(double));
        memcpy(m.seg_origin[s], d->seg_origin + 3 * s, 3 * sizeof(double));
        memcpy(m.seg_f_tip[s], d->seg_f_tip + 12 * s, 12 * sizeof(double));
    }
    if (d->T_kin_to_planning) {
        memcpy(m.T_kin_to_planning, d->T_kin_to_planning, 12 * sizeof(double));
    } else {
        const double I[12] = { 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0 };
        memcpy(m.T_kin_to_planning, I, sizeof(I));
    }
    memcpy(m.xyz_offset, d->xyz_offset, 3 * sizeof(double));

    // trees grouped by the link they ride on (checked inline while T_link is in registers)
    {
        std::vector<int> order(m.n_trees);
        for (int t = 0; t < m.n_trees; ++t) order[t] = t;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
            return m.node_link[m.tree_root[a]] < m.node_link[m.tree_root[b]];
        });
        int k = 0;
        for (int l = 0; l < m.n_links; ++l) {
            m.link_tree_begin[l] = k;
            while (k < m.n_trees && m.node_link[m.tree_root[order[k]]] == l) {
                m.tree_by_link[k] = order[k];
                ++k;
            }
            m.link_tree_end[l] = k;
        }
    }
    // shared-memory slots: links read again later (tree pairs, or a child that
    // is not the next link in the table)
    {
        std::vector<bool> keep(m.n_links, false);
        for (int p = 0; p < m.n_pairs; ++p) {
            keep[m.node_link[m.tree_root[m.pair_a[p]]]] = true;
            keep[m.node_link[m.tree_root[m.pair_b[p]]]] = true;
        }
        for (int l = 0; l < m.n_links; ++l) {
            const int p = m.link_parent[l];
            if (p >= 0 && p != l - 1) {
                keep[p] = true;
            }
        }
        int slots = 0;
        for (int l = 0; l < m.n_links; ++l) {
            if (keep[l]) {
                m.link_slot[l] = slots++;
            }
        }
        m.n_slots = slots;
        // threads per block: as many warps (<= 4) as the per-thread slot storage lets one block hold
        const size_t per_thread = (size_t)slots * 12 * sizeof(double) + 3 * sizeof(int) + 1;
        const size_t smem_max = 227 * 1024;
        int threads = VALIDITY_THREADS;
        while (threads > 32 && per_thread * threads > smem_max) {
            threads -= 32;
        }
        if (per_thread * threads > smem_max) return fail(ctx, SMPLGPU_ERR_LIMIT, "%d link slots need %zu B of shared memory per warp", slots, per_thread * 32);
        ctx->validity_threads = threads;
        const size_t smem = per_thread * threads + 16;
        CU(raise_smem_cap(states_valid_kernel, (int)std::max(smem, (size_t)1024)));
        CU(raise_smem_cap(edges_valid_kernel, (int)std::max(smem, (size_t)1024)));
        CU(raise_smem_cap(fk_centers_kernel, (int)std::max(smem, (size_t)1024)));
        const size_t smem_x1 = (size_t)slots * 12 * sizeof(double) * EXPAND1_THREADS;
        if (smem_x1 <= smem_max - 1024) {
            CU(raise_smem_cap(expand_state_kernel, (int)std::max(smem_x1, (size_t)1024)));
        }
    }
    ctx->has_robot = true;
    ++ctx->scene_epoch;
    // what was derived from the previous robot: lattice discretisation, primitive table, device lattices
    ctx->has_lattice = false;
    if (ctx->x1_dof != m.dof) ctx->x1_prims = -1;
    if (ctx->has_lat && ctx->lat_dof != m.dof) {
        for (int b = 0; b < SMPLGPU_EXPAND_BUFFERS; ++b) ctx->lat_n[b] = -1;
        free_lattice(ctx);
    }
    return upload_model(ctx);
}

///////////////////////////////////////////////////////////////////////////////
// distance field
///////////////////////////////////////////////////////////////////////////////

// the single-precision kernels index the field with 32-bit ints
static bool field_cells_ok(int nx, int ny, int nz)
{
    return (unsigned long long)nx * ny * nz < (1ull << 31);
}

static int set_df_common(smplgpu_ctx* ctx, int nx, int ny, int nz, const double origin[3], double res, int dmax_sq, double padding)
{
    if (nx <= 0 || ny <= 0 || nz <= 0 || !(res > 0.0) || dmax_sq < 0 || dmax_sq > 65534)
        return fail(ctx, SMPLGPU_ERR_INVALID, "bad distance field parameters");
    if (!field_cells_ok(nx, ny, nz)) return fail(ctx, SMPLGPU_ERR_INVALID, "distance field of 2^31 cells or more");
    // a bank run queued behind the caller's back still reads the field; a bank (and the walls derived from the
    // field) of another shape would be indexed with the wrong strides
    {
        const int fr = finish_bank_run(ctx);
        if (fr) return fr;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->has_df && (ctx->grid.nx != nx || ctx->grid.ny != ny || ctx->grid.nz != nz)) {
        ctx->has_bank = false;   // re-create with smplgpu_bfs_bank_create
    }
    ++ctx->scene_epoch;
    const size_t cells = (size_t)nx * ny * nz;
    if (cells != ctx->df_cells) {
        if (ctx->d_df) { CU(cudaFree(ctx->d_df)); ctx->d_df = nullptr; }
        CU(cudaMalloc(&ctx->d_df, cells * sizeof(uint16_t)));
        ctx->df_cells = cells;
    }
    ctx->grid.nx = nx; ctx->grid.ny = ny; ctx->grid.nz = nz;
    ctx->grid.inv_res = 1.0 / res;                 // m_inv_res(1.0 / resolution), distance_map.hpp:124
    ctx->grid.ox = origin[0] - res;                // (m_origin_x - m_res), :524
    ctx->grid.oy = origin[1] - res;
    ctx->grid.oz = origin[2] - res;
    ctx->res = res;
    ctx->padding = padding;
    ctx->dmax_sq = dmax_sq;
    ctx->lat.res = res;   // mprimActive's metric goal distance = BFS cells * resolution
    memcpy(ctx->origin, origin, 3 * sizeof(double));
    return 0;
}

int smplgpu_set_distance_field(smplgpu_ctx* ctx, const uint16_t* d2, int nx, int ny, int nz,
                               const double origin[3], double res, int dmax_sq, double padding)
{
    if (!ctx || !d2 || !origin) return SMPLGPU_ERR_INVALID;
    int r = set_df_common(ctx, nx, ny, nz, origin, res, dmax_sq, padding);
    if (r) return r;
    CU(cudaMemcpyAsync(ctx->d_df, d2, ctx->df_cells * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->has_df = true;
    return ctx->has_robot ? upload_model(ctx) : 0;
}

int smplgpu_set_distance_field_dev(smplgpu_ctx* ctx, const uint16_t* d2_dev, int nx, int ny, int nz,
                                   const double origin[3], double res, int dmax_sq, double padding)
{
    if (!ctx || !d2_dev || !origin) return SMPLGPU_ERR_INVALID;
    int r = set_df_common(ctx, nx, ny, nz, origin, res, dmax_sq, padding);
    if (r) return r;
    if (d2_dev != ctx->d_df) {
        CU(cudaMemcpyAsync(ctx->d_df, d2_dev, ctx->df_cells * sizeof(uint16_t), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->has_df = true;
    return ctx->has_robot ? upload_model(ctx) : 0;
}

// Voxelises a triangle mesh on the device (voxelize.cuh).  mode 0: bits = bitmap over the mesh's own voxel grid
// (gmin, gext); mode 1: occ = occupancy bytes of the distance-field grid (addPointsToField).  The per-triangle
// work sizes come back to the host once (they size the launch); vertices and triangles are host pointers.
static int voxelize_on_device(smplgpu_ctx* ctx, const double* vertices, int n_vertices, const int32_t* triangles,
                              int n_triangles, const VoxDisc& D, int mode, int3 gmin, int3 gext, unsigned int* bits,
                              uint8_t* occ)
{
    for (int i = 0; i < 3 * n_triangles; ++i) {
        if (triangles[i] < 0 || triangles[i] >= n_vertices)
            return fail(ctx, SMPLGPU_ERR_INVALID, "triangle %d: vertex index out of range", i / 3);
    }
    const size_t vb = (((size_t)n_vertices * 3 * sizeof(double)) + 255) / 256 * 256;
    const size_t tb = (((size_t)n_triangles * 3 * sizeof(int)) + 255) / 256 * 256;
    const size_t sb = (((size_t)n_triangles * sizeof(TriSetup)) + 255) / 256 * 256;
    const size_t ob = (((size_t)(n_triangles + 1) * sizeof(unsigned long long)) + 255) / 256 * 256;
    int r = grow(ctx, &ctx->d_vox, &ctx->vox_cap, vb + tb + sb + ob);
    if (r) return r;
    uint8_t* base = (uint8_t*)ctx->d_vox;
    double* d_vertices = (double*)base;
    int* d_tris = (int*)(base + vb);
    TriSetup* d_setup = (TriSetup*)(base + vb + tb);
    unsigned long long* d_off = (unsigned long long*)(base + vb + tb + sb);
    CU(cudaMemcpyAsync(d_vertices, vertices, (size_t)n_vertices * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_tris, triangles, (size_t)n_triangles * 3 * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    vox_setup_kernel<<<(n_triangles + 127) / 128, 128, 0, ctx->stream>>>(d_vertices, d_tris, n_triangles, D, d_setup, d_off);
    ++ctx->launches;
    CU(cudaGetLastError());
    std::vector<unsigned long long> off((size_t)n_triangles + 1);
    CU(cudaMemcpyAsync(off.data(), d_off, (size_t)n_triangles * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    unsigned long long total = 0;
    for (int i = 0; i < n_triangles; ++i) {
        const unsigned long long c = off[i];
        off[i] = total;
        total += c;
    }
    off[n_triangles] = total;
    if (total == 0) {
        return 0;
    }
    if (total > (1ull << 40)) return fail(ctx, SMPLGPU_ERR_LIMIT, "mesh covers %llu candidate voxels", total);
    CU(cudaMemcpyAsync(d_off, off.data(), off.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
    const unsigned long long want = (total + 255) / 256;
    const unsigned blocks = (unsigned)std::min<unsigned long long>(want, (unsigned long long)ctx->sm_count * 64);
    vox_cells_kernel<<<blocks, 256, 0, ctx->stream>>>(d_setup, d_off, n_triangles, total, D, mode, gmin, gext, bits, ctx->grid, occ);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));   // `off` is read by the copy above
    return 0;
}

int smplgpu_voxelize_mesh(smplgpu_ctx* ctx, const double* vertices, int n_vertices, const int32_t* triangles,
                          int n_triangles, double res, const double* voxel_origin, double* voxels, int max_voxels)
{
    if (!ctx || n_vertices < 0 || n_triangles < 0 || max_voxels < 0 || !(res > 0.0)) return SMPLGPU_ERR_INVALID;
    if (n_vertices == 0 || n_triangles == 0) return 0;
    if (!vertices || !triangles || (max_voxels > 0 && !voxels)) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    VoxDisc D;
    D.half_res = voxel_origin ? 0 : 1;
    D.res = res;
    for (int a = 0; a < 3; ++a) D.pivot[a] = voxel_origin ? voxel_origin[a] : 0.0;
    // the mesh's voxel grid (ComputeAxisAlignedBoundingBox, voxelize.cpp:224-259; VoxelGrid extent, voxel_grid.h:133-141)
    double mn[3], mx[3];
    for (int a = 0; a < 3; ++a) mn[a] = mx[a] = vertices[a];
    for (int i = 0; i < n_vertices; ++i) {
        for (int a = 0; a < 3; ++a) {
            mn[a] = std::min(mn[a], vertices[3 * (size_t)i + a]);
            mx[a] = std::max(mx[a], vertices[3 * (size_t)i + a]);
        }
    }
    int g0[3], g1[3];
    for (int a = 0; a < 3; ++a) {
        const double lo = mn[a], hi = mn[a] + (mx[a] - mn[a]);
        if (D.half_res) {
            g0[a] = (lo >= 0) ? (int)(lo / res) : ((int)(lo / res) - 1);
            g1[a] = (hi >= 0) ? (int)(hi / res) : ((int)(hi / res) - 1);
        } else {
            g0[a] = (int)std::floor((lo - D.pivot[a]) / res + 0.5);
            g1[a] = (int)std::floor((hi - D.pivot[a]) / res + 0.5);
        }
    }
    const int3 gmin = make_int3(g0[0], g0[1], g0[2]);
    const int3 gext = make_int3(g1[0] - g0[0] + 1, g1[1] - g0[1] + 1, g1[2] - g0[2] + 1);
    const unsigned long long n_cells = (unsigned long long)gext.x * gext.y * gext.z;
    if (gext.x <= 0 || gext.y <= 0 || gext.z <= 0 || n_cells > (1ull << 36))
        return fail(ctx, SMPLGPU_ERR_LIMIT, "voxel grid of %d x %d x %d cells", gext.x, gext.y, gext.z);
    const size_t n_words = (size_t)((n_cells + 31) / 32);
    const int n_blocks = (int)((n_words + VOX_SCAN_THREADS - 1) / VOX_SCAN_THREADS);
    const size_t wb = ((n_words * sizeof(unsigned int)) + 255) / 256 * 256;
    const size_t bb = (((size_t)n_blocks + 1) * sizeof(unsigned int) + 255) / 256 * 256;
    const size_t outb = (size_t)max_voxels * 3 * sizeof(double);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, 2 * wb + bb + outb + 256);
    if (r) return r;
    uint8_t* base = (uint8_t*)ctx->d_misc;
    unsigned int* d_bits = (unsigned int*)base;
    unsigned int* d_prefix = (unsigned int*)(base + wb);
    unsigned int* d_blocks = (unsigned int*)(base + 2 * wb);       // n_blocks entries + the grand total
    double* d_out = (double*)(base + 2 * wb + bb);
    CU(cudaMemsetAsync(d_bits, 0, wb, ctx->stream));
    r = voxelize_on_device(ctx, vertices, n_vertices, triangles, n_triangles, D, 0, gmin, gext, d_bits, nullptr);
    if (r) return r;
    vox_count_kernel<<<n_blocks, VOX_SCAN_THREADS, 0, ctx->stream>>>(d_bits, n_words, d_prefix, d_blocks);
    vox_scan_blocks_kernel<<<1, VOX_SCAN_THREADS, 0, ctx->stream>>>(d_blocks, n_blocks, d_blocks + n_blocks);
    vox_extract_kernel<<<n_blocks, VOX_SCAN_THREADS, 0, ctx->stream>>>(d_bits, n_words, d_prefix, d_blocks, D, gmin, gext, d_out,
                                                                       (unsigned int)max_voxels);
    ctx->launches += 3;
    CU(cudaGetLastError());
    unsigned int total = 0;
    CU(cudaMemcpyAsync(&total, d_blocks + n_blocks, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    const size_t m = std::min((size_t)total, (size_t)max_voxels);
    if (m > 0) {
        CU(cudaMemcpyAsync(voxels, d_out, m * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    return (int)total;
}

static int build_distance_field_impl(smplgpu_ctx* ctx, const double* vertices, int n_vertices, const int32_t* triangles,
                                     int n_triangles, const int32_t* cells_xyz, int n_cells, int nx, int ny, int nz,
                                     const double origin[3], double res, double max_dist, double padding);

int smplgpu_build_distance_field(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n_cells,
                                 int nx, int ny, int nz, const double origin[3], double res,
                                 double max_dist, double padding)
{
    return build_distance_field_impl(ctx, nullptr, 0, nullptr, 0, cells_xyz, n_cells, nx, ny, nz, origin, res, max_dist, padding);
}

int smplgpu_build_distance_field_from_meshes(smplgpu_ctx* ctx, const double* vertices, int n_vertices,
                                             const int32_t* triangles, int n_triangles, const int32_t* cells_xyz,
                                             int n_cells, int nx, int ny, int nz, const double origin[3], double res,
                                             double max_dist, double padding)
{
    if (n_vertices < 0 || n_triangles < 0 || (n_triangles > 0 && (!vertices || !triangles || n_vertices == 0)))
        return SMPLGPU_ERR_INVALID;
    return build_distance_field_impl(ctx, vertices, n_vertices, triangles, n_triangles, cells_xyz, n_cells, nx, ny, nz, origin,
                                     res, max_dist, padding);
}

static int build_distance_field_impl(smplgpu_ctx* ctx, const double* vertices, int n_vertices, const int32_t* triangles,
                                     int n_triangles, const int32_t* cells_xyz, int n_cells, int nx, int ny, int nz,
                                     const double origin[3], double res, double max_dist, double padding)
{
    if (!ctx || !origin || n_cells < 0 || (n_cells > 0 && !cells_xyz)) return SMPLGPU_ERR_INVALID;
    // m_dmax_int((int)std::ceil(m_max_dist * m_inv_res)), distance_map.hpp:125-126
    const double inv_res = 1.0 / res;
    const int dmax = (int)std::ceil(max_dist * inv_res);
    const int dmax_sq = dmax * dmax;
    int r = set_df_common(ctx, nx, ny, nz, origin, res, dmax_sq, padding);
    if (r) return r;
    const size_t cells = ctx->df_cells;
    // scratch: occupancy bytes + two u16 planes + the cell list
    const size_t need = cells + 2 * cells * sizeof(uint16_t) + (size_t)n_cells * 3 * sizeof(int) + 64;
    r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, need);
    if (r) return r;
    uint8_t* occ = (uint8_t*)ctx->d_misc;
    uint16_t* g1 = (uint16_t*)(occ + ((cells + 15) / 16) * 16);
    uint16_t* g2 = g1 + cells;
    int* d_cells = (int*)(g2 + cells + (cells & 1));
    CU(cudaMemsetAsync(occ, 0, cells, ctx->stream));
    if (n_cells > 0) {
        CU(cudaMemcpyAsync(d_cells, cells_xyz, (size_t)n_cells * 3 * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        edt_scatter_kernel<<<(n_cells + 255) / 256, 256, 0, ctx->stream>>>(d_cells, n_cells, nx, ny, nz, occ);
        ++ctx->launches;
    }
    if (n_triangles > 0) {
        // WorldCollisionModel::insertObject: voxelise with the grid origin as voxel origin, then addPointsToField
        VoxDisc D;
        D.half_res = 0;
        D.res = res;
        for (int a = 0; a < 3; ++a) D.pivot[a] = origin[a];
        r = voxelize_on_device(ctx, vertices, n_vertices, triangles, n_triangles, D, 1, make_int3(0, 0, 0), make_int3(0, 0, 0),
                               nullptr, occ);
        if (r) return r;
    }
    edt_pass_z_kernel<<<(nx * ny + 127) / 128, 128, 0, ctx->stream>>>(occ, nx, ny, nz, dmax, g1);
    const unsigned blocks = (unsigned)((cells + 255) / 256);
    edt_pass_axis_kernel<<<blocks, 256, 0, ctx->stream>>>(g1, nx, ny, nz, 1, dmax, dmax_sq, true, g2);
    edt_pass_axis_kernel<<<blocks, 256, 0, ctx->stream>>>(g2, nx, ny, nz, 0, dmax, dmax_sq, false, ctx->d_df);
    ctx->launches += 3;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->has_df = true;
    return ctx->has_robot ? upload_model(ctx) : 0;
}

// OccupancyGrid::addPointsToField / removePointsFromField on the resident field: the obstacle set is read back from the
// field itself (distance 0), changed, and the exact transform recomputed
static int update_distance_field_cells(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n, uint8_t value)
{
    if (!ctx || n < 0 || (n > 0 && !cells_xyz)) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "no distance field");
    if (n == 0) return 0;
    {
        const int fr = finish_bank_run(ctx);   // a bank run queued behind the caller's back still reads the field
        if (fr) return fr;
    }
    const int nx = ctx->grid.nx, ny = ctx->grid.ny, nz = ctx->grid.nz;
    const int dmax_sq = ctx->dmax_sq;
    int dmax = (int)std::sqrt((double)dmax_sq);
    while (dmax * dmax < dmax_sq) ++dmax;
    while (dmax > 0 && (dmax - 1) * (dmax - 1) >= dmax_sq) --dmax;
    const size_t cells = ctx->df_cells;
    const size_t need = cells + 2 * cells * sizeof(uint16_t) + (size_t)n * 3 * sizeof(int) + 64;
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, need);
    if (r) return r;
    uint8_t* occ = (uint8_t*)ctx->d_misc;
    uint16_t* g1 = (uint16_t*)(occ + ((cells + 15) / 16) * 16);
    uint16_t* g2 = g1 + cells;
    int* d_cells = (int*)(g2 + cells + (cells & 1));
    const unsigned blocks = (unsigned)((cells + 255) / 256);
    edt_occ_from_field_kernel<<<blocks, 256, 0, ctx->stream>>>(ctx->d_df, cells, occ);
    CU(cudaMemcpyAsync(d_cells, cells_xyz, (size_t)n * 3 * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    edt_scatter_value_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d_cells, n, nx, ny, nz, value, occ);
    edt_pass_z_kernel<<<(nx * ny + 127) / 128, 128, 0, ctx->stream>>>(occ, nx, ny, nz, dmax, g1);
    edt_pass_axis_kernel<<<blocks, 256, 0, ctx->stream>>>(g1, nx, ny, nz, 1, dmax, dmax_sq, true, g2);
    edt_pass_axis_kernel<<<blocks, 256, 0, ctx->stream>>>(g2, nx, ny, nz, 0, dmax, dmax_sq, false, ctx->d_df);
    ctx->launches += 5;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    ++ctx->scene_epoch;   // records of the old scene are stale (smplhost::ExpansionCache)
    return 0;
}

int smplgpu_distance_field_add_cells(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n)
{
    return update_distance_field_cells(ctx, cells_xyz, n, 1);
}

int smplgpu_distance_field_remove_cells(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n)
{
    return update_distance_field_cells(ctx, cells_xyz, n, 0);
}

int smplgpu_download_distance_field(smplgpu_ctx* ctx, uint16_t* out)
{
    if (!ctx || !out) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "no distance field");
    CU(cudaMemcpyAsync(out, ctx->d_df, ctx->df_cells * sizeof(uint16_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_distance_field_dev_ptr(smplgpu_ctx* ctx, void** ptr, int64_t* bytes)
{
    if (!ctx || !ptr || !bytes) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "no distance field");
    *ptr = ctx->d_df;
    *bytes = (int64_t)(ctx->df_cells * sizeof(uint16_t));
    return 0;
}

int smplgpu_reserve_distance_field(smplgpu_ctx* ctx, int nx, int ny, int nz, void** ptr, int64_t* bytes)
{
    if (!ctx || !ptr || !bytes) return SMPLGPU_ERR_INVALID;
    if (nx <= 0 || ny <= 0 || nz <= 0) return fail(ctx, SMPLGPU_ERR_INVALID, "bad distance field dimensions");
    if (!field_cells_ok(nx, ny, nz)) return fail(ctx, SMPLGPU_ERR_INVALID, "distance field of 2^31 cells or more");
    {
        const int fr = finish_bank_run(ctx);
        if (fr) return fr;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    const size_t cells = (size_t)nx * ny * nz;
    if (cells != ctx->df_cells) {
        ctx->has_df = false;
        ctx->has_bank = false;
        if (ctx->d_df) { CU(cudaFree(ctx->d_df)); ctx->d_df = nullptr; ctx->df_cells = 0; }
        CU(cudaMalloc(&ctx->d_df, cells * sizeof(uint16_t)));
        ctx->df_cells = cells;
    }
    ++ctx->scene_epoch;
    *ptr = ctx->d_df;
    *bytes = (int64_t)(cells * sizeof(uint16_t));
    return 0;
}

int smplgpu_set_distance_field_l2_persistence(smplgpu_ctx* ctx, int on, double* set_aside_mb)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "no distance field");
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, ctx->device));
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    double mb = 0.0;
    if (on) {
        const size_t bytes = ctx->df_cells * sizeof(uint16_t);
        const size_t set_aside = std::min<size_t>((size_t)prop.persistingL2CacheMaxSize, bytes);
        if (set_aside == 0) return fail(ctx, SMPLGPU_ERR_LIMIT, "device has no persisting L2");
        CU(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside));
        const size_t window = std::min<size_t>(bytes, (size_t)prop.accessPolicyMaxWindowSize);
        attr.accessPolicyWindow.base_ptr = ctx->d_df;
        attr.accessPolicyWindow.num_bytes = window;
        attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)set_aside / (double)window);
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        mb = (double)set_aside / 1e6;
    } else {
        attr.accessPolicyWindow.num_bytes = 0;   // disables the window
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    }
    CU(cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr));
    if (!on) {
        CU(cudaCtxResetPersistingL2Cache());
    }
    if (set_aside_mb) *set_aside_mb = mb;
    return 0;
}

///////////////////////////////////////////////////////////////////////////////
// validity
///////////////////////////////////////////////////////////////////////////////

static int need_scene(smplgpu_ctx* ctx)
{
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set (smplgpu_set_robot)");
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "distance field not set");
    return 0;
}

static size_t validity_smem(const smplgpu_ctx* ctx)
{
    // slot storage + the edge kernel's offsets / verdict scratch
    return (size_t)ctx->h_model->n_slots * 12 * sizeof(double) * ctx->validity_threads
           + (3 * (size_t)ctx->validity_threads + 2) * sizeof(int);
}

static int ensure_unc(smplgpu_ctx* ctx, size_t n)
{
    if (n <= ctx->unc_cap) {
        return 0;
    }
    if (ctx->d_unc_list) { CU(cudaFree(ctx->d_unc_list)); ctx->d_unc_list = nullptr; ctx->unc_cap = 0; }
    if (ctx->d_unc_mask) { CU(cudaFree(ctx->d_unc_mask)); ctx->d_unc_mask = nullptr; }
    const size_t cap = std::max(n, (size_t)1 << 16);
    CU(cudaMalloc(&ctx->d_unc_list, cap * sizeof(int)));
    CU(cudaMalloc(&ctx->d_unc_mask, cap * sizeof(int)));
    ctx->unc_cap = cap;
    return 0;
}

static bool use_f32(const smplgpu_ctx* ctx)
{
    return ctx->precision_mode == SMPLGPU_PRECISION_CERTIFIED_F32 && ctx->has_model32;
}

// CollisionSpace::isStateValid for n resident states: the certified single-precision pass, then the
// double-precision kernel on the states it could not decide (or the double kernel alone in EXACT mode)
static int launch_states(smplgpu_ctx* ctx, const double* dq, int n, uint8_t* dv)
{
    const int vt = ctx->validity_threads;
    if (!use_f32(ctx)) {
        states_valid_kernel<<<(n + vt - 1) / vt, vt, validity_smem(ctx), ctx->stream>>>(
            ctx->d_model, ctx->d_df, ctx->grid, dq, n, dv, ctx->d_stats, nullptr, nullptr);
        ++ctx->launches;
        CU(cudaGetLastError());
        return 0;
    }
    int r = ensure_unc(ctx, (size_t)n);
    if (r) return r;
    CU(cudaMemsetAsync(ctx->d_unc_count, 0, 2 * sizeof(int), ctx->stream));   // [0] undecided items, [1] the work cursor
    const int t32 = ctx->v32_threads;
    // one wave of resident blocks; their warps pull the states from the cursor
    const int wave = std::max(1, ctx->v32_blocks_per_sm) * ctx->sm_count;
    if (v32_persistent()) {
        states_valid32p_kernel<<<std::min((n + t32 - 1) / t32, wave), t32, v32_smem(ctx), ctx->stream>>>(
            ctx->d_blob, ctx->blob_words, ctx->d_model, ctx->d_df, ctx->grid32, dq, n, dv, ctx->d_unc_list,
            ctx->d_unc_count, ctx->d_stats);
    } else
    (ctx->v32_ptrees > 0 ? states_valid32_kernel<PAIRS_ROOTS> : states_valid32_kernel<PAIRS_DESCENT>)
        <<<std::min((n + t32 - 1) / t32, wave), t32, v32_smem(ctx), ctx->stream>>>(
        ctx->d_blob, ctx->blob_words, ctx->d_model, ctx->d_df, ctx->grid32, dq, n, dv, ctx->d_unc_list,
        ctx->d_unc_count, ctx->d_stats);
    if (warp_resolve()) {
        // the undecided states, a warp each (validity_warp.cuh): the list is a fraction of a percent of the batch
        const int blocks = std::max(1, std::min((n / 64 + RESOLVE_WARPS - 1) / RESOLVE_WARPS + 1, 8 * ctx->sm_count));
        states_resolve_kernel<<<blocks, 32 * RESOLVE_WARPS, 0, ctx->stream>>>(
            ctx->d_model, ctx->d_df, ctx->grid, dq, n, dv, ctx->d_unc_list, ctx->d_unc_count);
    } else {
        const int blocks = std::max(1, std::min((n + vt - 1) / vt, 2 * ctx->sm_count));
        states_valid_kernel<<<blocks, vt, validity_smem(ctx), ctx->stream>>>(
            ctx->d_model, ctx->d_df, ctx->grid, dq, n, dv, nullptr, ctx->d_unc_list, ctx->d_unc_count);
    }
    ctx->launches += 2;
    CU(cudaGetLastError());
    return 0;
}

static int launch_edges(smplgpu_ctx* ctx, const double* dq0, const double* dq1, int n, uint8_t* dv, int* dc)
{
    const int vt = ctx->validity_threads;
    if (!use_f32(ctx)) {
        edges_valid_kernel<<<(n + vt - 1) / vt, vt, validity_smem(ctx), ctx->stream>>>(
            ctx->d_model, ctx->d_df, ctx->grid, dq0, dq1, n, dv, dc, ctx->d_stats, nullptr, nullptr);
        ++ctx->launches;
        CU(cudaGetLastError());
        return 0;
    }
    int r = ensure_unc(ctx, (size_t)n);
    if (r) return r;
    CU(cudaMemsetAsync(ctx->d_unc_count, 0, 2 * sizeof(int), ctx->stream));   // [0] undecided items, [1] the batch cursor
    const int t32 = ctx->v32_threads;
    bool masked = false;   // the kernel recorded which waypoints of an undecided edge are undecided
    if (!v32_persistent() && v32_edge_batch() && ctx->v32_edge_batch_blocks_per_sm > 0) {
        const int epb = V32_EDGE_EPT * t32;
        const int wave = ctx->v32_edge_batch_blocks_per_sm * ctx->sm_count;
        edges_valid32b_kernel<<<std::min((n + epb - 1) / epb, wave), t32, v32_smem_edge_batch(ctx), ctx->stream>>>(
            ctx->d_blob, ctx->blob_words, ctx->d_model, ctx->d_df, ctx->grid32, dq0, dq1, n, dv, dc, ctx->d_unc_list,
            ctx->d_unc_count, ctx->d_stats);
    } else
    if (v32_persistent()) {
        const int epb = V32P_EDGES_PER_THREAD * t32;
        edges_valid32p_kernel<<<(n + epb - 1) / epb, t32, v32_smem(ctx), ctx->stream>>>(
            ctx->d_blob, ctx->blob_words, ctx->d_model, ctx->d_df, ctx->grid32, dq0, dq1, n, dv, dc, ctx->d_unc_list,
            ctx->d_unc_count, ctx->d_stats);
    } else
    {
        (ctx->v32_ptrees > 0 ? edges_valid32_kernel<PAIRS_ROOTS> : edges_valid32_kernel<PAIRS_DESCENT>)
            <<<(n + t32 - 1) / t32, t32, v32_smem(ctx), ctx->stream>>>(
            ctx->d_blob, ctx->blob_words, ctx->d_model, ctx->d_df, ctx->grid32, dq0, dq1, n, dv, dc, ctx->d_unc_list,
            ctx->d_unc_count, ctx->d_stats, ctx->d_unc_mask);
        masked = true;
    }
    if (warp_resolve()) {
        const int blocks = std::max(1, std::min((n / 64 + RESOLVE_WARPS - 1) / RESOLVE_WARPS + 1, 8 * ctx->sm_count));
        edges_resolve_kernel<<<blocks, 32 * RESOLVE_WARPS, 0, ctx->stream>>>(
            ctx->d_model, ctx->d_df, ctx->grid, dq0, dq1, n, dv, ctx->d_unc_list, ctx->d_unc_count,
            masked ? ctx->d_unc_mask : nullptr);
    } else {
        const int per_block = std::max(1, vt / 4);
        const int blocks = std::max(1, std::min((n + per_block - 1) / per_block, 2 * ctx->sm_count));
        edges_valid_kernel<<<blocks, vt, validity_smem(ctx), ctx->stream>>>(
            ctx->d_model, ctx->d_df, ctx->grid, dq0, dq1, n, dv, nullptr, nullptr, ctx->d_unc_list, ctx->d_unc_count);
    }
    ctx->launches += 2;
    CU(cudaGetLastError());
    return 0;
}

int smplgpu_is_states_valid_dev(smplgpu_ctx* ctx, const double* q_dev, int n, uint8_t* verdict_dev)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (n == 0) return 0;
    if (!q_dev || !verdict_dev) return fail(ctx, SMPLGPU_ERR_INVALID, "null device pointer");
    CU(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    return launch_states(ctx, q_dev, n, verdict_dev);
}

int smplgpu_is_edges_valid_dev(smplgpu_ctx* ctx, const double* q0_dev, const double* q1_dev, int n,
                               uint8_t* verdict_dev, int32_t* counts_dev)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (n == 0) return 0;
    if (!q0_dev || !q1_dev || !verdict_dev) return fail(ctx, SMPLGPU_ERR_INVALID, "null device pointer");
    CU(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    return launch_edges(ctx, q0_dev, q1_dev, n, verdict_dev, counts_dev);
}

// true when `p` is page-locked host memory the device can DMA from / to directly
static bool is_pinned_host(const void* p)
{
    if (p == nullptr) {
        return false;
    }
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// The same pipeline for lattice states: item i is dof 16-bit coordinates (ManipLattice::coordToState gives the
// joint values on the device), an edge adds one byte of motion-primitive id.  29 bytes per (state + edge) pair
// cross the bus instead of 116.
static int run_host_batched_lattice(smplgpu_ctx* ctx, const int16_t* coords, const uint8_t* prim8, bool edges, int n,
                                    uint8_t* verdict, int32_t* counts, const double* d_deltas, int n_prims)
{
    const int dof = ctx->h_model->dof;
    // Coordinates are a quarter of the doubles' bytes, so a stage is twice the size the double pipeline uses
    // (measured on B200: 3.17 -> 3.66 G states/s).  A small first stage that doubles up (SMPLGPU_HOST_FIRST_CHUNK,
    // so that the kernels start while most of the batch is still crossing the bus) was measured SLOWER -- 2.58 / 3.09 /
    // 3.36 G states/s for a first stage of 2^14 / 2^16 / 2^17 items: every stage carries a serial chain copy ->
    // convert -> f32 kernel -> f64 resolve -> verdict copy of ~100 us, more stages are more chains -- so by default
    // every stage has the full size.
    static const int chunk = [] {
        const char* e = getenv("SMPLGPU_HOST_CHUNK");
        const int v = e ? atoi(e) : 0;
        return v >= 1024 ? v : (1 << 19);
    }();
    static const int first_chunk = [] {
        const char* e = getenv("SMPLGPU_HOST_FIRST_CHUNK");
        const int v = e ? atoi(e) : 0;
        return v >= 1024 ? v : (1 << 30);
    }();
    std::vector<int> begin(1, 0);
    for (int size = std::min(first_chunk, chunk); begin.back() < n; size = std::min(2 * size, chunk)) {
        begin.push_back(std::min(n, begin.back() + size));
    }
    const int nchunks = (int)begin.size() - 1;
    const int cn = std::min(n, chunk);
    int r = ensure_state_buffers(ctx, (size_t)cn * 2, dof, edges);
    if (r) return r;
    const size_t row = (size_t)dof * sizeof(int16_t);
    if ((r = grow(ctx, (void**)&ctx->d_coord, &ctx->coord_cap, (size_t)cn * 2 * row))) return r;
    if (edges && (r = grow(ctx, (void**)&ctx->d_prim8, &ctx->prim8_cap, (size_t)cn * 2))) return r;
    const bool in_direct = is_pinned_host(coords) && (!edges || is_pinned_host(prim8));
    const bool out_direct = is_pinned_host(verdict) && (!counts || is_pinned_host(counts));
    if (!in_direct) {
        if ((r = grow_pinned(ctx, ctx->pinned, &ctx->pinned_cap, (size_t)cn * (row + 1)))) return r;
    }
    if (!out_direct) {
        if ((r = grow_pinned(ctx, ctx->pinned_out, &ctx->pinned_out_cap, (size_t)cn * (1 + (counts ? sizeof(int) : 0)) + 16))) return r;
    }
    CU(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    CU(cudaEventRecord(ctx->ev_in[0], ctx->stream));
    CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_in[0], 0));
    auto drain = [&](int c) -> int {
        const int b = c & 1;
        const int off = begin[c];
        const int m = begin[c + 1] - off;
        CU(cudaEventSynchronize(ctx->ev[b]));
        memcpy(verdict + off, ctx->pinned_out[b], (size_t)m);
        if (counts) {
            memcpy(counts + off, (uint8_t*)ctx->pinned_out[b] + (((size_t)m + 15) / 16) * 16, (size_t)m * sizeof(int));
        }
        return 0;
    };
    for (int c = 0; c < nchunks; ++c) {
        const int b = c & 1;
        const int off = begin[c];
        const int m = begin[c + 1] - off;
        double* dq0 = ctx->d_q0 + (size_t)b * cn * dof;
        double* dq1 = ctx->d_q1 + (size_t)b * cn * dof;
        uint8_t* dv = ctx->d_verdict + (size_t)b * cn;
        int* dc = ctx->d_counts + (size_t)b * cn;
        int16_t* dcoord = ctx->d_coord + (size_t)b * cn * dof;
        uint8_t* dprim = edges ? ctx->d_prim8 + (size_t)b * cn : nullptr;
        if (c >= 2) {
            if (!out_direct) {
                if ((r = drain(c - 2))) return r;
            } else if (!in_direct) {
                CU(cudaEventSynchronize(ctx->ev[b]));
            }
            CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev[b], 0));
        }
        const void* s0 = coords + (size_t)off * dof;
        const void* s1 = edges ? prim8 + off : nullptr;
        if (!in_direct) {
            uint8_t* pin = (uint8_t*)ctx->pinned[b];
            memcpy(pin, s0, (size_t)m * row);
            s0 = pin;
            if (edges) {
                memcpy(pin + (size_t)cn * row, s1, (size_t)m);
                s1 = pin + (size_t)cn * row;
            }
        }
        CU(cudaMemcpyAsync(dcoord, s0, (size_t)m * row, cudaMemcpyHostToDevice, ctx->copy_stream));
        if (edges) {
            CU(cudaMemcpyAsync(dprim, s1, (size_t)m, cudaMemcpyHostToDevice, ctx->copy_stream));
        }
        CU(cudaEventRecord(ctx->ev_in[b], ctx->copy_stream));
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[b], 0));
        const size_t total = (size_t)m * dof;
        lattice_states_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(
            dcoord, dprim, d_deltas, n_prims, ctx->lattice, dof, m, dq0, edges ? dq1 : nullptr);
        ++ctx->launches;
        r = edges ? launch_edges(ctx, dq0, dq1, m, dv, counts ? dc : nullptr) : launch_states(ctx, dq0, m, dv);
        if (r) return r;
        uint8_t* ov = out_direct ? verdict + off : (uint8_t*)ctx->pinned_out[b];
        CU(cudaMemcpyAsync(ov, dv, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
        if (counts) {
            void* oc = out_direct ? (void*)(counts + off) : (void*)((uint8_t*)ctx->pinned_out[b] + (((size_t)m + 15) / 16) * 16);
            CU(cudaMemcpyAsync(oc, dc, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        }
        CU(cudaEventRecord(ctx->ev[b], ctx->stream));
    }
    if (!out_direct) {
        for (int c = std::max(0, nchunks - 2); c < nchunks; ++c) {
            if ((r = drain(c))) return r;
        }
    }
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// Host-pointer entry points.  The batch is cut into chunks; the host->device copy of chunk k+1 runs on a
// second stream while the kernels of chunk k run, and verdicts stream back behind the kernels.  Page-locked
// caller buffers are used as DMA source / target directly; pageable ones go through pinned staging.
// With `prim_id` the edges are (parent, motion primitive) pairs: only the parents and one int per edge cross
// the bus, the successors are formed on the device from the primitive table `d_deltas`.
static int run_host_batched(smplgpu_ctx* ctx, const double* q0, const double* q1, int n,
                            uint8_t* verdict, int32_t* counts, const int32_t* prim_id = nullptr,
                            const double* d_deltas = nullptr, int n_prims = 0,
                            const int16_t* coords = nullptr, const uint8_t* prim8 = nullptr, bool coord_edges = false)
{
    const int dof = ctx->h_model->dof;
    if (coords != nullptr) {
        return run_host_batched_lattice(ctx, coords, prim8, coord_edges, n, verdict, counts, d_deltas, n_prims);
    }
    const bool by_prim = prim_id != nullptr;
    const bool edges = q1 != nullptr || by_prim;
    static const int chunk = [] {
        const char* e = getenv("SMPLGPU_HOST_CHUNK");   // items per pipeline stage (tuning knob)
        const int v = e ? atoi(e) : 0;
        return v >= 1024 ? v : (1 << 18);
    }();
    const int cn = std::min(n, chunk);
    int r = ensure_state_buffers(ctx, (size_t)cn * 2, dof, edges); // two chunks in flight
    if (r) return r;
    const size_t row = (size_t)dof * sizeof(double);
    const bool in_direct = is_pinned_host(q0) && (!edges || is_pinned_host(by_prim ? (const void*)prim_id : (const void*)q1));
    if (by_prim) {
        r = grow(ctx, (void**)&ctx->d_prim, &ctx->prim_cap, (size_t)cn * 2 * sizeof(int));
        if (r) return r;
    }
    const bool out_direct = is_pinned_host(verdict) && (!counts || is_pinned_host(counts));
    if (!in_direct) {
        r = grow_pinned(ctx, ctx->pinned, &ctx->pinned_cap, (size_t)cn * row * (edges ? 2 : 1));
        if (r) return r;
    }
    if (!out_direct) {
        r = grow_pinned(ctx, ctx->pinned_out, &ctx->pinned_out_cap, (size_t)cn * (1 + (counts ? sizeof(int) : 0)) + 16);
        if (r) return r;
    }
    CU(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    // the copy stream starts after whatever the caller queued on the compute stream
    CU(cudaEventRecord(ctx->ev_in[0], ctx->stream));
    CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_in[0], 0));

    const int nchunks = (n + chunk - 1) / chunk;
    auto drain = [&](int c) -> int {   // staged output of chunk c -> caller buffers
        const int b = c & 1;
        const int off = c * chunk;
        const int m = std::min(chunk, n - off);
        CU(cudaEventSynchronize(ctx->ev[b]));
        memcpy(verdict + off, ctx->pinned_out[b], (size_t)m);
        if (counts) {
            memcpy(counts + off, (uint8_t*)ctx->pinned_out[b] + (((size_t)m + 15) / 16) * 16, (size_t)m * sizeof(int));
        }
        return 0;
    };
    for (int c = 0; c < nchunks; ++c) {
        const int b = c & 1;
        const int off = c * chunk;
        const int m = std::min(chunk, n - off);
        double* dq0 = ctx->d_q0 + (size_t)b * cn * dof;
        double* dq1 = ctx->d_q1 + (size_t)b * cn * dof;
        uint8_t* dv = ctx->d_verdict + (size_t)b * cn;
        int* dc = ctx->d_counts + (size_t)b * cn;
        if (c >= 2) {
            if (!out_direct) {
                r = drain(c - 2);      // also proves the kernels of chunk c-2 are done with buffer b
                if (r) return r;
            } else if (!in_direct) {
                CU(cudaEventSynchronize(ctx->ev[b]));
            }
            CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev[b], 0));   // device buffer b is free again
        }
        const double* s0 = q0 + (size_t)off * dof;
        // second input of an edge batch: the successor states, or one primitive id per edge
        const void* s1 = by_prim ? (const void*)(prim_id + off) : (edges ? (const void*)(q1 + (size_t)off * dof) : nullptr);
        const size_t s1_bytes = by_prim ? (size_t)m * sizeof(int) : (size_t)m * row;
        int* dprim = by_prim ? ctx->d_prim + (size_t)b * cn : nullptr;
        if (!in_direct) {
            uint8_t* pin = (uint8_t*)ctx->pinned[b];
            memcpy(pin, s0, (size_t)m * row);
            s0 = (const double*)pin;
            if (edges) {
                memcpy(pin + (size_t)cn * row, s1, s1_bytes);
                s1 = pin + (size_t)cn * row;
            }
        }
        CU(cudaMemcpyAsync(dq0, s0, (size_t)m * row, cudaMemcpyHostToDevice, ctx->copy_stream));
        if (edges) {
            CU(cudaMemcpyAsync(by_prim ? (void*)dprim : (void*)dq1, s1, s1_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
        }
        CU(cudaEventRecord(ctx->ev_in[b], ctx->copy_stream));
        CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[b], 0));
        if (by_prim) {
            const size_t total = (size_t)m * dof;
            apply_mprims_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(dq0, dprim, d_deltas, n_prims, dof, m, dq1);
            ++ctx->launches;
        }
        r = edges ? launch_edges(ctx, dq0, dq1, m, dv, counts ? dc : nullptr) : launch_states(ctx, dq0, m, dv);
        if (r) return r;
        if (out_direct) {
            CU(cudaMemcpyAsync(verdict + off, dv, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
            if (counts) {
                CU(cudaMemcpyAsync(counts + off, dc, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            }
        } else {
            CU(cudaMemcpyAsync(ctx->pinned_out[b], dv, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
            if (counts) {
                CU(cudaMemcpyAsync((uint8_t*)ctx->pinned_out[b] + (((size_t)m + 15) / 16) * 16, dc, (size_t)m * sizeof(int),
                                   cudaMemcpyDeviceToHost, ctx->stream));
            }
        }
        CU(cudaEventRecord(ctx->ev[b], ctx->stream));
    }
    if (!out_direct) {
        for (int c = std::max(0, nchunks - 2); c < nchunks; ++c) {
            r = drain(c);
            if (r) return r;
        }
    }
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_is_states_valid(smplgpu_ctx* ctx, const double* q, int n, uint8_t* verdict)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (n == 0) return 0;
    if (!q || !verdict) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    return run_host_batched(ctx, q, nullptr, n, verdict, nullptr);
}

int smplgpu_is_edges_valid(smplgpu_ctx* ctx, const double* q0, const double* q1, int n,
                           uint8_t* verdict, int32_t* waypoint_counts)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (n == 0) return 0;
    if (!q0 || !q1 || !verdict) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    return run_host_batched(ctx, q0, q1, n, verdict, waypoint_counts);
}

int smplgpu_is_mprim_edges_valid(smplgpu_ctx* ctx, const double* q0, const int32_t* prim_id, int n,
                                 const double* deltas, int n_prims, uint8_t* verdict, int32_t* waypoint_counts)
{
    if (!ctx || n < 0 || n_prims < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (n == 0) return 0;
    if (!q0 || !prim_id || !verdict || (n_prims > 0 && !deltas)) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const size_t bytes = (size_t)std::max(1, n_prims) * ctx->h_model->dof * sizeof(double);
    r = grow(ctx, (void**)&ctx->d_deltas, &ctx->deltas_cap, bytes);
    if (r) return r;
    if (n_prims > 0) {
        CU(cudaMemcpyAsync(ctx->d_deltas, deltas, (size_t)n_prims * ctx->h_model->dof * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));   // `deltas` may be pageable: do not leave the copy reading it
    }
    return run_host_batched(ctx, q0, nullptr, n, verdict, waypoint_counts, prim_id, ctx->d_deltas, n_prims);
}

int smplgpu_is_indexed_edges_valid(smplgpu_ctx* ctx, const double* points, int n_points, const int32_t* idx_a,
                                   const int32_t* idx_b, int n, uint8_t* verdict, int32_t* waypoint_counts)
{
    if (!ctx || n < 0 || n_points < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (n == 0) return 0;
    if (!points || !idx_a || !idx_b || !verdict) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    for (int e = 0; e < n; ++e) {
        if (idx_a[e] < 0 || idx_a[e] >= n_points || idx_b[e] < 0 || idx_b[e] >= n_points)
            return fail(ctx, SMPLGPU_ERR_INVALID, "edge %d: point index out of range", e);
    }
    const int dof = ctx->h_model->dof;
    // resident for the whole call: the point table, the index pairs, every verdict (and waypoint count)
    const size_t pb = (((size_t)n_points * dof * sizeof(double)) + 255) / 256 * 256;
    const size_t ib = (((size_t)n * sizeof(int)) + 255) / 256 * 256;
    const size_t vb = ((size_t)n + 255) / 256 * 256;
    r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, pb + 2 * ib + vb + (waypoint_counts ? ib : 0));
    if (r) return r;
    uint8_t* base = (uint8_t*)ctx->d_misc;
    double* d_points = (double*)base;
    int* d_a = (int*)(base + pb);
    int* d_b = (int*)(base + pb + ib);
    uint8_t* d_v = base + pb + 2 * ib;
    int* d_c = waypoint_counts ? (int*)(base + pb + 2 * ib + vb) : nullptr;
    const int chunk = 1 << 18;
    const int cn = std::min(n, chunk);
    r = ensure_state_buffers(ctx, (size_t)cn, dof, true);
    if (r) return r;
    CU(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    CU(cudaMemcpyAsync(d_points, points, (size_t)n_points * dof * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_a, idx_a, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_b, idx_b, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    for (int off = 0; off < n; off += chunk) {
        const int m = std::min(chunk, n - off);
        const size_t total = (size_t)m * dof;
        gather_edges_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(d_points, d_a + off, d_b + off, dof, m,
                                                                                       ctx->d_q0, ctx->d_q1);
        ++ctx->launches;
        r = launch_edges(ctx, ctx->d_q0, ctx->d_q1, m, d_v + off, d_c ? d_c + off : nullptr);
        if (r) return r;
    }
    CU(cudaMemcpyAsync(verdict, d_v, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (waypoint_counts) {
        CU(cudaMemcpyAsync(waypoint_counts, d_c, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_set_precision_mode(smplgpu_ctx* ctx, int mode)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    if (mode != SMPLGPU_PRECISION_CERTIFIED_F32 && mode != SMPLGPU_PRECISION_EXACT_F64)
        return fail(ctx, SMPLGPU_ERR_INVALID, "unknown precision mode %d", mode);
    ctx->precision_mode = mode;
    return 0;
}

int smplgpu_certified_bounds(smplgpu_ctx* ctx, double* e_pos, double* eps_cells)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    if (e_pos) *e_pos = ctx->e_pos;
    if (eps_cells) *eps_cells = ctx->eps_cells;
    return ctx->has_model32 ? 1 : 0;
}

// Roofline probe for the validity kernels: how many INDEPENDENT random distance-field lookups per second this device
// sustains on the loaded field (uint16 cells, one 32-byte sector per lookup, the field L2 / L1 resident as in the real
// kernels).  Each thread walks its own LCG sequence of cell indices, eight loads in flight per thread, the whole
// machine occupied; the kernels' lookups are dependent (a descent), so this is their ceiling, not their target.
__global__ void df_gather_probe_kernel(const uint16_t* __restrict__ df, unsigned int n_cells, int iters,
                                       unsigned int* __restrict__ sink)
{
    unsigned int x = (blockIdx.x * blockDim.x + threadIdx.x) * 2654435761u + 12345u;
    unsigned int acc = 0;
    for (int it = 0; it < iters; ++it) {
        unsigned int idx[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            x = x * 1664525u + 1013904223u;
            idx[k] = (unsigned int)(((unsigned long long)x * n_cells) >> 32);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) acc += __ldg(&df[idx[k]]);
    }
    if (acc == 0xFFFFFFFFu) sink[0] = acc;   // keeps the loads alive
}

int smplgpu_probe_df_lookup_rate(smplgpu_ctx* ctx, double* lookups_per_s)
{
    if (!ctx || !lookups_per_s) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    const unsigned int n_cells = (unsigned int)((size_t)ctx->grid.nx * ctx->grid.ny * ctx->grid.nz);
    const int blocks = 16 * ctx->sm_count, threads = 256, iters = 256;
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    for (int pass = 0; pass < 2; ++pass) {   // the first pass warms the caches
        CU(cudaEventRecord(e0, ctx->stream));
        df_gather_probe_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->d_df, n_cells, iters, (unsigned int*)ctx->d_stats);
        CU(cudaEventRecord(e1, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        ++ctx->launches;
    }
    float ms = 0.0f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *lookups_per_s = (double)blocks * threads * iters * 8.0 / ((double)ms * 1e-3);
    return 0;
}

int smplgpu_last_f64_resolved(smplgpu_ctx* ctx, int64_t* items)
{
    if (!ctx || !items) return SMPLGPU_ERR_INVALID;
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    *items = (int64_t)ctx->h_stats[3];
    return 0;
}

int smplgpu_fk_sphere_centers_f32(smplgpu_ctx* ctx, const double* q, int n, float* out)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_model32) return fail(ctx, SMPLGPU_ERR_STATE, "single-precision model not built (robot + distance field needed)");
    if (n == 0) return 0;
    if (!q || !out) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const int dof = ctx->h_model->dof, nn = ctx->h_model->n_nodes;
    const size_t qb = (size_t)n * dof * sizeof(double), ob = (size_t)n * nn * 3 * sizeof(float);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, qb + ob + 64);
    if (r) return r;
    double* dq = (double*)ctx->d_misc;
    float* dout = (float*)(dq + (size_t)n * dof);
    CU(cudaMemcpyAsync(dq, q, qb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemsetAsync(dout, 0, ob, ctx->stream));
    const int t32 = ctx->v32_threads;
    fk_centers32_kernel<<<(n + t32 - 1) / t32, t32, v32_smem(ctx), ctx->stream>>>(
        ctx->d_blob, ctx->blob_words, dq, n, ctx->res, ctx->fk32_origin[0], ctx->fk32_origin[1], ctx->fk32_origin[2], dout);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dout, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_last_validity_stats(smplgpu_ctx* ctx, int64_t* df_lookups, int64_t* pair_tests, int64_t* waypoints)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    CU(cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (df_lookups) *df_lookups = (int64_t)ctx->h_stats[0];
    if (pair_tests) *pair_tests = (int64_t)ctx->h_stats[1];
    if (waypoints) *waypoints = (int64_t)ctx->h_stats[2];
    return 0;
}

int smplgpu_fk_sphere_centers(smplgpu_ctx* ctx, const double* q, int n, double* out)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set");
    if (n == 0) return 0;
    if (!q || !out) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const int dof = ctx->h_model->dof, nn = ctx->h_model->n_nodes;
    const size_t qb = (size_t)n * dof * sizeof(double), ob = (size_t)n * nn * 3 * sizeof(double);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, qb + ob + 64);
    if (r) return r;
    double* dq = (double*)ctx->d_misc;
    double* dout = dq + (size_t)n * dof;
    CU(cudaMemcpyAsync(dq, q, qb, cudaMemcpyHostToDevice, ctx->stream));
    const int vt = ctx->validity_threads;
    fk_centers_kernel<<<(n + vt - 1) / vt, vt, validity_smem(ctx), ctx->stream>>>(
        ctx->d_model, dq, n, dout);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dout, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_collision_distance(smplgpu_ctx* ctx, const double* q, int n, double* out)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (n == 0) return 0;
    if (!q || !out) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const int dof = ctx->h_model->dof;
    const size_t qb = (size_t)n * dof * sizeof(double), ob = (size_t)n * sizeof(double);
    r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, qb + ob + 64);
    if (r) return r;
    double* dq = (double*)ctx->d_misc;
    double* dout = dq + (size_t)n * dof;
    CU(cudaMemcpyAsync(dq, q, qb, cudaMemcpyHostToDevice, ctx->stream));
    collision_distance_kernel<<<(n + 63) / 64, 64, 0, ctx->stream>>>(ctx->d_model, ctx->d_df, ctx->grid, ctx->res, ctx->padding, dq, n, dout);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dout, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_check_joint_limits(smplgpu_ctx* ctx, const double* q, int n, uint8_t* ok)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set");
    if (n == 0) return 0;
    if (!q || !ok) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const int dof = ctx->h_model->dof;
    const size_t qb = (size_t)n * dof * sizeof(double);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, qb + n + 64);
    if (r) return r;
    double* dq = (double*)ctx->d_misc;
    uint8_t* dok = (uint8_t*)(dq + (size_t)n * dof);
    CU(cudaMemcpyAsync(dq, q, qb, cudaMemcpyHostToDevice, ctx->stream));
    joint_limits_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_model, dq, n, dok);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(ok, dok, n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

///////////////////////////////////////////////////////////////////////////////
// BFS
///////////////////////////////////////////////////////////////////////////////

static int alloc_grid(smplgpu_ctx* ctx, BfsGrid& g, int nx, int ny, int nz, size_t* words, size_t* cells)
{
    if (nx <= 0 || ny <= 0 || nz <= 0) return fail(ctx, SMPLGPU_ERR_INVALID, "bad BFS dimensions");
    if ((long long)(nx + 2) * (ny + 2) * (nz + 2) > 0x7FFFFFFFLL) return fail(ctx, SMPLGPU_ERR_LIMIT, "BFS grid too large for int nodes");
    free_grid(g);
    g.nx = nx; g.ny = ny; g.nz = nz;
    g.DX = nx + 2; g.DY = ny + 2; g.DZ = nz + 2;
    g.W = ((g.DX + 31) / 32 + 3) / 4 * 4;
    g.rows = g.DY * g.DZ;
    *words = (size_t)g.rows * g.W;
    *cells = (size_t)g.rows * g.DX;
    const size_t wb = *words * sizeof(uint32_t);
    CU(cudaMalloc(&g.wall, wb));
    CU(cudaMalloc(&g.blocked, wb));
    CU(cudaMalloc(&g.front0, wb));
    CU(cudaMalloc(&g.front1, wb));
    CU(cudaMalloc(&g.cand0, (size_t)g.rows * sizeof(uint32_t)));
    CU(cudaMalloc(&g.cand1, (size_t)g.rows * sizeof(uint32_t)));
    CU(cudaMalloc(&g.dist, *cells * sizeof(int)));
    CU(cudaMalloc(&g.ctrl, 16 * sizeof(int)));
    return 0;
}

static int alloc_bfs(smplgpu_ctx* ctx, int nx, int ny, int nz)
{
    if (ctx->has_bfs && ctx->bfs.nx == nx && ctx->bfs.ny == ny && ctx->bfs.nz == nz) {
        return 0;
    }
    ctx->has_bfs = false;
    int r = alloc_grid(ctx, ctx->bfs, nx, ny, nz, &ctx->bfs_words, &ctx->bfs_cells);
    if (r) return r;
    r = alloc_tiles(ctx, ctx->bfs, ctx->bfs_tiles, ctx->bfs_words);
    if (r) return r;
    ctx->has_bfs = true;
    return 0;
}

// largest d2 with res*sqrt(d2) <= radius  (grid()->getDistance(x,y,z) <= radius, bfs_heuristic.cpp:343)
static int wall_threshold(const smplgpu_ctx* ctx, double inflation_radius)
{
    int kmax = -1;
    for (int k = 0; k <= ctx->dmax_sq; ++k) {
        if (ctx->res * std::sqrt((double)k) <= inflation_radius) {
            kmax = k;
        } else {
            break;
        }
    }
    return kmax;
}

// With the LEVEL kernel forced for the banks (smplgpu_bfs_set_mode / SMPLGPU_BFS_MODE=1), asynchronous bank runs are one
// cooperative launch per run, taking turns per device, or -- with SMPLGPU_BANK_STEPWISE=1 -- one launch per level
// (bfs_level_step_kernel).  Measured on one B200, 6 contexts x 342 queries: cooperative 1960-2040 plan queries/s, level
// by level 1340-2010 (142 launches per run and context).  The default for the banks is the tile kernel, one launch per
// super-step (run_grid): 2320-2460.
static bool bank_stepwise()
{
    static const bool on = [] {
        const char* e = getenv("SMPLGPU_BANK_STEPWISE");
        return e != nullptr && atoi(e) != 0;
    }();
    return on;
}

constexpr int BANK_LEVEL_CHUNK = 128;   // level launches queued at a time (a 150^3 tabletop bank needs ~140 levels)
constexpr int BANK_TILE_CHUNK = 24;     // super-step launches queued at a time (TILE_K levels each)

static int launch_bank_level_chunk(smplgpu_ctx* ctx, cudaStream_t stream)
{
    BfsGrid& g = ctx->bank;
    if (ctx->bank_step_tiles != 0) {
        // the tile kernel, one super-step per launch; bank_next_level counts super-steps from 1
        const BfsTiles& t = ctx->bank_tiles;
        const bool large = ctx->bank_step_tiles == TILE_RPT_LARGE;
        const int threads = large ? TILE_THREADS / TILE_RPT_LARGE : TILE_THREADS;
        // SMPLGPU_BANK_TILE_CHUNK: a smaller chunk, for the tests of the continuation path
        static const int chunk = getenv("SMPLGPU_BANK_TILE_CHUNK") ? std::max(1, atoi(getenv("SMPLGPU_BANK_TILE_CHUNK"))) : BANK_TILE_CHUNK;
        for (int k = 0; k < chunk; ++k) {
            const int step = ctx->bank_next_level - 1 + k;
            if (large) {
                bfs_tiles_kernel<TILE_RPT_LARGE><<<ctx->bank_step_blocks, threads, 0, stream>>>(g, t, step + 1, step, 1, ctx->bank_done);
            } else {
                bfs_tiles_kernel<1><<<ctx->bank_step_blocks, threads, 0, stream>>>(g, t, step + 1, step, 1, ctx->bank_done);
            }
        }
        ctx->launches += chunk;
        ctx->bank_next_level += chunk;
        CU(cudaGetLastError());
        return 0;
    }
    const int groups = (g.rows + 7) / 8;
    const int blocks = std::max(1, std::min(groups, 2 * ctx->sm_count));
    for (int k = 0; k < BANK_LEVEL_CHUNK; ++k) {
        bfs_level_step_kernel<<<blocks, BFS_THREADS, 0, stream>>>(g, (uint32_t)(ctx->bank_next_level + k), ctx->bank_done);
    }
    ctx->launches += BANK_LEVEL_CHUNK;
    ctx->bank_next_level += BANK_LEVEL_CHUNK;
    CU(cudaGetLastError());
    return 0;
}

// which kernel a bank run uses (a single grid always takes the tile kernel unless a mode is forced)
static bool bank_uses_tiles(const smplgpu_ctx* ctx)
{
    return ctx->bfs_mode == SMPLGPU_BFS_TILES || ctx->bfs_mode == SMPLGPU_BFS_AUTO;
}

// asynchronous bank runs launch step by step (no co-residency needed, the contexts' runs overlap): always with the tile
// kernel, with the level kernel only on request (SMPLGPU_BANK_STEPWISE=1)
static bool bank_async_stepwise(const smplgpu_ctx* ctx)
{
    static const bool cooperative = getenv("SMPLGPU_BANK_COOPERATIVE") != nullptr && atoi(getenv("SMPLGPU_BANK_COOPERATIVE")) != 0;
    return (bank_uses_tiles(ctx) && !cooperative) || (!bank_uses_tiles(ctx) && bank_stepwise());
}

// reset + seed + all levels on one grid; seeds already on the device (padded-grid-free coordinates)
static int run_grid(smplgpu_ctx* ctx, BfsGrid& g, size_t words, const int* d_seeds, int n_seeds, int* levels_out,
                    const uint8_t* d_slot_mask = nullptr, int slot_dz = 1, cudaStream_t stream = nullptr,
                    int* d_seed_count = nullptr)
{
    if (stream == nullptr) stream = ctx->stream;
    if (d_seed_count == nullptr) d_seed_count = ctx->d_seed_count;
    const int total = (int)words;
    BfsTiles& t = (&g == &ctx->bank) ? ctx->bank_tiles : ctx->bfs_tiles;
    // AUTO: the tile kernel everywhere.  For the stacked planner banks it does a query in 0.085 ms against the level
    // kernel's 0.157 ms (tools/bank_bfs_time.py) and, inside the planner, 2320-2460 against 1960-2040 plan queries/s
    // (DESIGN.md section 7).  A run queued behind the caller's back goes ONE SUPER-STEP PER LAUNCH: a cooperative launch
    // of blocks that fill the register file of every SM they sit on has to wait until all of them fit at once, which
    // nothing guarantees while other contexts' expansion rounds keep arriving; SMPLGPU_BANK_COOPERATIVE=1 restores the
    // single cooperative launch (same throughput: 2370-2410).
    const bool single = &g != &ctx->bank;
    const bool tiles = single ? ctx->bfs_mode != SMPLGPU_BFS_LEVELS : bank_uses_tiles(ctx);
    {
        // one warp per 32 bitmap words; at least one thread per row for the candidate stamps
        const long long threads = std::max<long long>(g.rows, std::min<long long>((long long)total, 148LL * 2048 * 4));
        bfs_reset_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(g, d_slot_mask, slot_dz);
    }
    ++ctx->launches;
    if (tiles && t.tb[0] == nullptr) {
        const int r = alloc_tiles(ctx, g, t, words);
        if (r) return r;
    }
    if (tiles) {
        bfs_tiles_reset_kernel<<<(unsigned)std::min<long long>(((long long)t.ntiles * TILE_WORDS + 255) / 256, 148 * 16), 256, 0, stream>>>(g, t, d_slot_mask, slot_dz);
        ++ctx->launches;
        CU(cudaMemsetAsync(t.ver, 0, ((size_t)7 * t.ntiles + 16) * sizeof(uint32_t), stream));
    }
    if (n_seeds <= 0) {
        CU(cudaGetLastError());
        return 0;
    }
    CU(cudaMemsetAsync(d_seed_count, 0, sizeof(int), stream));
    bfs_seed_kernel<<<(n_seeds + 127) / 128, 128, 0, stream>>>(g, d_seeds, n_seeds, d_seed_count);
    ++ctx->launches;
    long long cap = (long long)g.nx * g.ny * g.nz;
    if (tiles) {
        bfs_tiles_seed_kernel<<<(n_seeds + 127) / 128, 128, 0, stream>>>(g, t, d_seeds, n_seeds);
        ++ctx->launches;
        // persistent cooperative kernel, TILE_K levels per grid barrier: 1024-thread blocks, one per SM, for grids with
        // few tiles; 256-thread blocks, four per SM, for large ones (bfs_tiles.cuh; SMPLGPU_BFS_TILE_RPT forces 1 or 4)
        static const int forced = getenv("SMPLGPU_BFS_TILE_RPT") ? atoi(getenv("SMPLGPU_BFS_TILE_RPT")) : 0;
        const bool warp_tiles = forced == 32;   // bfs_warp_tiles_kernel: one warp per tile, rows in registers
        const bool large = forced > 0 ? forced >= 2 : t.ntiles >= 4096;
        const int rpt = forced == 2 ? 2 : TILE_RPT_LARGE;
        const void* kern = warp_tiles ? (const void*)bfs_warp_tiles_kernel
                                      : (large ? (rpt == 2 ? (const void*)bfs_tiles_kernel<2> : (const void*)bfs_tiles_kernel<TILE_RPT_LARGE>)
                                               : (const void*)bfs_tiles_kernel<1>);
        const int threads = warp_tiles ? WTILE_WARPS * 32 : (large ? TILE_THREADS / rpt : TILE_THREADS);
        int per_sm = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, 0));
        if (per_sm < 1) return fail(ctx, SMPLGPU_ERR_CUDA, "BFS tile kernel does not fit an SM");
        per_sm = std::min(per_sm, warp_tiles ? WTILE_BLOCKS_PER_SM : (large ? rpt : 1));
        // A run queued behind the caller's back (smplgpu_bfs_bank_run_slots_async) leaves room for the expansion
        // rounds that are meant to keep flowing meanwhile: three of the four block slots of every SM (large grids), or
        // seven eighths of the SMs (1024-thread blocks); a synchronous run takes the whole machine.
        const bool async_run = stream == ctx->bfs_stream;
        if (async_run && (large || warp_tiles)) per_sm = std::max(1, per_sm - 1);
        const int sms = (async_run && !large && !warp_tiles) ? ctx->sm_count - std::max(1, ctx->sm_count / 8) : ctx->sm_count;
        const int tiles_per_block = warp_tiles ? WTILE_WARPS : 1;
        const int blocks = std::max(1, std::min(sms * per_sm, (t.ntiles + tiles_per_block - 1) / tiles_per_block));
        int max_steps = (int)std::min<long long>(cap / TILE_K + 2, 0x7FFFFFFFLL / blocks - 1);
        if (async_run && &g == &ctx->bank && !warp_tiles && rpt != 2 && bank_async_stepwise(ctx)) {
            // behind the caller's back: one launch per super-step, first chunk here, the rest from
            // smplgpu_bfs_bank_run_done / _wait
            if (!ctx->bank_done) {
                int* p = nullptr;
                CU(cudaHostAlloc((void**)&p, 64, cudaHostAllocMapped));
                ctx->bank_done = p;
            }
            *ctx->bank_done = 0;
            ctx->bank_next_level = 1;
            ctx->bank_level_cap = max_steps;
            ctx->bank_step_tiles = large ? TILE_RPT_LARGE : 1;
            ctx->bank_step_blocks = std::max(1, std::min(ctx->sm_count * (large ? TILE_RPT_LARGE : 1), t.ntiles));
            const int r = launch_bank_level_chunk(ctx, stream);
            if (r) return r;
        } else {
            int first_step = 0, stepwise = 0;
            volatile int* no_flag = nullptr;
            void* args[] = { (void*)&g, (void*)&t, (void*)&max_steps, (void*)&first_step, (void*)&stepwise, (void*)&no_flag };
            CU(cudaLaunchCooperativeKernel(kern, dim3(blocks), dim3(threads), args, 0, stream));
            ++ctx->launches;
        }
    } else if (&g == &ctx->bank && stream == ctx->bfs_stream && bank_stepwise()) {
        // behind the caller's back: one launch per level (bfs_level_step_kernel), first chunk here, the rest from
        // smplgpu_bfs_bank_run_done / _wait
        if (!ctx->bank_done) {
            int* p = nullptr;
            CU(cudaHostAlloc((void**)&p, 64, cudaHostAllocMapped));
            ctx->bank_done = p;
        }
        *ctx->bank_done = 0;
        ctx->bank_next_level = 1;
        ctx->bank_level_cap = std::min<long long>(cap, 1LL << 22);
        ctx->bank_step_tiles = 0;
        const int r = launch_bank_level_chunk(ctx, stream);
        if (r) return r;
    } else {
        // persistent cooperative kernel, one block per SM (the grid barrier costs one arrival per block)
        int per_sm = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bfs_levels_kernel, BFS_THREADS, 0));
        if (per_sm < 1) return fail(ctx, SMPLGPU_ERR_CUDA, "BFS kernel does not fit an SM");
        const int groups = (g.rows + 7) / 8;
        // A block of this kernel takes a whole SM (1024 threads x 62 registers).  A run queued behind the caller's
        // back (smplgpu_bfs_bank_run_slots_async) leaves an eighth of the SMs to the expansion batches that are
        // meant to keep flowing meanwhile; a synchronous run takes them all.
        const int sms = stream == ctx->bfs_stream ? ctx->sm_count - std::max(1, ctx->sm_count / 8) : ctx->sm_count;
        const int blocks = std::max(1, std::min(sms, groups));
        int max_levels = (int)std::min<long long>(cap, (1LL << 22));
        max_levels = (int)std::min<long long>(max_levels, 0x7FFFFFFFLL / blocks - 1);   // barrier target level * blocks
        void* args[] = { (void*)&g, (void*)&max_levels };
        CU(cudaLaunchCooperativeKernel((void*)bfs_levels_kernel, dim3(blocks), dim3(BFS_THREADS), args, 0, stream));
        ++ctx->launches;
    }
    if (levels_out) {
        CU(cudaMemcpyAsync(levels_out, g.ctrl, sizeof(int), cudaMemcpyDeviceToHost, stream));
    }
    return 0;
}

int smplgpu_bfs_set_mode(smplgpu_ctx* ctx, int mode)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    if (mode != SMPLGPU_BFS_TILES && mode != SMPLGPU_BFS_LEVELS && mode != SMPLGPU_BFS_AUTO) return fail(ctx, SMPLGPU_ERR_INVALID, "unknown BFS mode %d", mode);
    ctx->bfs_mode = mode;
    return 0;
}

int smplgpu_bfs_set_walls_dev(smplgpu_ctx* ctx, int nx, int ny, int nz, const uint8_t* walls_dev)
{
    if (!ctx || !walls_dev) return SMPLGPU_ERR_INVALID;
    int r = alloc_bfs(ctx, nx, ny, nz);
    if (r) return r;
    ++ctx->scene_epoch;
    const int total = (int)ctx->bfs_words;
    bfs_walls_from_bytes_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(ctx->bfs, walls_dev);
    ++ctx->launches;
    CU(cudaGetLastError());
    return 0;
}

int smplgpu_bfs_set_walls(smplgpu_ctx* ctx, int nx, int ny, int nz, const uint8_t* walls)
{
    if (!ctx || !walls) return SMPLGPU_ERR_INVALID;
    const size_t n = (size_t)nx * ny * nz;
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, n);
    if (r) return r;
    CU(cudaMemcpyAsync(ctx->d_misc, walls, n, cudaMemcpyHostToDevice, ctx->stream));
    r = smplgpu_bfs_set_walls_dev(ctx, nx, ny, nz, (const uint8_t*)ctx->d_misc);
    if (r) return r;
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_bfs_set_walls_from_df(smplgpu_ctx* ctx, double inflation_radius)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "distance field not set");
    int r = alloc_bfs(ctx, ctx->grid.nx, ctx->grid.ny, ctx->grid.nz);
    if (r) return r;
    ++ctx->scene_epoch;
    const int kmax = wall_threshold(ctx, inflation_radius);
    unsigned int* d_count = (unsigned int*)ctx->d_seed_count;
    CU(cudaMemsetAsync(d_count, 0, sizeof(unsigned int), ctx->stream));
    const int total = (int)ctx->bfs_words;
    bfs_walls_from_df_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(ctx->bfs, ctx->d_df, kmax, ctx->bfs.DZ, d_count, nullptr);
    ++ctx->launches;
    CU(cudaGetLastError());
    unsigned int count = 0;
    CU(cudaMemcpyAsync(&count, d_count, sizeof(count), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return (int)count;
}

int smplgpu_bfs_run(smplgpu_ctx* ctx, const int32_t* seeds_xyz, int n_seeds)
{
    if (!ctx || n_seeds < 0 || (n_seeds > 0 && !seeds_xyz)) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_bfs) return fail(ctx, SMPLGPU_ERR_STATE, "BFS walls not set");
    BfsGrid& g = ctx->bfs;
    // in-bounds seeds only (BFS_3D::run returns 0 for an out-of-bounds origin, bfs3d.cpp:169-171)
    std::vector<int> inb;
    for (int i = 0; i < n_seeds; ++i) {
        const int x = seeds_xyz[3 * i], y = seeds_xyz[3 * i + 1], z = seeds_xyz[3 * i + 2];
        if (x >= 0 && y >= 0 && z >= 0 && x < g.nx && y < g.ny && z < g.nz) {
            inb.push_back(x); inb.push_back(y); inb.push_back(z);
        }
    }
    const int n_in = (int)inb.size() / 3;
    if (n_in > 0) {
        int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, inb.size() * sizeof(int));
        if (r) return r;
        CU(cudaMemcpyAsync(ctx->d_misc, inb.data(), inb.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    }
    ctx->bfs_levels = 0;
    ++ctx->scene_epoch;
    int r = run_grid(ctx, g, ctx->bfs_words, (const int*)ctx->d_misc, n_in, &ctx->bfs_levels);
    if (r) return r;
    CU(cudaStreamSynchronize(ctx->stream));
#ifdef SMPLGPU_BFS_STATS
    {
        int c[8];
        cudaMemcpy(c, g.ctrl, sizeof(c), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[bfs stats] queued tile-steps %d, with frontier %d, sub-levels run %d\n", c[3], c[6], c[7]);
        if (ctx->bfs_tiles.qn) {
            unsigned long long tt[4];
            cudaMemcpy(tt, ctx->bfs_tiles.qn + 8, sizeof(tt), cudaMemcpyDeviceToHost);
            fprintf(stderr, "[bfs stats] block-cycles: load %.1f M, levels %.1f M, write-back %.1f M, grid barrier %.1f M\n",
                    tt[0] * 1e-6, tt[1] * 1e-6, tt[2] * 1e-6, tt[3] * 1e-6);
            static unsigned long long dbg[4][2048];
            cudaMemcpyFromSymbol(dbg, bfs_dbg, sizeof(dbg));
            unsigned long long sum_max = 0, sum_all = 0, multi = 0, steps = 0, sum_q = 0;
            for (int i = 0; i < 2048; ++i) {
                if (dbg[0][i] == 0) continue;
                ++steps; sum_max += dbg[1][i]; sum_all += dbg[3][i]; sum_q += dbg[0][i];
                if (dbg[2][i] > 1) ++multi;
                if (getenv("SMPLGPU_BFS_STATS_STEPS")) fprintf(stderr, "  step %d: queue %llu, slowest block %llu cycles, most tiles per block %llu, mean busy %llu\n", i, dbg[0][i], dbg[1][i], dbg[2][i], dbg[3][i] / 592);
            }
            fprintf(stderr, "[bfs stats] %llu super-steps, %llu tiles queued, sum of slowest-block cycles %.2f M, sum of all busy cycles %.1f M, super-steps where a block took > 1 tile: %llu\n",
                    steps, sum_q, sum_max * 1e-6, sum_all * 1e-6, multi);
            static unsigned long long zero[4][2048];
            cudaMemcpyToSymbol(bfs_dbg, zero, sizeof(zero));
        }
    }
#endif
    return n_in;
}

int smplgpu_bfs_distances(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n, int32_t* out)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_bfs) return fail(ctx, SMPLGPU_ERR_STATE, "BFS walls not set");
    if (n == 0) return 0;
    if (!cells_xyz || !out) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, (size_t)n * 4 * sizeof(int));
    if (r) return r;
    int* dc = (int*)ctx->d_misc;
    int* dout = dc + (size_t)n * 3;
    CU(cudaMemcpyAsync(dc, cells_xyz, (size_t)n * 3 * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    bfs_gather_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->bfs, dc, n, dout);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dout, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_bfs_download(smplgpu_ctx* ctx, int32_t* padded_grid)
{
    if (!ctx || !padded_grid) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_bfs) return fail(ctx, SMPLGPU_ERR_STATE, "BFS walls not set");
    CU(cudaMemcpyAsync(padded_grid, ctx->bfs.dist, ctx->bfs_cells * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_bfs_dims(smplgpu_ctx* ctx, int32_t dims[3])
{
    if (!ctx || !dims) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_bfs) return fail(ctx, SMPLGPU_ERR_STATE, "BFS walls not set");
    dims[0] = ctx->bfs.nx; dims[1] = ctx->bfs.ny; dims[2] = ctx->bfs.nz;
    return 0;
}

int smplgpu_bfs_last_levels(smplgpu_ctx* ctx) { return ctx ? ctx->bfs_levels : SMPLGPU_ERR_INVALID; }

///////////////////////////////////////////////////////////////////////////////
// heuristic
///////////////////////////////////////////////////////////////////////////////

int smplgpu_goal_heuristics_dev(smplgpu_ctx* ctx, const double* q_dev, int n, int cost_per_cell, int32_t* h_dev)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set");
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "distance field (grid geometry) not set");
    if (!ctx->has_bfs) return fail(ctx, SMPLGPU_ERR_STATE, "BFS walls not set");
    if (ctx->bfs.nx != ctx->grid.nx || ctx->bfs.ny != ctx->grid.ny || ctx->bfs.nz != ctx->grid.nz)
        return fail(ctx, SMPLGPU_ERR_STATE, "BFS grid (%dx%dx%d) does not match the distance field (%dx%dx%d): set the walls again",
                    ctx->bfs.nx, ctx->bfs.ny, ctx->bfs.nz, ctx->grid.nx, ctx->grid.ny, ctx->grid.nz);
    if (n == 0) return 0;
    if (!q_dev || !h_dev) return fail(ctx, SMPLGPU_ERR_INVALID, "null device pointer");
    goal_heuristic_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(
        ctx->d_model, ctx->grid, ctx->bfs.dist, ctx->bfs.DX, ctx->bfs.DY, ctx->bfs.DZ, q_dev, n, cost_per_cell, h_dev);
    ++ctx->launches;
    CU(cudaGetLastError());
    return 0;
}

int smplgpu_goal_heuristics(smplgpu_ctx* ctx, const double* q, int n, int cost_per_cell, int32_t* h)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set");
    if (n == 0) return 0;
    if (!q || !h) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const int dof = ctx->h_model->dof;
    const size_t qb = (size_t)n * dof * sizeof(double);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, qb + (size_t)n * sizeof(int) + 64);
    if (r) return r;
    double* dq = (double*)ctx->d_misc;
    int* dh = (int*)(dq + (size_t)n * dof);
    CU(cudaMemcpyAsync(dq, q, qb, cudaMemcpyHostToDevice, ctx->stream));
    r = smplgpu_goal_heuristics_dev(ctx, dq, n, cost_per_cell, dh);
    if (r) return r;
    CU(cudaMemcpyAsync(h, dh, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int smplgpu_planning_frame_fk(smplgpu_ctx* ctx, const double* q, int n, double* pose6)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set");
    if (n == 0) return 0;
    if (!q || !pose6) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const int dof = ctx->h_model->dof;
    const size_t qb = (size_t)n * dof * sizeof(double), ob = (size_t)n * 6 * sizeof(double);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, qb + ob + 64);
    if (r) return r;
    double* dq = (double*)ctx->d_misc;
    double* dout = dq + (size_t)n * dof;
    CU(cudaMemcpyAsync(dq, q, qb, cudaMemcpyHostToDevice, ctx->stream));
    planning_fk_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_model, dq, n, dout);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(pose6, dout, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

///////////////////////////////////////////////////////////////////////////////
// many queries at once: BFS bank + fused expansion batch
///////////////////////////////////////////////////////////////////////////////

int smplgpu_bfs_bank_max_slots(smplgpu_ctx* ctx)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "distance field not set");
    const long long nx = ctx->grid.nx, ny = ctx->grid.ny, nz = ctx->grid.nz;
    // (nx+2)(ny+2)(n (nz+2)) <= 2^31 - 1
    long long by_index = 0x7FFFFFFFLL / ((nx + 2) * (ny + 2)) / (nz + 2);
    // distances (4 B per padded cell) + four bitmaps + candidate words: ~4.7 B per cell, + the tile kernel's four
    // tile-major bitmaps (0.5 B per cell, padded to whole tiles: ~0.7 B); keep half the free memory
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
        size_t have = free_b + (ctx->has_bank ? (size_t)ctx->bank_cells * 5 : 0);
        long long by_mem = (long long)((double)have * 0.5 / (5.4 * (double)((nx + 2) * (ny + 2) * (nz + 2))));
        by_index = std::min(by_index, by_mem);
    }
    return (int)std::max(1LL, std::min(by_index, 1LL << 20));
}

// the staging of a bank run of n_seeds seeds: seeds | slot mask, on the device and in page-locked memory
static int reserve_bank_stage(smplgpu_ctx* ctx, size_t n_seeds, size_t* seed_cap)
{
    *seed_cap = (n_seeds * 3 * sizeof(int) + 15) / 16 * 16;
    const size_t need = *seed_cap + (size_t)ctx->bank_slots + 64;
    int r = grow(ctx, &ctx->d_bank_stage, &ctx->bank_stage_cap, need);
    if (r) return r;
    if (need > ctx->h_bank_stage_cap) {
        if (ctx->h_bank_stage) { CU(cudaFreeHost(ctx->h_bank_stage)); ctx->h_bank_stage = nullptr; ctx->h_bank_stage_cap = 0; }
        CU(cudaMallocHost(&ctx->h_bank_stage, need));
        ctx->h_bank_stage_cap = need;
    }
    return 0;
}

int smplgpu_bfs_bank_create(smplgpu_ctx* ctx, int n_slots, double inflation_radius)
{
    if (!ctx || n_slots <= 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_df) return fail(ctx, SMPLGPU_ERR_STATE, "distance field not set");
    {
        const int fr = finish_bank_run(ctx);
        if (fr) return fr;
    }
    const int nx = ctx->grid.nx, ny = ctx->grid.ny, nz = ctx->grid.nz;
    const long long total_nz = (long long)n_slots * (nz + 2) - 2;
    if ((long long)(nx + 2) * (ny + 2) * (total_nz + 2) > 0x7FFFFFFFLL)
        return fail(ctx, SMPLGPU_ERR_LIMIT, "%d slots of %dx%dx%d exceed int node indices", n_slots, nx, ny, nz);
    // the bank is a scene-level resource: keep the (multi-gigabyte) allocation when the shape is unchanged --
    // allocating it takes anything from 0.1 to 0.7 s
    const bool same_shape = ctx->has_bank && ctx->bank_slots == n_slots && ctx->bank.nx == nx && ctx->bank.ny == ny &&
                            ctx->bank.nz == (int)total_nz;
    ctx->has_bank = false;
    if (!same_shape) {
        int r = alloc_grid(ctx, ctx->bank, nx, ny, (int)total_nz, &ctx->bank_words, &ctx->bank_cells);
        if (r) return r;
        free_tiles(ctx->bank_tiles);   // allocated by the first run that uses the tile kernel on the bank (run_grid)
    }
    ctx->bank_slots = n_slots;
    ctx->bank_slot_dz = nz + 2;
    {
        // room for a full goal set in every slot: runs queued while planners work never allocate
        size_t seed_cap = 0;
        const int r = reserve_bank_stage(ctx, (size_t)n_slots * SMPLGPU_MAX_GOAL_SET, &seed_cap);
        if (r) return r;
    }
    const int kmax = wall_threshold(ctx, inflation_radius);
    ctx->bank_kmax = kmax;
    unsigned int* d_count = (unsigned int*)ctx->d_seed_count;
    CU(cudaMemsetAsync(d_count, 0, sizeof(unsigned int), ctx->stream));
    const int total = (int)ctx->bank_words;
    bfs_walls_from_df_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(ctx->bank, ctx->d_df, kmax, ctx->bank_slot_dz, d_count, nullptr);
    ++ctx->launches;
    CU(cudaGetLastError());
    unsigned int count = 0;
    CU(cudaMemcpyAsync(&count, d_count, sizeof(count), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->has_bank = true;
    return (int)count;
}

// queues one bank run (walls of the listed slots from the field, reset, wavefront) on `stream`; the seeds and the
// slot mask are staged in page-locked memory owned by the context, so nothing of the caller is read afterwards.
// Slot slots[i] is seeded at seeds_xyz[seed_offsets[i] .. seed_offsets[i + 1] - 1] (seed_offsets null: seed i alone).
static int launch_bank_run(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz, const int32_t* seed_offsets,
                           int n, cudaStream_t stream, int* d_seed_count, int* n_seeds_out)
{
    const int nx = ctx->grid.nx, ny = ctx->grid.ny, nz = ctx->grid.nz;
    ctx->bank_next_level = 0;   // set again by run_grid when this run goes level by level
    size_t seed_cap = 0;
    int r = reserve_bank_stage(ctx, seed_offsets ? (size_t)seed_offsets[n] : (size_t)n, &seed_cap);
    if (r) return r;
    int* h_seeds = (int*)ctx->h_bank_stage;
    uint8_t* h_mask = (uint8_t*)ctx->h_bank_stage + seed_cap;
    memset(h_mask, 0, (size_t)ctx->bank_slots);
    int n_in = 0;
    for (int i = 0; i < n; ++i) {
        const int s = slots[i];
        if (s < 0 || s >= ctx->bank_slots) return fail(ctx, SMPLGPU_ERR_INVALID, "slot %d out of range", s);
        if (h_mask[s]) return fail(ctx, SMPLGPU_ERR_INVALID, "slot %d listed twice", s);
        h_mask[s] = 1;
        const int e0 = seed_offsets ? seed_offsets[i] : i, e1 = seed_offsets ? seed_offsets[i + 1] : i + 1;
        for (int e = e0; e < e1; ++e) {
            const int x = seeds_xyz[3 * e], y = seeds_xyz[3 * e + 1], z = seeds_xyz[3 * e + 2];
            if (x >= 0 && y >= 0 && z >= 0 && x < nx && y < ny && z < nz) {
                h_seeds[3 * n_in] = x; h_seeds[3 * n_in + 1] = y; h_seeds[3 * n_in + 2] = s * ctx->bank_slot_dz + z;
                ++n_in;
            }
        }
    }
    uint8_t* d_mask = (uint8_t*)ctx->d_bank_stage + seed_cap;
    if (n_in > 0) {
        CU(cudaMemcpyAsync(ctx->d_bank_stage, h_seeds, (size_t)n_in * 3 * sizeof(int), cudaMemcpyHostToDevice, stream));
    }
    CU(cudaMemcpyAsync(d_mask, h_mask, (size_t)ctx->bank_slots, cudaMemcpyHostToDevice, stream));
    // every run starts from the scene's walls: a fresh BfsHeuristic per query (seeding a wall cell
    // un-walls it for the lifetime of a BFS_3D object, bfs3d.cpp:181-187 -- not across queries here)
    unsigned int* d_count = (unsigned int*)d_seed_count;
    CU(cudaMemsetAsync(d_count, 0, sizeof(unsigned int), stream));
    bfs_walls_from_df_kernel<<<((int)ctx->bank_words + 255) / 256, 256, 0, stream>>>(
        ctx->bank, ctx->d_df, ctx->bank_kmax, ctx->bank_slot_dz, d_count, d_mask);
    ++ctx->launches;
    r = run_grid(ctx, ctx->bank, ctx->bank_words, (const int*)ctx->d_bank_stage, n_in, nullptr, d_mask, ctx->bank_slot_dz, stream,
                 d_seed_count);
    if (r) return r;
    *n_seeds_out = n_in;
    return 0;
}

// A block of the wavefront kernel takes a whole SM and waits at grid barriers, so two bank runs queued at once
// (several planner contexts share a GPU) would deal the second one's blocks onto the SMs the first one leaves to the
// expansion batches and stall there.  Asynchronous runs therefore take turns: one per device in the GPU's queue;
// the others stay staged on the host until the turn is free (checked whenever their owner polls).
static std::atomic<int> g_bank_turn[64];   // per device: 1 while an asynchronous run is queued or running

static int launch_staged_bank_run(smplgpu_ctx* ctx)
{
    // after whatever the caller queued on the main stream (e.g. the bank's creation)
    CU(cudaEventRecord(ctx->ev_bfs, ctx->stream));
    CU(cudaStreamWaitEvent(ctx->bfs_stream, ctx->ev_bfs, 0));
    int n_in = 0;
    int r = launch_bank_run(ctx, ctx->staged_slots.data(), ctx->staged_seeds.data(), ctx->staged_offsets.data(),
                            (int)ctx->staged_slots.size(), ctx->bfs_stream, ctx->d_bank_seed_count, &n_in);
    if (r) return r;
    CU(cudaEventRecord(ctx->ev_bfs, ctx->bfs_stream));
    ctx->bank_run_state = 2;
    return 0;
}

static bool take_bank_turn(smplgpu_ctx* ctx)
{
    if (bank_async_stepwise(ctx)) {
        return true;   // step-by-step runs need no co-residency: the contexts' runs simply overlap
    }
    int expected = 0;
    return g_bank_turn[ctx->device & 63].compare_exchange_strong(expected, 1);
}

// A level-by-level run whose last chunk has ended without the device raising the flag gets its next chunk.
// Returns 1 when the run is complete, 0 when more levels were queued, negative on error.
static int continue_bank_levels(smplgpu_ctx* ctx)
{
    if (ctx->bank_next_level == 0 || *ctx->bank_done != 0 || ctx->bank_next_level > ctx->bank_level_cap) {
        return 1;
    }
    const int r = launch_bank_level_chunk(ctx, ctx->bfs_stream);
    if (r) return r;
    CU(cudaEventRecord(ctx->ev_bfs, ctx->bfs_stream));
    return 0;
}

static void release_bank_turn(smplgpu_ctx* ctx)
{
    g_bank_turn[ctx->device & 63].store(0);
}

// blocks until the context's asynchronous run (if any) has finished
static int finish_bank_run(smplgpu_ctx* ctx)
{
    if (ctx->bank_run_state == 1) {
        while (!take_bank_turn(ctx)) {
            std::this_thread::yield();
        }
        const int r = launch_staged_bank_run(ctx);
        if (r) {
            ctx->bank_run_state = 0;
            release_bank_turn(ctx);
            return r;
        }
    }
    if (ctx->bank_run_state == 2) {
        for (;;) {
            const cudaError_t e = cudaEventSynchronize(ctx->ev_bfs);
            if (e != cudaSuccess) {
                ctx->bank_run_state = 0;
                release_bank_turn(ctx);
                return fail(ctx, SMPLGPU_ERR_CUDA, "bank run: %s", cudaGetErrorString(e));
            }
            const int c = continue_bank_levels(ctx);
            if (c < 0) {
                ctx->bank_run_state = 0;
                release_bank_turn(ctx);
                return c;
            }
            if (c == 1) {
                break;
            }
        }
        ctx->bank_run_state = 0;
        release_bank_turn(ctx);
    }
    return 0;
}

// seed_offsets[n + 1] non-decreasing from 0 (null: one seed per slot)
static int check_seed_offsets(smplgpu_ctx* ctx, const int32_t* seed_offsets, int n)
{
    if (!seed_offsets) return 0;
    if (seed_offsets[0] != 0) return fail(ctx, SMPLGPU_ERR_INVALID, "seed_offsets[0] is %d, not 0", seed_offsets[0]);
    for (int i = 0; i < n; ++i) {
        if (seed_offsets[i + 1] < seed_offsets[i]) return fail(ctx, SMPLGPU_ERR_INVALID, "seed_offsets decrease at %d", i + 1);
    }
    return 0;
}

static int bank_run_slots(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz, const int32_t* seed_offsets, int n)
{
    if (!ctx->has_bank) return fail(ctx, SMPLGPU_ERR_STATE, "BFS bank not created");
    if (n == 0) return 0;
    int r = check_seed_offsets(ctx, seed_offsets, n);
    if (r) return r;
    r = finish_bank_run(ctx);   // one run at a time: the staging buffers and the wavefront state are shared
    if (r) return r;
    int n_in = 0;
    r = launch_bank_run(ctx, slots, seeds_xyz, seed_offsets, n, ctx->stream, ctx->d_seed_count, &n_in);
    if (r) return r;
    CU(cudaStreamSynchronize(ctx->stream));
    return n_in;
}

int smplgpu_bfs_bank_run_slots(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz, int n)
{
    if (!ctx || n < 0 || (n > 0 && (!slots || !seeds_xyz))) return SMPLGPU_ERR_INVALID;
    return bank_run_slots(ctx, slots, seeds_xyz, nullptr, n);
}

int smplgpu_bfs_bank_run_slots_multi(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz,
                                     const int32_t* seed_offsets, int n)
{
    if (!ctx || n < 0 || (n > 0 && (!slots || !seed_offsets || (!seeds_xyz && seed_offsets[n] > 0)))) return SMPLGPU_ERR_INVALID;
    return bank_run_slots(ctx, slots, seeds_xyz, seed_offsets, n);
}

static int bank_run_slots_async(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz, const int32_t* seed_offsets,
                                int n)
{
    if (!ctx->has_bank) return fail(ctx, SMPLGPU_ERR_STATE, "BFS bank not created");
    if (ctx->bank_run_state != 0) return fail(ctx, SMPLGPU_ERR_STATE, "a bank run is already in flight");
    if (n == 0) return 0;
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= ctx->bank_slots) return fail(ctx, SMPLGPU_ERR_INVALID, "slot %d out of range", slots[i]);
    }
    const int r = check_seed_offsets(ctx, seed_offsets, n);
    if (r) return r;
    ctx->staged_slots.assign(slots, slots + n);
    if (seed_offsets) {
        ctx->staged_offsets.assign(seed_offsets, seed_offsets + n + 1);
    } else {
        ctx->staged_offsets.resize(n + 1);
        for (int i = 0; i <= n; ++i) ctx->staged_offsets[i] = i;
    }
    ctx->staged_seeds.assign(seeds_xyz, seeds_xyz + 3 * (size_t)ctx->staged_offsets[n]);
    ctx->bank_run_state = 1;
    if (take_bank_turn(ctx)) {
        const int r = launch_staged_bank_run(ctx);
        if (r) {
            ctx->bank_run_state = 0;
            release_bank_turn(ctx);
            return r;
        }
    }
    return n;
}

int smplgpu_bfs_bank_run_slots_async(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz, int n)
{
    if (!ctx || n < 0 || (n > 0 && (!slots || !seeds_xyz))) return SMPLGPU_ERR_INVALID;
    return bank_run_slots_async(ctx, slots, seeds_xyz, nullptr, n);
}

int smplgpu_bfs_bank_run_slots_multi_async(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz,
                                           const int32_t* seed_offsets, int n)
{
    if (!ctx || n < 0 || (n > 0 && (!slots || !seed_offsets || (!seeds_xyz && seed_offsets[n] > 0)))) return SMPLGPU_ERR_INVALID;
    return bank_run_slots_async(ctx, slots, seeds_xyz, seed_offsets, n);
}

int smplgpu_bfs_bank_run_done(smplgpu_ctx* ctx)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    if (ctx->bank_run_state == 0) return 1;
    if (ctx->bank_run_state == 1) {
        if (!take_bank_turn(ctx)) return 0;   // another context's run has the GPU
        const int r = launch_staged_bank_run(ctx);
        if (r) {
            ctx->bank_run_state = 0;
            release_bank_turn(ctx);
            return r;
        }
        return 0;
    }
    const cudaError_t e = cudaEventQuery(ctx->ev_bfs);
    if (e == cudaErrorNotReady) return 0;
    if (e == cudaSuccess) {
        const int c = continue_bank_levels(ctx);
        if (c == 0) return 0;        // more levels queued
        if (c < 0) {
            ctx->bank_run_state = 0;
            release_bank_turn(ctx);
            return c;
        }
    }
    ctx->bank_run_state = 0;
    release_bank_turn(ctx);
    if (e != cudaSuccess) return fail(ctx, SMPLGPU_ERR_CUDA, "bank run: %s", cudaGetErrorString(e));
    return 1;
}

int smplgpu_bfs_bank_run_wait(smplgpu_ctx* ctx)
{
    if (!ctx) return SMPLGPU_ERR_INVALID;
    return finish_bank_run(ctx);
}

int smplgpu_bfs_bank_run(smplgpu_ctx* ctx, const int32_t* seeds_xyz)
{
    if (!ctx || !seeds_xyz) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_bank) return fail(ctx, SMPLGPU_ERR_STATE, "BFS bank not created");
    std::vector<int32_t> slots(ctx->bank_slots);
    for (int s = 0; s < ctx->bank_slots; ++s) slots[s] = s;
    return smplgpu_bfs_bank_run_slots(ctx, slots.data(), seeds_xyz, ctx->bank_slots);
}

int smplgpu_bfs_bank_distances(smplgpu_ctx* ctx, const int32_t* slot, const int32_t* cells_xyz, int n, int32_t* out)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_bank) return fail(ctx, SMPLGPU_ERR_STATE, "BFS bank not created");
    if (n == 0) return 0;
    if (!slot || !cells_xyz || !out) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    for (int i = 0; i < n; ++i) {
        if (slot[i] < 0 || slot[i] >= ctx->bank_slots) return fail(ctx, SMPLGPU_ERR_INVALID, "slot %d out of range", slot[i]);
    }
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, (size_t)n * 5 * sizeof(int));
    if (r) return r;
    int* dc = (int*)ctx->d_misc;
    int* ds = dc + (size_t)n * 3;
    int* dout = ds + n;
    CU(cudaMemcpyAsync(dc, cells_xyz, (size_t)n * 3 * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ds, slot, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    bank_gather_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->bank.dist, ctx->grid.nx, ctx->grid.ny, ctx->grid.nz, ds, dc, n, dout);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dout, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

static int grow_pinned1(smplgpu_ctx* ctx, void** p, size_t* cap, size_t need)
{
    if (need <= *cap) {
        return 0;
    }
    if (*p) {
        CU(cudaFreeHost(*p));
        *p = nullptr;
        *cap = 0;
    }
    const size_t n = std::max(need + need / 2, (size_t)1 << 16);
    CU(cudaMallocHost(p, n));
    *cap = n;
    return 0;
}

static int reserve_expand(smplgpu_ctx* ctx, int b, int n)
{
    const int dof = ctx->h_model->dof;
    const size_t row = (size_t)dof * sizeof(double);
    const size_t in_bytes = 2 * n * row + (size_t)n * sizeof(int);
    const size_t in_pad = (in_bytes + 63) / 64 * 64;
    const size_t out_bytes = (size_t)n * (3 * sizeof(double) + 2 * sizeof(int) + 1);
    int r;
    if ((r = grow_pinned1(ctx, &ctx->exp_in[b], &ctx->exp_in_cap[b], in_bytes))) return r;
    if ((r = grow_pinned1(ctx, &ctx->exp_out[b], &ctx->exp_out_cap[b], out_bytes + 32))) return r;
    if ((r = grow(ctx, &ctx->d_exp[b], &ctx->d_exp_cap[b], in_pad + out_bytes + 256))) return r;
    return 0;
}

int smplgpu_expand_batch_reserve(smplgpu_ctx* ctx, int max_n)
{
    if (!ctx || max_n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set");
    for (int b = 0; b < SMPLGPU_EXPAND_BUFFERS; ++b) {
        if (ctx->exp_n[b] >= 0) return fail(ctx, SMPLGPU_ERR_STATE, "expansion buffer %d is in flight", b);
        int r = reserve_expand(ctx, b, std::max(max_n, 1));
        if (r) return r;
    }
    return ensure_unc(ctx, (size_t)std::max(max_n, 1));
}

int64_t smplgpu_expand_batch_resolved(const smplgpu_ctx* ctx)
{
    if (!ctx) return 0;
    // + the lattice rounds' running total (written by the device into page-locked memory; exact once the rounds
    // in flight have been waited for)
    return ctx->exp_resolved_total + (ctx->lat_resolved ? (int64_t)*((volatile unsigned long long*)ctx->lat_resolved) : 0);
}

int smplgpu_expand_batch_submit(smplgpu_ctx* ctx, const double* q0, const double* q1, const int32_t* slot, int n,
                                int cost_per_cell, int buffer)
{
    if (!ctx || n < 0 || buffer < 0 || buffer >= SMPLGPU_EXPAND_BUFFERS) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (!ctx->has_bank) return fail(ctx, SMPLGPU_ERR_STATE, "BFS bank not created");
    if (ctx->exp_n[buffer] >= 0) return fail(ctx, SMPLGPU_ERR_STATE, "expansion buffer %d is still in flight", buffer);
    if (n > 0 && (!q0 || !q1 || !slot)) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    for (int i = 0; i < n; ++i) {
        if (slot[i] < 0 || slot[i] >= ctx->bank_slots) return fail(ctx, SMPLGPU_ERR_INVALID, "edge %d: slot %d out of range", i, slot[i]);
    }
    if (n == 0) {
        ctx->exp_n[buffer] = 0;
        return 0;
    }
    const int b = buffer;
    const int dof = ctx->h_model->dof;
    const size_t row = (size_t)dof * sizeof(double);
    const size_t in_bytes = 2 * n * row + (size_t)n * sizeof(int);
    const size_t in_pad = (in_bytes + 63) / 64 * 64;
    const size_t out_bytes = (size_t)n * (3 * sizeof(double) + 2 * sizeof(int) + 1);
    if ((r = reserve_expand(ctx, b, n))) return r;   // no-op once smplgpu_expand_batch_reserve has sized the buffers
    uint8_t* pin = (uint8_t*)ctx->exp_in[b];
    memcpy(pin, q0, n * row);
    memcpy(pin + n * row, q1, n * row);
    memcpy(pin + 2 * n * row, slot, (size_t)n * sizeof(int));
    uint8_t* dbase = (uint8_t*)ctx->d_exp[b];
    CU(cudaMemcpyAsync(dbase, pin, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    double* dq0 = (double*)dbase;
    double* dq1 = (double*)(dbase + n * row);
    int* dslot = (int*)(dbase + 2 * n * row);
    uint8_t* obase = dbase + in_pad;
    double* doff = (double*)obase;
    int* dh = (int*)(obase + (size_t)n * 3 * sizeof(double));
    int* dg = dh + n;
    uint8_t* dv = (uint8_t*)(dg + n);
    CU(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    r = launch_edges(ctx, dq0, dq1, n, dv, nullptr);
    if (r) return r;
    expand_info_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(
        ctx->d_model, ctx->grid, ctx->bank.dist, ctx->bank.DX, ctx->bank.DY, ctx->bank_slot_dz, dq1, dslot, n,
        cost_per_cell, dh, dg, doff);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(ctx->exp_out[b], obase, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    // edges of this batch that the double-precision kernels had to resolve (behind the results, 8-byte aligned)
    CU(cudaMemcpyAsync((uint8_t*)ctx->exp_out[b] + (out_bytes + 15) / 16 * 16, ctx->d_stats + 3, sizeof(unsigned long long),
                       cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaEventRecord(ctx->ev_exp[b], ctx->stream));
    ctx->exp_n[buffer] = n;   // in flight only once everything is queued: an error above leaves the buffer free
    return 0;
}

int smplgpu_expand_batch_wait(smplgpu_ctx* ctx, int buffer, uint8_t* verdict, int32_t* h, int32_t* goal_dist_cells,
                              double* offset_xyz)
{
    if (!ctx || buffer < 0 || buffer >= SMPLGPU_EXPAND_BUFFERS) return SMPLGPU_ERR_INVALID;
    const int n = ctx->exp_n[buffer];
    if (n < 0) return fail(ctx, SMPLGPU_ERR_STATE, "expansion buffer %d has nothing in flight", buffer);
    ctx->exp_n[buffer] = -1;
    if (n == 0) return 0;
    if (!verdict || !h || !goal_dist_cells || !offset_xyz) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    CU(cudaEventSynchronize(ctx->ev_exp[buffer]));
    const uint8_t* pout = (const uint8_t*)ctx->exp_out[buffer];
    memcpy(offset_xyz, pout, (size_t)n * 3 * sizeof(double));
    memcpy(h, pout + (size_t)n * 3 * sizeof(double), (size_t)n * sizeof(int));
    memcpy(goal_dist_cells, pout + (size_t)n * (3 * sizeof(double) + sizeof(int)), (size_t)n * sizeof(int));
    memcpy(verdict, pout + (size_t)n * (3 * sizeof(double) + 2 * sizeof(int)), (size_t)n);
    const size_t out_bytes = (size_t)n * (3 * sizeof(double) + 2 * sizeof(int) + 1);
    unsigned long long resolved = 0;
    memcpy(&resolved, pout + (out_bytes + 15) / 16 * 16, sizeof(resolved));
    ctx->exp_resolved_total += (int64_t)resolved;
    return n;
}

int smplgpu_expand_batch(smplgpu_ctx* ctx, const double* q0, const double* q1, const int32_t* slot, int n,
                         int cost_per_cell, uint8_t* verdict, int32_t* h, int32_t* goal_dist_cells, double* offset_xyz)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (n == 0) return 0;
    if (!q0 || !q1 || !slot || !verdict || !h || !goal_dist_cells || !offset_xyz) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    int r = smplgpu_expand_batch_submit(ctx, q0, q1, slot, n, cost_per_cell, 0);
    if (r < 0) return r;
    r = smplgpu_expand_batch_wait(ctx, 0, verdict, h, goal_dist_cells, offset_xyz);
    return r < 0 ? r : 0;
}

///////////////////////////////////////////////////////////////////////////////
// device-resident lattices
///////////////////////////////////////////////////////////////////////////////

// the staging of smplgpu_lattice_begin_goal_sets for n queries of n_rec goal records: starts | goal records |
// slots | start distances | goal offsets | record -> query
static size_t lattice_begin_bytes(int dof, size_t n, size_t n_rec)
{
    const size_t sb = (n * sizeof(int) + 7) / 8 * 8, ob = ((n + 1) * sizeof(int) + 7) / 8 * 8;
    return n * dof * sizeof(double) + n_rec * sizeof(LatticeGoal) + 2 * sb + ob + (n_rec * sizeof(int) + 7) / 8 * 8 + 64;
}

// the slot's lattice, its goal set, and its share of the begin staging for a full goal set (reserved when the
// lattices are created, so that no query admission allocates)
static size_t lattice_bytes_per_slot(int dof, int cap, int table_size)
{
    return (size_t)cap * dof * (sizeof(double) + sizeof(int)) + (size_t)cap * sizeof(int) + (size_t)table_size * sizeof(int) +
           2 * sizeof(int) + SMPLGPU_MAX_GOAL_SET * sizeof(LatticeGoal) + lattice_begin_bytes(dof, 1, SMPLGPU_MAX_GOAL_SET);
}

static int lattice_table_size(int cap)
{
    int t = 256;
    while (t < 2 * cap) t <<= 1;
    return t;
}

int smplgpu_lattice_max_slots(smplgpu_ctx* ctx, int max_states)
{
    if (!ctx || max_states < 2) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set");
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    size_t have = free_b;
    if (ctx->has_lat) {
        have += (size_t)ctx->lat.n_slots * lattice_bytes_per_slot(ctx->h_model->dof, ctx->lat.cap, ctx->lat.table_size);
    }
    const size_t per = lattice_bytes_per_slot(ctx->h_model->dof, max_states, lattice_table_size(max_states));
    return (int)std::max<size_t>(1, std::min<size_t>((size_t)(0.4 * (double)have) / per, (size_t)1 << 20));
}

// round buffers for up to one expansion per slot (lat_max_n) of lat.stride words: every allocation happens here,
// not while planners run
static int lattice_round_buffers(smplgpu_ctx* ctx)
{
    const int dof = ctx->h_model->dof;
    const int max_n = ctx->lat_max_n;
    const size_t ne = (size_t)max_n * ctx->lat.stride;
    int r;
    for (int b = 0; b < SMPLGPU_EXPAND_BUFFERS; ++b) {
        const size_t in_bytes = 2 * (size_t)max_n * sizeof(int) + 64;
        const size_t out_bytes = (2 * ne + (size_t)max_n + 2) * sizeof(int) + 64;   // succ | h | count | resolved (8 B)
        const size_t dev_bytes = 2 * ne * dof * sizeof(double) + 2 * ((ne + 63) / 64 * 64) + 256;
        if (in_bytes > ctx->lat_in_cap[b]) {
            if (ctx->lat_in[b]) { CU(cudaFreeHost(ctx->lat_in[b])); ctx->lat_in[b] = nullptr; ctx->lat_in_cap[b] = 0; }
            CU(cudaHostAlloc(&ctx->lat_in[b], in_bytes, cudaHostAllocMapped));
            ctx->lat_in_cap[b] = in_bytes;
        }
        if (out_bytes > ctx->lat_out_cap[b]) {
            if (ctx->lat_out[b]) { CU(cudaFreeHost(ctx->lat_out[b])); ctx->lat_out[b] = nullptr; ctx->lat_out_cap[b] = 0; }
            CU(cudaHostAlloc(&ctx->lat_out[b], out_bytes, cudaHostAllocMapped));
            ctx->lat_out_cap[b] = out_bytes;
        }
        if ((r = grow(ctx, &ctx->d_lat[b], &ctx->d_lat_cap[b], dev_bytes))) return r;
    }
    if ((r = ensure_unc(ctx, ne))) return r;
    if (!ctx->lat_resolved) {
        CU(cudaHostAlloc((void**)&ctx->lat_resolved, 64, cudaHostAllocMapped));
        *ctx->lat_resolved = 0;
    }
    return 0;
}

int smplgpu_lattice_create(smplgpu_ctx* ctx, const smplgpu_lattice_params* p, int n_slots)
{
    if (!ctx || !p || n_slots <= 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (!p->resolutions || p->n_prims <= 0 || !p->deltas || !p->prim_short || p->max_states < 2)
        return fail(ctx, SMPLGPU_ERR_INVALID, "incomplete lattice parameters");
    const int dof = ctx->h_model->dof;
    r = smplgpu_set_lattice(ctx, p->resolutions, nullptr);   // discretisation (also used by the 16-bit entry points)
    if (r) return r;
    std::vector<int> long_list, short_list;
    for (int k = 0; k < p->n_prims; ++k) {
        (p->prim_short[k] ? short_list : long_list).push_back(k);
    }
    const int stride = (int)std::max(long_list.size(), p->use_short_dist ? short_list.size() : (size_t)0);
    if (stride < 1 || stride > LATTICE_MAX_STRIDE)
        return fail(ctx, SMPLGPU_ERR_LIMIT, "%d active motion primitives per expansion (limit %d)", stride, LATTICE_MAX_STRIDE);
    for (int b = 0; b < SMPLGPU_EXPAND_BUFFERS; ++b) {
        if (ctx->lat_n[b] >= 0) return fail(ctx, SMPLGPU_ERR_STATE, "lattice buffer %d is in flight", b);
    }
    CU(cudaStreamSynchronize(ctx->stream));
    const int cap = p->max_states;
    const int tsize = lattice_table_size(cap);
    const bool same_shape = ctx->has_lat && ctx->lat.n_slots == n_slots && ctx->lat.cap == cap && ctx->lat_prim_stride == stride &&
                            ctx->lat_dof == dof;
    if (!same_shape) {
        // the lattices are a scene-level allocation (gigabytes for thousands of queries): kept across calls
        free_lattice(ctx);
        LatticeBank& B = ctx->lat;
        B.n_slots = n_slots; B.cap = cap; B.table_size = tsize;
        ctx->lat_dof = dof;
        CU(cudaMalloc(&B.q, (size_t)n_slots * cap * dof * sizeof(double)));
        CU(cudaMalloc(&B.coord, (size_t)n_slots * cap * dof * sizeof(int)));
        CU(cudaMalloc(&B.gdist, (size_t)n_slots * cap * sizeof(int)));
        CU(cudaMalloc(&B.table, (size_t)n_slots * tsize * sizeof(int)));
        CU(cudaMalloc(&B.count, (size_t)n_slots * sizeof(int)));
        CU(cudaMalloc(&B.goal, (size_t)n_slots * SMPLGPU_MAX_GOAL_SET * sizeof(LatticeGoal)));
        CU(cudaMalloc(&B.n_goals, (size_t)n_slots * sizeof(int)));
        CU(cudaMemset(B.count, 0, (size_t)n_slots * sizeof(int)));
        CU(cudaMemset(B.n_goals, 0, (size_t)n_slots * sizeof(int)));
    }
    r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, lattice_begin_bytes(dof, n_slots, (size_t)n_slots * SMPLGPU_MAX_GOAL_SET));
    if (r) return r;
    LatticeBank& B = ctx->lat;
    B.stride = stride;
    ctx->lat_prim_stride = stride;
    B.snap = 0;   // smplgpu_lattice_set_snaps turns them on
    B.n_long = (int)long_list.size();
    B.n_short = (int)short_list.size();
    B.use_short_dist = p->use_short_dist ? 1 : 0;
    B.short_dist_thresh = p->short_dist_thresh;
    B.res = ctx->res;
    B.cost_per_cell = p->cost_per_cell;
    for (int a = 0; a < 3; ++a) ctx->lat_xyz_tol[a] = p->xyz_tolerance[a];
    // deltas | long list | short list
    const size_t db = (size_t)p->n_prims * dof * sizeof(double);
    const size_t lb = ((size_t)p->n_prims * sizeof(int) + 7) / 8 * 8;
    if (ctx->d_lat_aux) { CU(cudaFree(ctx->d_lat_aux)); ctx->d_lat_aux = nullptr; }
    CU(cudaMalloc(&ctx->d_lat_aux, db + 2 * lb + 64));
    uint8_t* aux = (uint8_t*)ctx->d_lat_aux;
    CU(cudaMemset(aux, 0, db + 2 * lb + 64));
    CU(cudaMemcpy(aux, p->deltas, db, cudaMemcpyHostToDevice));
    if (!long_list.empty()) CU(cudaMemcpy(aux + db, long_list.data(), long_list.size() * sizeof(int), cudaMemcpyHostToDevice));
    if (!short_list.empty()) CU(cudaMemcpy(aux + db + lb, short_list.data(), short_list.size() * sizeof(int), cudaMemcpyHostToDevice));
    B.deltas = (const double*)aux;
    B.long_list = (const int*)(aux + db);
    B.short_list = (const int*)(aux + db + lb);
    ctx->lat_params = ctx->lattice;
    for (int v = 0; v < MAX_DOF; ++v) ctx->lat_vals.v[v] = ctx->lattice_vals[v];
    ctx->lat_max_n = n_slots;
    if ((r = lattice_round_buffers(ctx))) return r;
    // SMPLGPU_LATTICE_FUSED=1: one kernel per round (lattice_round_kernel; measured slower at the default number of
    // planner contexts, see lattice.cuh) when the single-precision model is in use and a block's shared memory holds
    // the blob, the per-thread f32 state and one warp's double-precision slots
    {
        static const bool want = [] {
            const char* e = getenv("SMPLGPU_LATTICE_FUSED");
            return e != nullptr && atoi(e) != 0;
        }();
        const size_t smem = (size_t)ctx->blob_words * 4
                            + ((size_t)ctx->v32_slots * 12 + (size_t)ctx->v32_ptrees * 3) * sizeof(float) * LROUND_THREADS
                            + (size_t)ctx->h_model->n_slots * 12 * sizeof(double) * 32 + 64;
        ctx->lat_fused = want && use_f32(ctx) && smem <= (size_t)200 * 1024;
        ctx->lat_round_smem = smem;
        if (ctx->lat_fused) {
            CU(raise_smem_cap(lattice_round_kernel, (int)std::max(smem, (size_t)1024)));
        }
    }
    ctx->has_lat = true;
    return stride;
}

// Quaterniond(AngleAxisd(yaw, Z) * AngleAxisd(pitch, Y) * AngleAxisd(roll, X)), x y z w: the operation order of the
// oracle's Eigen stand-in (oracle/goals/goal_lattice.cpp quatFromRpy), with the host's libm
static void quat_from_rpy(double roll, double pitch, double yaw, double* q)
{
    const double hz = 0.5 * yaw, hy = 0.5 * pitch, hx = 0.5 * roll;
    const double sz = std::sin(hz), sy = std::sin(hy), sx = std::sin(hx);
    const double a[4] = { sz * 0.0, sz * 0.0, sz * 1.0, std::cos(hz) };
    const double b[4] = { sy * 0.0, sy * 1.0, sy * 0.0, std::cos(hy) };
    const double c[4] = { sx * 1.0, sx * 0.0, sx * 0.0, std::cos(hx) };
    auto mul = [](const double* l, const double* r, double* o) {   // Eigen's generic quat_product
        o[3] = l[3] * r[3] - l[0] * r[0] - l[1] * r[1] - l[2] * r[2];
        o[0] = l[3] * r[0] + l[0] * r[3] + l[1] * r[2] - l[2] * r[1];
        o[1] = l[3] * r[1] + l[1] * r[3] + l[2] * r[0] - l[0] * r[2];
        o[2] = l[3] * r[2] + l[2] * r[3] + l[0] * r[1] - l[1] * r[0];
    };
    double ab[4];
    mul(a, b, ab);
    mul(ab, c, q);
}

static bool bad_tolerance(double t)
{
    return std::isnan(t) || t < 0.0;
}

// KDL Rotation::RPY(roll, pitch, yaw) = Rz(yaw) Ry(pitch) Rx(roll), row-major: the IK's goal rotation, with the host's
// libm and the expression of the oracle (oracle/snap/snap_lattice.cpp rpyMatrix)
static void rpy_matrix(double roll, double pitch, double yaw, double* R)
{
    const double ca1 = std::cos(yaw), sa1 = std::sin(yaw);
    const double cb1 = std::cos(pitch), sb1 = std::sin(pitch);
    const double cc1 = std::cos(roll), sc1 = std::sin(roll);
    R[0] = ca1 * cb1;  R[1] = ca1 * sb1 * sc1 - sa1 * cc1;  R[2] = ca1 * sb1 * cc1 + sa1 * sc1;
    R[3] = sa1 * cb1;  R[4] = sa1 * sb1 * sc1 + ca1 * cc1;  R[5] = sa1 * sb1 * cc1 - ca1 * sc1;
    R[6] = -sb1;       R[7] = cb1 * sc1;                    R[8] = cb1 * cc1;
}

// goals[goal_offsets[k] .. goal_offsets[k + 1] - 1] = the goal set of query k (offsets checked by the caller)
static int lattice_begin_records(smplgpu_ctx* ctx, const int32_t* slots, const double* starts, const int32_t* start_gd,
                                 const std::vector<LatticeGoal>& goals, const int32_t* goal_offsets, int n)
{
    const int dof = ctx->h_model->dof;
    const size_t n_rec = goals.size();
    const size_t sb = ((size_t)n * sizeof(int) + 7) / 8 * 8, ob = ((size_t)(n + 1) * sizeof(int) + 7) / 8 * 8,
                 qb = (size_t)n * dof * sizeof(double), gb = n_rec * sizeof(LatticeGoal);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, lattice_begin_bytes(dof, n, n_rec));   // reserved by smplgpu_lattice_create
    if (r) return r;
    std::vector<int32_t> goal_set(n_rec);
    for (int k = 0; k < n; ++k) {
        std::fill(goal_set.begin() + goal_offsets[k], goal_set.begin() + goal_offsets[k + 1], k);
    }
    uint8_t* base = (uint8_t*)ctx->d_misc;
    double* d_starts = (double*)base;
    LatticeGoal* d_goals = (LatticeGoal*)(base + qb);
    int* d_slots = (int*)(base + qb + gb);
    int* d_gd = (int*)(base + qb + gb + sb);
    int* d_offsets = (int*)(base + qb + gb + 2 * sb);
    int* d_goal_set = (int*)(base + qb + gb + 2 * sb + ob);
    CU(cudaMemcpyAsync(d_starts, starts, qb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_goals, goals.data(), gb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_slots, slots, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_gd, start_gd, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_offsets, goal_offsets, (size_t)(n + 1) * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_goal_set, goal_set.data(), n_rec * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    const size_t total = (size_t)n * ctx->lat.table_size;
    const int threads = (int)std::max<size_t>((size_t)n, n_rec);
    lattice_clear_kernel<<<(unsigned)std::min<size_t>((total + 255) / 256, (size_t)ctx->sm_count * 16), 256, 0, ctx->stream>>>(ctx->lat, d_slots, n);
    lattice_begin_kernel<<<(threads + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_model, ctx->lat, ctx->lat_params, ctx->lat_vals,
                                                                        d_slots, d_starts, d_gd, d_goals, d_goal_set,
                                                                        d_offsets, n, (int)n_rec);
    ctx->launches += 2;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));   // the inputs may be pageable
    return 0;
}

static int lattice_begin_check(smplgpu_ctx* ctx, const int32_t* slots, const double* starts, const int32_t* start_gd,
                               const void* goals, int n)
{
    if (!ctx->has_lat) return fail(ctx, SMPLGPU_ERR_STATE, "lattices not created (smplgpu_lattice_create)");
    if (n == 0) return 0;
    if (!slots || !starts || !start_gd || !goals) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= ctx->lat.n_slots) return fail(ctx, SMPLGPU_ERR_INVALID, "slot %d out of range", slots[i]);
    }
    return 0;
}

int smplgpu_lattice_begin(smplgpu_ctx* ctx, const int32_t* slots, const double* starts, const int32_t* start_gd,
                          const double* goals_xyz, int n)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = lattice_begin_check(ctx, slots, starts, start_gd, goals_xyz, n);
    if (r || n == 0) return r;
    std::vector<LatticeGoal> recs(n);   // zero-filled
    for (int i = 0; i < n; ++i) {
        LatticeGoal& g = recs[i];
        g.type = SMPLGPU_GOAL_XYZ;
        for (int a = 0; a < 3; ++a) {
            g.xyz[a] = goals_xyz[3 * i + a];
            g.xyz_tol[a] = ctx->lat_xyz_tol[a];
        }
        rpy_matrix(0.0, 0.0, 0.0, g.R);
    }
    std::vector<int32_t> offsets(n + 1);
    for (int i = 0; i <= n; ++i) offsets[i] = i;
    return lattice_begin_records(ctx, slots, starts, start_gd, recs, offsets.data(), n);
}

int smplgpu_lattice_begin_goals(smplgpu_ctx* ctx, const int32_t* slots, const double* starts, const int32_t* start_gd,
                                const smplgpu_goal* goals, int n)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    std::vector<int32_t> offsets(n + 1);
    for (int i = 0; i <= n; ++i) offsets[i] = i;
    return smplgpu_lattice_begin_goal_sets(ctx, slots, starts, start_gd, goals, offsets.data(), n);
}

int smplgpu_lattice_begin_goal_sets(smplgpu_ctx* ctx, const int32_t* slots, const double* starts, const int32_t* start_gd,
                                    const smplgpu_goal* goals, const int32_t* goal_offsets, int n)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = lattice_begin_check(ctx, slots, starts, start_gd, goals, n);
    if (r || n == 0) return r;
    if (!goal_offsets) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    if (goal_offsets[0] != 0) return fail(ctx, SMPLGPU_ERR_INVALID, "goal_offsets[0] is %d, not 0", goal_offsets[0]);
    for (int k = 0; k < n; ++k) {
        const long long m = (long long)goal_offsets[k + 1] - goal_offsets[k];
        if (m < 1 || m > SMPLGPU_MAX_GOAL_SET)
            return fail(ctx, SMPLGPU_ERR_INVALID, "query %d: goal set of %lld records (1 to %d)", k, m, SMPLGPU_MAX_GOAL_SET);
    }
    const int dof = ctx->h_model->dof;
    std::vector<LatticeGoal> recs(goal_offsets[n]);   // zero-filled
    for (int i = 0; i < goal_offsets[n]; ++i) {
        const smplgpu_goal& in = goals[i];
        LatticeGoal& g = recs[i];
        g.type = in.type;
        if (in.type == SMPLGPU_GOAL_XYZ || in.type == SMPLGPU_GOAL_XYZ_RPY) {
            for (int a = 0; a < 3; ++a) {
                if (bad_tolerance(in.xyz_tolerance[a])) return fail(ctx, SMPLGPU_ERR_INVALID, "goal %d: xyz tolerance %d is NaN or negative", i, a);
                g.xyz[a] = in.pose[a];
                g.xyz_tol[a] = in.xyz_tolerance[a];
            }
            rpy_matrix(in.pose[3], in.pose[4], in.pose[5], g.R);   // the snap's IK target: the full pose of the record
            if (in.type == SMPLGPU_GOAL_XYZ_RPY) {
                if (bad_tolerance(in.rpy_tolerance)) return fail(ctx, SMPLGPU_ERR_INVALID, "goal %d: rpy tolerance is NaN or negative", i);
                g.rpy_tol = in.rpy_tolerance;
                quat_from_rpy(in.pose[3], in.pose[4], in.pose[5], g.qg);
            }
        } else if (in.type == SMPLGPU_GOAL_JOINT_STATE) {
            for (int v = 0; v < dof; ++v) {
                if (bad_tolerance(in.angle_tolerances[v])) return fail(ctx, SMPLGPU_ERR_INVALID, "goal %d: angle tolerance %d is NaN or negative", i, v);
                g.angles[v] = in.angles[v];
                g.angle_tol[v] = in.angle_tolerances[v];
            }
        } else {
            return fail(ctx, SMPLGPU_ERR_INVALID, "goal %d: unknown goal type %d", i, in.type);
        }
    }
    return lattice_begin_records(ctx, slots, starts, start_gd, recs, goal_offsets, n);
}

int smplgpu_lattice_expand_submit(smplgpu_ctx* ctx, const int32_t* slot, const int32_t* parent_id, int n, int buffer)
{
    if (!ctx || n < 0 || buffer < 0 || buffer >= SMPLGPU_EXPAND_BUFFERS) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_lat) return fail(ctx, SMPLGPU_ERR_STATE, "lattices not created (smplgpu_lattice_create)");
    if (!ctx->has_bank) return fail(ctx, SMPLGPU_ERR_STATE, "BFS bank not created");
    if (ctx->lat.n_slots > ctx->bank_slots) return fail(ctx, SMPLGPU_ERR_STATE, "more lattices than BFS bank slots");
    if (ctx->lat_n[buffer] >= 0) return fail(ctx, SMPLGPU_ERR_STATE, "lattice buffer %d is still in flight", buffer);
    if (n > ctx->lat_max_n) return fail(ctx, SMPLGPU_ERR_LIMIT, "%d expansions in a round, room for %d", n, ctx->lat_max_n);
    if (n > 0 && (!slot || !parent_id)) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    if (n == 0) {
        ctx->lat_n[buffer] = 0;
        return 0;
    }
    const int b = buffer;
    const int dof = ctx->h_model->dof;
    const LatticeBank& B = ctx->lat;
    int* in_slot = (int*)ctx->lat_in[b];
    int* in_parent = in_slot + n;
    for (int i = 0; i < n; ++i) {
        if (slot[i] < 0 || slot[i] >= B.n_slots) return fail(ctx, SMPLGPU_ERR_INVALID, "expansion %d: slot %d out of range", i, slot[i]);
        if (parent_id[i] < 1 || parent_id[i] >= B.cap) return fail(ctx, SMPLGPU_ERR_INVALID, "expansion %d: state id %d out of range", i, parent_id[i]);
        in_slot[i] = slot[i];
        in_parent[i] = parent_id[i];
    }
    const size_t ne = (size_t)n * B.stride;
    const size_t nep = (ne + 63) / 64 * 64;
    uint8_t* dbase = (uint8_t*)ctx->d_lat[b];
    double* dq0 = (double*)dbase;
    double* dq1 = dq0 + ne * dof;
    uint8_t* dactive = (uint8_t*)(dq1 + ne * dof);
    uint8_t* dverdict = dactive + nep;
    int* out_succ = (int*)ctx->lat_out[b];
    int* out_h = out_succ + ne;
    int* out_count = out_h + ne;
    // the kernels read the (slot, state id) pairs from, and write the results to, page-locked host memory directly
    if (ctx->lat_fused && !B.snap) {
        lattice_round_kernel<<<n, LROUND_THREADS, ctx->lat_round_smem, ctx->stream>>>(
            ctx->d_blob, ctx->blob_words, ctx->d_model, ctx->d_df, ctx->grid32, ctx->grid, B, ctx->lat_params, ctx->lat_vals,
            ctx->bank.dist, ctx->bank.DX, ctx->bank.DY, ctx->bank_slot_dz, in_slot, in_parent, n, out_succ, out_h, out_count,
            ctx->lat_resolved);
        ++ctx->launches;
        CU(cudaGetLastError());
        CU(cudaEventRecord(ctx->ev_exp[b], ctx->stream));
        ctx->lat_n[buffer] = n;
        return 0;
    }
    lattice_gen_kernel<<<(unsigned)((ne + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_model, B, in_slot, in_parent, n, dq0, dq1, dactive,
                                                                              ctx->d_stats);
    ++ctx->launches;
    if (B.snap) {
        lattice_snap_kernel<<<(unsigned)(((size_t)n * B.snap + IK_WARPS - 1) / IK_WARPS), 32 * IK_WARPS, 0, ctx->stream>>>(
            ctx->d_model, B, in_slot, in_parent, n, dq1, dactive, ctx->d_snap_counters);
        ++ctx->launches;
    }
    int r = launch_edges(ctx, dq0, dq1, (int)ne, dverdict, nullptr);
    if (r) return r;
    lattice_commit_kernel<<<(unsigned)((n * 32 + 127) / 128), 128, 0, ctx->stream>>>(
        ctx->d_model, ctx->grid, B, ctx->lat_params, ctx->lat_vals, ctx->bank.dist, ctx->bank.DX, ctx->bank.DY, ctx->bank_slot_dz,
        in_slot, in_parent, n, dq1, dactive, dverdict, out_succ, out_h, out_count, ctx->d_stats, ctx->lat_resolved);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->ev_exp[b], ctx->stream));
    ctx->lat_n[buffer] = n;
    return 0;
}

int smplgpu_lattice_expand_wait(smplgpu_ctx* ctx, int buffer, const int32_t** succ, const int32_t** h, const int32_t** count)
{
    if (!ctx || buffer < 0 || buffer >= SMPLGPU_EXPAND_BUFFERS) return SMPLGPU_ERR_INVALID;
    const int n = ctx->lat_n[buffer];
    if (n < 0) return fail(ctx, SMPLGPU_ERR_STATE, "lattice buffer %d has nothing in flight", buffer);
    ctx->lat_n[buffer] = -1;
    if (n == 0) return 0;
    if (!succ || !h || !count) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    CU(cudaEventSynchronize(ctx->ev_exp[buffer]));
    const size_t ne = (size_t)n * ctx->lat.stride;
    const int* out = (const int*)ctx->lat_out[buffer];
    *succ = out;
    *h = out + ne;
    *count = out + 2 * ne;
    for (int i = 0; i < n; ++i) {
        if ((*count)[i] < 0) return fail(ctx, SMPLGPU_ERR_LIMIT, "a lattice ran out of room (%d states per query)", ctx->lat.cap);
    }
    return n;
}

int smplgpu_lattice_states(smplgpu_ctx* ctx, const int32_t* slot, const int32_t* id, int n, double* q_out)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_lat) return fail(ctx, SMPLGPU_ERR_STATE, "lattices not created");
    if (n == 0) return 0;
    if (!slot || !id || !q_out) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    for (int i = 0; i < n; ++i) {
        if (slot[i] < 0 || slot[i] >= ctx->lat.n_slots || id[i] < 0 || id[i] >= ctx->lat.cap)
            return fail(ctx, SMPLGPU_ERR_INVALID, "state %d: (slot %d, id %d) out of range", i, slot[i], id[i]);
    }
    const int dof = ctx->h_model->dof;
    const size_t ib = ((size_t)n * sizeof(int) + 7) / 8 * 8, ob = (size_t)n * dof * sizeof(double);
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, 2 * ib + ob + 64);
    if (r) return r;
    uint8_t* base = (uint8_t*)ctx->d_misc;
    double* d_out = (double*)base;
    int* d_slot = (int*)(base + ob);
    int* d_id = (int*)(base + ob + ib);
    CU(cudaMemcpyAsync(d_slot, slot, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_id, id, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    lattice_gather_kernel<<<(n * dof + 127) / 128, 128, 0, ctx->stream>>>(ctx->lat, dof, d_slot, d_id, n, d_out);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(q_out, d_out, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

///////////////////////////////////////////////////////////////////////////////
// planning-link IK and the snap action
///////////////////////////////////////////////////////////////////////////////

static bool bad_ik_params(const smplgpu_ik_params* p)
{
    return p->max_iterations < 1 || !(p->tolerance > 0.0);
}

// the batched IK of smplgpu_planning_link_ik (width 6: x y z roll pitch yaw) and smplgpu_planning_link_ik_position
// (width 3: x y z); ROWS = the width
static int planning_link_ik(smplgpu_ctx* ctx, int ROWS, const double* targets, const double* seeds, int n,
                            const smplgpu_ik_params* params, double* q_out, uint8_t* ok, int32_t* iterations)
{
    if (!ctx || n < 0 || !params) return SMPLGPU_ERR_INVALID;
    if (bad_ik_params(params)) return fail(ctx, SMPLGPU_ERR_INVALID, "IK: max_iterations < 1, or a tolerance that is not positive");
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set (smplgpu_set_robot)");
    if (n == 0) return 0;
    if (!targets || !seeds || !q_out || !ok || !iterations) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const int dof = ctx->h_model->dof;
    std::vector<IkTarget> tg(n);   // zero-filled: the position-only IK reads no rotation
    for (int k = 0; k < n; ++k) {
        const double* P = targets + (size_t)ROWS * k;
        for (int a = 0; a < 3; ++a) tg[k].p[a] = P[a];
        if (ROWS == 6) rpy_matrix(P[3], P[4], P[5], tg[k].R);
    }
    const size_t tb = (size_t)n * sizeof(IkTarget), qb = (size_t)n * dof * sizeof(double);
    const size_t ib = ((size_t)n * sizeof(int) + 7) / 8 * 8, ob = ((size_t)n + 7) / 8 * 8;
    int r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, tb + 2 * qb + ib + ob + 64);
    if (r) return r;
    uint8_t* base = (uint8_t*)ctx->d_misc;
    IkTarget* d_tg = (IkTarget*)base;
    double* d_seeds = (double*)(base + tb);
    double* d_q = (double*)(base + tb + qb);
    int* d_it = (int*)(base + tb + 2 * qb);
    uint8_t* d_ok = base + tb + 2 * qb + ib;
    CU(cudaMemcpyAsync(d_tg, tg.data(), tb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_seeds, seeds, qb, cudaMemcpyHostToDevice, ctx->stream));
    auto* kernel = ROWS == 6 ? planning_link_ik_kernel<6> : planning_link_ik_kernel<3>;
    kernel<<<(unsigned)((n + IK_WARPS - 1) / IK_WARPS), 32 * IK_WARPS, 0, ctx->stream>>>(
        ctx->d_model, d_tg, d_seeds, n, params->max_iterations, params->tolerance, d_q, d_ok, d_it);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(q_out, d_q, qb, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(ok, d_ok, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(iterations, d_it, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    int n_ok = 0;
    for (int k = 0; k < n; ++k) n_ok += ok[k] ? 1 : 0;
    return n_ok;
}

int smplgpu_planning_link_ik(smplgpu_ctx* ctx, const double* pose6, const double* seeds, int n,
                             const smplgpu_ik_params* params, double* q_out, uint8_t* ok, int32_t* iterations)
{
    return planning_link_ik(ctx, 6, pose6, seeds, n, params, q_out, ok, iterations);
}

int smplgpu_planning_link_ik_position(smplgpu_ctx* ctx, const double* xyz, const double* seeds, int n,
                                      const smplgpu_ik_params* params, double* q_out, uint8_t* ok, int32_t* iterations)
{
    return planning_link_ik(ctx, 3, xyz, seeds, n, params, q_out, ok, iterations);
}

// The Euclidean-space motions of the path shortcut (euclid.cuh).  All step counts in one launch and one copy back;
// then the motions in order, packed into chunks of at most SMPLGPU_EUCLID_CHUNK_EDGES waypoint edges: per chunk the
// IK chains (a warp each), the chunk's edges through launch_edges, and the AND of each motion's verdicts.
int smplgpu_euclid_motions(smplgpu_ctx* ctx, const double* points, int n_points, const int32_t* idx_a,
                           const int32_t* idx_b, int n, const smplgpu_euclid_params* params, uint8_t* ok, double* cost,
                           int32_t* n_steps, const int64_t* state_offsets, double* states, int64_t counters[2])
{
    if (!ctx || n < 0 || n_points < 0 || !params) return SMPLGPU_ERR_INVALID;
    if (!(params->max_step_m > 0.0) || !std::isfinite(params->max_step_m) || !(params->max_step_rad > 0.0) ||
        !std::isfinite(params->max_step_rad) || params->max_steps < 1 || params->max_steps > SMPLGPU_EUCLID_MAX_STEPS ||
        bad_ik_params(&params->ik) || !std::isfinite(params->ik.tolerance))
        return fail(ctx, SMPLGPU_ERR_INVALID, "euclid_motions: step bounds must be positive and finite, max_steps in 1 .. %d, "
                    "IK max_iterations >= 1 and a positive finite tolerance", SMPLGPU_EUCLID_MAX_STEPS);
    int r = need_scene(ctx);
    if (r) return r;
    if (counters) counters[0] = counters[1] = 0;
    if (n == 0) return 0;
    if (!points || !idx_a || !idx_b || !ok || !cost || !n_steps || (states && !state_offsets))
        return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    for (int e = 0; e < n; ++e) {
        if (idx_a[e] < 0 || idx_a[e] >= n_points || idx_b[e] < 0 || idx_b[e] >= n_points)
            return fail(ctx, SMPLGPU_ERR_INVALID, "motion %d: point index out of range", e);
        if (states && state_offsets[e] < 0)
            return fail(ctx, SMPLGPU_ERR_INVALID, "motion %d: negative state offset", e);
    }
    const int dof = ctx->h_model->dof;
    const EuclidParams P{ params->max_step_m, params->max_step_rad, params->max_steps, params->ik.max_iterations,
                          params->ik.tolerance };
    // resident for the whole call: points | idx_a | idx_b | steps | edge offsets | cost | chain_ok | ok | counters
    auto up = [](size_t b) { return (b + 255) / 256 * 256; };
    const size_t pb = up((size_t)n_points * dof * sizeof(double)), ib = up((size_t)n * sizeof(int));
    const size_t cb = up((size_t)n * sizeof(double)), vb = up((size_t)n);
    r = grow(ctx, &ctx->d_misc, &ctx->misc_cap, pb + 4 * ib + cb + 2 * vb + 256);
    if (r) return r;
    uint8_t* base = (uint8_t*)ctx->d_misc;
    double* d_points = (double*)base;
    int* d_a = (int*)(base + pb);
    int* d_b = (int*)(base + pb + ib);
    int* d_steps = (int*)(base + pb + 2 * ib);
    int* d_off = (int*)(base + pb + 3 * ib);
    double* d_cost = (double*)(base + pb + 4 * ib);
    uint8_t* d_chain = base + pb + 4 * ib + cb;
    uint8_t* d_ok = d_chain + vb;
    unsigned long long* d_ctr = (unsigned long long*)(d_ok + vb);
    CU(cudaMemsetAsync(d_ctr, 0, 2 * sizeof(unsigned long long), ctx->stream));
    CU(cudaMemcpyAsync(d_points, points, (size_t)n_points * dof * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_a, idx_a, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_b, idx_b, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    euclid_steps_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_model, d_points, d_a, d_b, n, P, d_steps);
    ++ctx->launches;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(n_steps, d_steps, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));

    // chunks: consecutive motions while their edges fit (a refused motion has none)
    std::vector<int> off(n), chunk_begin(1, 0), chunk_edges;
    int fill = 0, max_fill = 0;
    for (int e = 0; e < n; ++e) {
        const int ne = n_steps[e] <= P.max_steps ? n_steps[e] : 0;
        if (fill + ne > SMPLGPU_EUCLID_CHUNK_EDGES) {
            chunk_begin.push_back(e);
            chunk_edges.push_back(fill);
            fill = 0;
        }
        off[e] = fill;
        fill += ne;
        max_fill = std::max(max_fill, fill);
    }
    chunk_begin.push_back(n);
    chunk_edges.push_back(fill);
    CU(cudaMemcpyAsync(d_off, off.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    r = ensure_state_buffers(ctx, (size_t)std::max(max_fill, 1), dof, true);
    if (r) return r;
    CU(cudaMemsetAsync(ctx->d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    std::vector<double> h_q1;
    std::vector<uint8_t> h_chain;
    for (size_t c = 0; c + 1 < chunk_begin.size(); ++c) {
        const int first = chunk_begin[c], count = chunk_begin[c + 1] - first, edges = chunk_edges[c];
        euclid_chain_kernel<<<(unsigned)((count + IK_WARPS - 1) / IK_WARPS), 32 * IK_WARPS, 0, ctx->stream>>>(
            ctx->d_model, d_points, d_a, d_b, first, count, P, d_off, ctx->d_q0, ctx->d_q1, d_chain, d_cost, d_ctr);
        ++ctx->launches;
        CU(cudaGetLastError());
        if (edges > 0) {
            r = launch_edges(ctx, ctx->d_q0, ctx->d_q1, edges, ctx->d_verdict, nullptr);
            if (r) return r;
        }
        euclid_reduce_kernel<<<(count + 127) / 128, 128, 0, ctx->stream>>>(first, count, P.max_steps, d_steps, d_off,
                                                                             d_chain, ctx->d_verdict, d_ok);
        ++ctx->launches;
        CU(cudaGetLastError());
        if (states) {
            // the interior states of the completed chains: state k of motion e is the end of its edge k - 1
            h_q1.resize((size_t)edges * dof);
            h_chain.resize((size_t)count);
            CU(cudaMemcpyAsync(h_q1.data(), ctx->d_q1, h_q1.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaMemcpyAsync(h_chain.data(), d_chain + first, (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
            for (int e = first; e < first + count; ++e) {
                if (h_chain[e - first] && n_steps[e] > 1) {
                    std::memcpy(states + (size_t)state_offsets[e] * dof, h_q1.data() + (size_t)off[e] * dof,
                                (size_t)(n_steps[e] - 1) * dof * sizeof(double));
                }
            }
        }
    }
    CU(cudaMemcpyAsync(ok, d_ok, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(cost, d_cost, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    unsigned long long ctr[2];
    CU(cudaMemcpyAsync(ctr, d_ctr, sizeof(ctr), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (counters) {
        counters[0] = (int64_t)ctr[0];
        counters[1] = (int64_t)ctr[1];
    }
    return 0;
}

int smplgpu_lattice_set_snap(smplgpu_ctx* ctx, const smplgpu_snap_params* p)
{
    if (!ctx || !p) return SMPLGPU_ERR_INVALID;
    smplgpu_snap_kinds k = {};
    k.enabled[SMPLGPU_SNAP_XYZ_RPY] = p->enabled;
    k.dist_thresh[SMPLGPU_SNAP_XYZ_RPY] = p->dist_thresh;
    k.ik = p->ik;
    return smplgpu_lattice_set_snaps(ctx, &k);
}

int smplgpu_lattice_set_snaps(smplgpu_ctx* ctx, const smplgpu_snap_kinds* p)
{
    if (!ctx || !p) return SMPLGPU_ERR_INVALID;
    for (int k = 0; k < 3; ++k) {
        if (std::isnan(p->dist_thresh[k]) || p->dist_thresh[k] < 0.0)
            return fail(ctx, SMPLGPU_ERR_INVALID, "snap kind %d: threshold is NaN or negative", k);
    }
    if (bad_ik_params(&p->ik)) return fail(ctx, SMPLGPU_ERR_INVALID, "IK: max_iterations < 1, or a tolerance that is not positive");
    if (!ctx->has_lat) return fail(ctx, SMPLGPU_ERR_STATE, "lattices not created (smplgpu_lattice_create)");
    for (int b = 0; b < SMPLGPU_EXPAND_BUFFERS; ++b) {
        if (ctx->lat_n[b] >= 0) return fail(ctx, SMPLGPU_ERR_STATE, "lattice buffer %d is in flight", b);
    }
    int snap = 0, kind_of_word[3] = { 0, 0, 0 };
    for (int k = 0; k < 3; ++k) {
        if (p->enabled[k]) kind_of_word[snap++] = k;
    }
    const int stride = ctx->lat_prim_stride + snap;
    if (stride > LATTICE_MAX_STRIDE)
        return fail(ctx, SMPLGPU_ERR_LIMIT, "%d successors per expansion with %d snap kinds (limit %d)", stride, snap, LATTICE_MAX_STRIDE);
    if (snap && !ctx->d_snap_counters) {
        CU(cudaMalloc(&ctx->d_snap_counters, 6 * sizeof(unsigned long long)));
        CU(cudaMemset(ctx->d_snap_counters, 0, 6 * sizeof(unsigned long long)));
    }
    CU(cudaStreamSynchronize(ctx->stream));
    LatticeBank& B = ctx->lat;
    B.snap = snap;
    B.stride = stride;
    for (int k = 0; k < 3; ++k) {
        B.snap_kind[k] = kind_of_word[k];
        B.snap_thresh[k] = p->dist_thresh[k];
    }
    B.ik_max_iterations = p->ik.max_iterations;
    B.ik_tolerance = p->ik.tolerance;
    const int r = lattice_round_buffers(ctx);
    return r ? r : stride;
}

int smplgpu_lattice_snap_counters_by_kind(smplgpu_ctx* ctx, int64_t counters[6])
{
    if (!ctx || !counters) return SMPLGPU_ERR_INVALID;
    for (int k = 0; k < 6; ++k) counters[k] = 0;
    if (!ctx->d_snap_counters) return 0;
    unsigned long long c[6];
    CU(cudaMemcpyAsync(c, ctx->d_snap_counters, sizeof(c), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 6; ++k) counters[k] = (int64_t)c[k];
    return 0;
}

int smplgpu_lattice_snap_counters(smplgpu_ctx* ctx, int64_t counters[2])
{
    if (!ctx || !counters) return SMPLGPU_ERR_INVALID;
    int64_t c[6];
    const int r = smplgpu_lattice_snap_counters_by_kind(ctx, c);
    if (r) return r;
    counters[0] = c[0] + c[2] + c[4];
    counters[1] = c[1] + c[3] + c[5];
    return 0;
}
///////////////////////////////////////////////////////////////////////////////
// lattice states: 16-bit coordinates on the wire
///////////////////////////////////////////////////////////////////////////////

int smplgpu_set_lattice(smplgpu_ctx* ctx, const double* resolutions, int32_t* coord_vals)
{
    if (!ctx || !resolutions) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set (smplgpu_set_robot)");
    const DevModel& m = *ctx->h_model;
    ctx->has_lattice = false;
    for (int v = 0; v < m.dof; ++v) {
        const double res = resolutions[v];
        if (!(res > 0.0)) return fail(ctx, SMPLGPU_ERR_INVALID, "resolution of variable %d is not positive", v);
        int vals;
        double delta;
        if (m.var_type[v] == SMPLGPU_VAR_CONTINUOUS) {          // manip_lattice.cpp:127-129
            vals = (int)std::round((2.0 * M_PI) / res);
            delta = (2.0 * M_PI) / (double)vals;
            ctx->lattice.bounded[v] = 0;
            ctx->lattice.base[v] = 0.0;
        } else {                                                 // :130-133 (every KDL planning variable has limits)
            const double span = std::fabs(m.var_max[v] - m.var_min[v]);
            vals = std::max(1, (int)std::round(span / res));
            delta = span / (double)vals;
            ctx->lattice.bounded[v] = 1;
            ctx->lattice.base[v] = m.var_min[v];
        }
        if (vals > 32767) return fail(ctx, SMPLGPU_ERR_LIMIT, "variable %d has %d lattice values: more than 16-bit coordinates hold", v, vals);
        ctx->lattice.delta[v] = delta;
        ctx->lattice_vals[v] = vals;
        if (coord_vals) coord_vals[v] = vals;
    }
    ctx->has_lattice = true;
    return 0;
}

int smplgpu_is_lattice_states_valid(smplgpu_ctx* ctx, const int16_t* coords, int n, uint8_t* verdict)
{
    if (!ctx || n < 0) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (!ctx->has_lattice) return fail(ctx, SMPLGPU_ERR_STATE, "lattice resolutions not set (smplgpu_set_lattice)");
    if (n == 0) return 0;
    if (!coords || !verdict) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    return run_host_batched(ctx, nullptr, nullptr, n, verdict, nullptr, nullptr, nullptr, 0, coords, nullptr, false);
}

int smplgpu_is_lattice_edges_valid(smplgpu_ctx* ctx, const int16_t* parent_coords, const uint8_t* prim_id, int n,
                                   const double* deltas, int n_prims, uint8_t* verdict, int32_t* waypoint_counts)
{
    if (!ctx || n < 0 || n_prims < 0 || n_prims > 255) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (!ctx->has_lattice) return fail(ctx, SMPLGPU_ERR_STATE, "lattice resolutions not set (smplgpu_set_lattice)");
    if (n == 0) return 0;
    if (!parent_coords || !prim_id || !verdict || (n_prims > 0 && !deltas)) return fail(ctx, SMPLGPU_ERR_INVALID, "null pointer");
    const size_t bytes = (size_t)std::max(1, n_prims) * ctx->h_model->dof * sizeof(double);
    r = grow(ctx, (void**)&ctx->d_deltas, &ctx->deltas_cap, bytes);
    if (r) return r;
    if (n_prims > 0) {
        CU(cudaMemcpyAsync(ctx->d_deltas, deltas, (size_t)n_prims * ctx->h_model->dof * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    return run_host_batched(ctx, nullptr, nullptr, n, verdict, waypoint_counts, nullptr, ctx->d_deltas, n_prims, parent_coords,
                            prim_id, true);
}

///////////////////////////////////////////////////////////////////////////////
// one expansion at a time (unchanged callers)
///////////////////////////////////////////////////////////////////////////////

int smplgpu_set_motion_primitives(smplgpu_ctx* ctx, const double* deltas, int n_prims)
{
    if (!ctx || n_prims < 0 || (n_prims > 0 && !deltas)) return SMPLGPU_ERR_INVALID;
    if (!ctx->has_robot) return fail(ctx, SMPLGPU_ERR_STATE, "robot tables not set (smplgpu_set_robot)");
    if (n_prims > 4096) return fail(ctx, SMPLGPU_ERR_LIMIT, "%d motion primitives", n_prims);
    const int dof = ctx->h_model->dof;
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->d_x1_deltas) { CU(cudaFree(ctx->d_x1_deltas)); ctx->d_x1_deltas = nullptr; }
    ctx->x1_prims = -1;
    CU(cudaMalloc(&ctx->d_x1_deltas, std::max<size_t>(1, (size_t)n_prims * dof) * sizeof(double)));
    if (n_prims > 0) {
        CU(cudaMemcpy(ctx->d_x1_deltas, deltas, (size_t)n_prims * dof * sizeof(double), cudaMemcpyHostToDevice));
    }
    if ((size_t)n_prims + 1 > ctx->x1_out_cap) {
        if (ctx->x1_out) { CU(cudaFreeHost(ctx->x1_out)); ctx->x1_out = nullptr; ctx->x1_out_cap = 0; }
        CU(cudaHostAlloc((void**)&ctx->x1_out, ((size_t)n_prims + 1) * sizeof(smplgpu_succ_info) + 64, cudaHostAllocMapped));
        ctx->x1_out_cap = (size_t)n_prims + 1;
    }
    if (!ctx->d_x1_done) {
        CU(cudaMalloc(&ctx->d_x1_done, sizeof(unsigned int)));
        CU(cudaMemset(ctx->d_x1_done, 0, sizeof(unsigned int)));
    }
    ctx->x1_prims = n_prims;
    ctx->x1_dof = dof;
    ++ctx->scene_epoch;
    return 0;
}

int smplgpu_expand_state(smplgpu_ctx* ctx, const double* parent, int cost_per_cell, const smplgpu_succ_info** info)
{
    if (!ctx || !parent || !info) return SMPLGPU_ERR_INVALID;
    int r = need_scene(ctx);
    if (r) return r;
    if (ctx->x1_prims < 0 || ctx->x1_dof != ctx->h_model->dof)
        return fail(ctx, SMPLGPU_ERR_STATE, "motion primitives not set for this robot (smplgpu_set_motion_primitives)");
    const bool bfs_ok = ctx->has_bfs && ctx->bfs.nx == ctx->grid.nx && ctx->bfs.ny == ctx->grid.ny && ctx->bfs.nz == ctx->grid.nz;
    Expand1Parent p;
    const int dof = ctx->h_model->dof;
    for (int v = 0; v < MAX_DOF; ++v) p.q[v] = v < dof ? parent[v] : 0.0;
    unsigned long long* flag = reinterpret_cast<unsigned long long*>(ctx->x1_out + ctx->x1_out_cap);
    volatile unsigned long long* vflag = flag;
    const unsigned long long seq = ++ctx->x1_seq;
    size_t smem = (size_t)ctx->h_model->n_slots * 12 * sizeof(double) * EXPAND1_THREADS;
    const bool f32 = use_f32(ctx);
    if (f32) {
        smem += (size_t)ctx->blob_words * 4 + ((size_t)ctx->v32_slots * 12 + (size_t)ctx->v32_ptrees * 3) * sizeof(float) * EXPAND1_THREADS + 16;
    }
    if (smem > (size_t)226 * 1024) return fail(ctx, SMPLGPU_ERR_LIMIT, "%d link slots do not fit the expansion kernel", ctx->h_model->n_slots);
    if (smem > ctx->x1_smem_set) {
        CU(raise_smem_cap(expand_state_kernel, (int)std::max(smem, (size_t)1024)));
        ctx->x1_smem_set = smem;
    }
    expand_state_kernel<<<ctx->x1_prims + 1, EXPAND1_THREADS, smem, ctx->stream>>>(
        ctx->d_model, ctx->d_df, ctx->grid, f32 ? ctx->d_blob : nullptr, f32 ? ctx->blob_words : 0, ctx->grid32,
        bfs_ok ? ctx->bfs.dist : nullptr, ctx->bfs.DX, ctx->bfs.DY, ctx->bfs.DZ, p,
        ctx->d_x1_deltas, cost_per_cell, ctx->x1_out, ctx->d_x1_done, flag, seq);
    ++ctx->launches;
    CU(cudaGetLastError());
    // the kernel's last block publishes `seq` behind the records; spinning on it costs less than a stream
    // synchronisation, which stays the fallback (and the way errors surface)
    for (int spin = 0; spin < (1 << 22) && *vflag != seq; ++spin) {
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    if (*vflag != seq) {
        CU(cudaStreamSynchronize(ctx->stream));
        if (*vflag != seq) return fail(ctx, SMPLGPU_ERR_CUDA, "expansion record was not published");
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    *info = ctx->x1_out;
    return 0;
}

} // extern "C"
