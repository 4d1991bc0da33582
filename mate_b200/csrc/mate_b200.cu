// mate_b200.cu -- host side of the C ABI declared in include/mate_b200.h.
//
// Owns the struct-of-arrays device state of one batch of environments and launches the
// fused step kernel (mate_step.cuh).  No torch types, no CPU simulation fallback.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <memory>
#include <sched.h>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "mate_step.cuh"
#include "mate_wrappers.cuh"
#include "mate_agents.cuh"
#include "mate_hostpath.cuh"
#include "mate_snapshot.cuh"
#include "mate_messages.cuh"
#include "mate_render.cuh"

using namespace mate;

static thread_local std::string g_error;

static int fail(int code, const std::string& msg) {
    g_error = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t err__ = (expr);                                                           \
        if (err__ != cudaSuccess)                                                             \
            return fail(MATE_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(err__));   \
    } while (0)

// ---- supported entity-count shapes (compile-time specialisations of the kernel) ------------
// All 17 presets of the reference (mate/assets/MATE-*.yaml).
#if defined(MATE_DEV_SHAPE_OTHERS)   // development builds: the other BASELINE shapes
#define MATE_SHAPES(X) X(4, 2, 9) X(4, 8, 0) X(8, 8, 9) X(0, 8, 32)
#elif defined(MATE_DEV_SHAPE)   // development builds: a single specialisation (profiles/tools/build_variant.sh)
#define MATE_SHAPES(X) X(4, 8, 9)
#else
#define MATE_SHAPES(X)                                                                        \
    X(1, 1, 0) X(1, 1, 9) X(1, 2, 0) X(1, 2, 9) X(2, 2, 0) X(2, 2, 9) X(2, 4, 0) X(2, 4, 9)   \
    X(4, 2, 0) X(4, 2, 9) X(4, 4, 0) X(4, 4, 9) X(4, 8, 0) X(4, 8, 9) X(8, 8, 0) X(8, 8, 9)   \
    X(0, 8, 32)
#endif

struct KernelInfo {
    void (*launch_wrappers)(const Params&, const ObsOps&, const float*, const float*, int num_envs, cudaStream_t);
    cudaError_t (*prepare_wrappers)();
    void (*launch)(const Params&, int grid, cudaStream_t);
    int envs_per_cta, dc, dt;
    cudaError_t (*prepare)();
    void (*launch_fov)(const Params&, const int32_t*, const int32_t*, const double*, double*, long long, cudaStream_t);
    void (*launch_soft)(const Params&, const uint8_t*, const uint8_t*, double*, float*, cudaStream_t);
    void (*launch_render)(const Params&, const int32_t*, int count, int size, uint8_t*, cudaStream_t);
};

// ---- L2 persistence for the fp32 obstacle entries -------------------------------------------------
// The simulation phase of a step reads obs_f4 and the packer reads it again 60 us later, while the observation rows
// stream through the L2.  When the rows of one launch are several times the L2 (MATE-4v8-9 x 65 536: 407 MB against
// 126 MB) the entries are evicted in between and the re-reads go to HBM in the middle of the write phase.  Such a
// simulator sets aside a part of the L2 for persisting lines while it lives (12 MB by default, MATE_B200_L2_KEEP=<MB>,
// 0 = off) and its step launches carry a persisting access window over the array.  Measured (profiles/r2v_summary.md):
// 10 - 16 MB set aside -1.5 to -2.2 % ms/step, 24 MB +4 %, 32 MB +22 % (the write stream needs the rest of the L2);
// no gain for the smaller workloads and a loss when the array does not fit the set-aside (MATE-Navigation), so only
// simulators that meet both conditions take part.  The device limit is reference-counted and restored afterwards.
struct L2Keep {
    std::mutex mu;
    int users[64] = {};
    size_t previous[64] = {};
};
static L2Keep g_l2;
static size_t l2_keep_wanted() {
    size_t mb = 12;
    if (const char* v = getenv("MATE_B200_L2_KEEP")) mb = (size_t)std::max(0, atoi(v));
    return mb << 20;
}
// returns the window a simulator of this size gets (0 = none) and takes a reference on the device's set-aside
static size_t l2_keep_acquire(int dev, size_t array_bytes, size_t row_bytes_per_launch) {
    const size_t want = l2_keep_wanted();
    if (want == 0 || array_bytes == 0 || array_bytes > want || dev < 0 || dev >= 64) return 0;
    int l2 = 0, max_persist = 0, max_window = 0;
    cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev);
    cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
    cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev);
    if (l2 <= 0 || row_bytes_per_launch < 3 * (size_t)l2) return 0;     // the rows do not flush the L2 between the two reads
    if ((size_t)std::max(max_persist, 0) < want || (size_t)std::max(max_window, 0) < array_bytes) return 0;
    std::lock_guard<std::mutex> lock(g_l2.mu);
    if (g_l2.users[dev] == 0) {
        size_t current = 0;
        cudaDeviceGetLimit(&current, cudaLimitPersistingL2CacheSize);
        g_l2.previous[dev] = current;
        if (current < want && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) != cudaSuccess) { cudaGetLastError(); return 0; }
    }
    ++g_l2.users[dev];
    return array_bytes;
}
static void l2_keep_release(int dev) {
    std::lock_guard<std::mutex> lock(g_l2.mu);
    if (dev < 0 || dev >= 64 || g_l2.users[dev] == 0) return;
    if (--g_l2.users[dev] == 0) {
        cudaCtxResetPersistingL2Cache();
        if (g_l2.previous[dev] < l2_keep_wanted()) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, g_l2.previous[dev]);
        cudaGetLastError();
    }
}

template <int NC, int NT, int NO>
static void launch_shape2(const Params& p, int grid, cudaStream_t stream) {
    using S = Shape2<NC, NT, NO>;
    Params q = p;
    q.warp_stride = S::WARP_BYTES + (p.obs_ops.n > 0 ? S::OPS_BYTES : 0);   // scratch of the folded observation wrappers
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(S::WARPS * 32);
    cfg.dynamicSmemBytes = (size_t)S::WARPS * q.warp_stride; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    if (NO > 0 && q.l2_window_bytes > 0 && q.mode == MODE_STEP) {   // resets and prepared episodes are written once: nothing to keep
        attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
        attr[0].val.accessPolicyWindow.base_ptr = q.obs_f4;
        attr[0].val.accessPolicyWindow.num_bytes = (size_t)q.l2_window_bytes;
        attr[0].val.accessPolicyWindow.hitRatio = 1.0f;
        attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cfg.attrs = attr; cfg.numAttrs = 1;
    }
    cudaLaunchKernelEx(&cfg, mate_step_kernel2<NC, NT, NO>, q);
}
template <int NC, int NT, int NO>
static void launch_fov_shape(const Params& p, const int32_t* env, const int32_t* camera, const double* angle, double* out,
                             long long n, cudaStream_t stream) {
    fov_range_kernel<NC, NO><<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(p, env, camera, angle, out, n);
}
template <int NC, int NT, int NO>
static void launch_soft_shape(const Params& p, const uint8_t* mask_ct, const uint8_t* done, double* edges, float* out, cudaStream_t stream) {
    const long long warps = (long long)p.num_envs * (NC > 0 ? NC : 1);
    soft_edges_kernel<NC, NO><<<(unsigned)((warps * 2 + 127) / 128), 128, 0, stream>>>(p, done, edges);
    soft_coverage_kernel<NC, NT, NO><<<(unsigned)((warps + 3) / 4), 128, 0, stream>>>(p, mask_ct, done, edges, out);
}
template <int NC, int NT, int NO>
static void launch_render_shape(const Params& p, const int32_t* env, int count, int size, uint8_t* out, cudaStream_t stream) {
    const int tiles = ((size + kRenderRows - 1) / kRenderRows) * ((size + kRenderCols - 1) / kRenderCols);
    const int words = size % 4 == 0 && ((uintptr_t)out & 3) == 0;   // every 4-pixel group is 3 aligned words
    render_kernel<NC, NT, NO><<<dim3((unsigned)tiles, (unsigned)std::min(count, 65535)), kRenderThreads, 0, stream>>>(
        p, env, count, size, words, out);
}
template <int NC, int NT, int NO>
static cudaError_t prepare_shape2() {
    using S = Shape2<NC, NT, NO>;
    return cudaFuncSetAttribute(mate_step_kernel2<NC, NT, NO>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                S::SMEM_BYTES + S::WARPS * S::OPS_BYTES);
}

template <int NC, int NT, int NO>
static void launch_wrappers_shape(const Params& p, const ObsOps& ops, const float* cam_affine, const float* tgt_affine,
                                  int num_envs, cudaStream_t stream) {
    using W = WShape<NC, NT, NO>;
    const int grid = (num_envs + W::WARPS - 1) / W::WARPS;
    obs_transform_kernel<NC, NT, NO><<<grid, W::WARPS * 32, W::SMEM_BYTES, stream>>>(p, ops, cam_affine, tgt_affine);
}
template <int NC, int NT, int NO>
static cudaError_t prepare_wrappers_shape() {
    return cudaFuncSetAttribute(obs_transform_kernel<NC, NT, NO>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                WShape<NC, NT, NO>::SMEM_BYTES);
}

static bool find_kernel(int nc, int nt, int no, KernelInfo* out) {
#define X(NC, NT, NO)                                                                          \
    if (nc == NC && nt == NT && no == NO) {                                                    \
        using S = Shape2<NC, NT, NO>;                                                          \
        *out = KernelInfo{&launch_wrappers_shape<NC, NT, NO>, &prepare_wrappers_shape<NC, NT, NO>,       \
                          &launch_shape2<NC, NT, NO>, S::ENVS_PER_CTA, S::DC, S::DT,             \
                          &prepare_shape2<NC, NT, NO>, &launch_fov_shape<NC, NT, NO>,            \
                          &launch_soft_shape<NC, NT, NO>, &launch_render_shape<NC, NT, NO>};    \
        return true;                                                                           \
    }
    MATE_SHAPES(X)
#undef X
    return false;
}

struct MateSim {
    MateConfig cfg;
    int num_envs = 0, bpad = 0, device = 0;
    long long env_index_base = 0;
    KernelInfo kernel{};
    Params base{};            // state pointers + scalars; per-call fields are filled per launch
    void* state_block = nullptr;
    size_t state_bytes = 0;
    void* host_block = nullptr;   // pinned host copy of the state block (get_state / set_state), made on first use
    Params host{};                // the state pointers of host_block, carved like those of base
    double* d_ranges = nullptr;
    unsigned long long seed = 0;
    uint64_t config_hash = 0; // fingerprint of cfg (config_fingerprint): snapshots load only into handles of the same configuration
    long long launches = 0;
    // prepared resets (mate_step.cuh): second state block, parameter block that addresses it, side stream
    void* next_block = nullptr;
    Params next_base{};       // = base with the state pointers of the second block
    Params* d_next = nullptr; // device copy of next_base (Params::next of the step launches)
    cudaStream_t side = nullptr;
    cudaEvent_t side_event = nullptr;
    double* soft_edges = nullptr;   // scratch of mate_b200_soft_coverage, allocated on first use
    int refill_mode = 0;      // 0 = off, 1 = side stream every refill_period steps, 2 = same stream after every step (tests)
    int refill_period = 512;
    int tile_envs = 32;       // environments per warp tile (Params::tile_envs), chosen from the batch size at creation
    int obs_format = MATE_OBS_FORMAT_F32;   // element type of the observation rows (mate_b200_set_observation_format)
    MateMessageFilter message_filter = {{INFINITY, INFINITY}, {1.0, 1.0}, {nullptr, nullptr}, {nullptr, nullptr}};   // deliver everything
    bool rows_written = false;              // a reset / step / step_host / observe has run: the format is fixed
    long long steps_since_refill = 0;
    // host-path (step_host) resources
    static constexpr int kHostStreams = 4;
    cudaStream_t hstreams[kHostStreams] = {};
    cudaEvent_t hevents[kHostStreams] = {};
    float *h_cam_act = nullptr, *h_tgt_act = nullptr, *h_cam_obs = nullptr, *h_tgt_obs = nullptr, *h_rewards = nullptr;
    uint8_t* h_done = nullptr;
    bool host_ready = false;                  // ensure_host_path has run to the end
    size_t l2_window = 0;                     // bytes of obs_f4 the step launches keep in the L2 (0: none), see l2_keep_acquire
    // compacted device -> host leg (mate_hostpath.cuh): region 0 = camera rows, 1 = target rows
    static constexpr int kMaxHostChunks = 64;
    int compact_mode = 0;                     // 1: rows cross the link compacted and are expanded by host threads
    uint4* d_compact[2] = {nullptr, nullptr}; // compact streams (a launch chunk's stream starts where its dense rows start)
    CompactEntry* d_table[2] = {nullptr, nullptr};
    unsigned int* d_count = nullptr;          // [kMaxHostChunks][2] chunks kept
    uint4* p_compact[2] = {nullptr, nullptr}; // pinned host copies of the above
    CompactEntry* p_table[2] = {nullptr, nullptr};
    // MATE_STEP_HOST_ROWS_KEPT: the rows of the previous call stay on the device (second pair of row buffers, used in turn);
    // only the 64-byte groups that differ from them cross the link and are rewritten in the caller's buffers
    float* h_rows2[2] = {nullptr, nullptr};
    int row_parity = 0;
    const float* kept_rows[2] = {nullptr, nullptr};  // the caller's buffers that hold the previous call's rows
    bool kept_valid = false;
    int last_leg = 0;                                // device -> host leg of the last step_host call (mate_b200_host_leg_info)
    unsigned long long last_link_bytes = 0;
    unsigned int* p_count = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t e_counts[kMaxHostChunks] = {}, e_stream[kMaxHostChunks] = {}, e_tables[kMaxHostChunks] = {};
    unsigned int* p_count_dev = nullptr;      // device address of the pinned p_count (the sizes are stored there by a kernel, not copied)
    std::unique_ptr<ExpandPool> pool;

    // Releases whatever mate_b200_create and ensure_host_path have made, also when either stopped part-way.
    ~MateSim() {
        for (int i = 0; i < kHostStreams; ++i) { if (hstreams[i]) cudaStreamDestroy(hstreams[i]); if (hevents[i]) cudaEventDestroy(hevents[i]); }
        cudaFree(h_cam_act); cudaFree(h_tgt_act); cudaFree(h_cam_obs); cudaFree(h_tgt_obs);
        cudaFree(h_rewards); cudaFree(h_done);
        pool.reset();   // before the events its threads wait on and the pinned buffers they read
        for (int r = 0; r < 2; ++r) { cudaFree(d_compact[r]); cudaFree(d_table[r]); cudaFreeHost(p_compact[r]); cudaFreeHost(p_table[r]); cudaFree(h_rows2[r]); }
        cudaFree(d_count); cudaFreeHost(p_count);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        for (int i = 0; i < kMaxHostChunks; ++i) {
            if (e_counts[i]) cudaEventDestroy(e_counts[i]);
            if (e_stream[i]) cudaEventDestroy(e_stream[i]);
            if (e_tables[i]) cudaEventDestroy(e_tables[i]);
        }
        if (side) { cudaStreamSynchronize(side); cudaStreamDestroy(side); }
        if (side_event) cudaEventDestroy(side_event);
        cudaFree(soft_edges);
        cudaFree(next_block);
        cudaFree(d_next);
        cudaFree(state_block);
        cudaFreeHost(host_block);
        cudaFree(d_ranges);
        if (l2_window) l2_keep_release(device);
    }
};

extern "C" const char* mate_b200_last_error(void) { return g_error.c_str(); }
extern "C" int mate_b200_abi_version(void) { return MATE_B200_ABI_VERSION; }

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// The per-environment struct-of-arrays members of a state block, in carve order, each with its rows per environment
// (a row is bpad elements, indexed [row * bpad + env]).  `stats` is not per environment; masks, vals and ready exist
// in the second block only.
template <typename F>
static void for_each_state_array(Params& p, int nc, int nt, int no, F&& f) {
    f(p.cam_x, nc); f(p.cam_y, nc); f(p.cam_phi, nc); f(p.cam_theta, nc);
    f(p.tgt_x, nt); f(p.tgt_y, nt);
    f(p.obs_x, no); f(p.obs_y, no); f(p.obs_r, no);
    f(p.obs_f4, no);
    f(p.tgt_pack, nt);
    f(p.cargo, 2); f(p.env_a, 1); f(p.env_b, 1);
    f(p.cc_clear, 1);
}

// Points the state arrays of `p` into `block`, each 256-byte aligned: the per-environment arrays, then `stats`, then
// (`prepared`: the second block of prepared resets) the first-view masks, the entity values and the ready tags.
// Returns the bytes of the block; with block == nullptr the pointers are left alone and only the size is computed.
static size_t carve_state(Params& p, char* block, int nc, int nt, int no, size_t bpad, bool prepared) {
    size_t off = 0;
    auto carve = [&](auto*& ptr, size_t count) {
        if (block) ptr = reinterpret_cast<std::remove_reference_t<decltype(ptr)>>(block + off);
        off = align_up(off + sizeof(*ptr) * count, 256);
    };
    for_each_state_array(p, nc, nt, no, [&](auto*& ptr, int rows) { carve(ptr, (size_t)rows * bpad); });
    carve(p.stats, 16);
    if (prepared) {
        carve(p.masks, (size_t)(nc + nt) * (no <= 16 ? 1 : 2) * bpad);
        carve(p.vals, (size_t)(3 * nt + 5 * nc) * bpad);
        carve(p.ready, bpad);
    }
    return off;
}

// 64-bit FNV-1a over the scalar fields of a MateConfig (reserved0 excepted) and the values of its three range arrays,
// in declaration order (MateSnapshotInfo::config_hash)
static uint64_t config_fingerprint(const MateConfig& c) {
    uint64_t h = 14695981039346656037ull;
    auto mix = [&](const void* data, size_t bytes) {
        for (size_t i = 0; i < bytes; ++i) { h ^= static_cast<const unsigned char*>(data)[i]; h *= 1099511628211ull; }
    };
    for (const int32_t v : {c.num_cameras, c.num_targets, c.num_obstacles, c.max_episode_steps, c.num_cargoes_per_target,
                            c.num_high_capacity_targets, c.targets_start_with_cargoes, c.shuffle_entities, c.reward_sparse})
        mix(&v, sizeof(v));
    for (const double v : {c.bounty_factor, c.camera_radius, c.camera_min_viewing_angle, c.camera_max_sight_range,
                           c.camera_rotation_step, c.camera_zooming_step, c.target_step_size, c.target_sight_range,
                           c.obstacle_transmittance, c.obstacle_radius_low, c.obstacle_radius_high})
        mix(&v, sizeof(v));
    if (c.num_cameras > 0) mix(c.camera_location_ranges, sizeof(double) * 4 * c.num_cameras);
    mix(c.target_location_ranges, sizeof(double) * 4 * c.num_targets);
    if (c.num_obstacles > 0) mix(c.obstacle_location_ranges, sizeof(double) * 4 * c.num_obstacles);
    return h;
}

extern "C" int mate_b200_create(const MateConfig* cfg, int32_t num_envs, int32_t device,
                                int64_t env_index_base, MateSim** out) {
    if (!cfg || !out) return fail(MATE_EINVAL, "null argument");
    if (num_envs <= 0) return fail(MATE_EINVAL, "num_envs must be positive");
    const int nc = cfg->num_cameras, nt = cfg->num_targets, no = cfg->num_obstacles;
    KernelInfo kernel;
    if (!find_kernel(nc, nt, no, &kernel)) {
        char buf[256];
        snprintf(buf, sizeof(buf),
                 "no kernel specialisation for (cameras=%d, targets=%d, obstacles=%d); add it to MATE_SHAPES in "
                 "mate_b200/csrc/mate_b200.cu and rebuild", nc, nt, no);
        return fail(MATE_EINVAL, buf);
    }
    if ((nc > 0 && !cfg->camera_location_ranges) || !cfg->target_location_ranges || (no > 0 && !cfg->obstacle_location_ranges))
        return fail(MATE_EINVAL, "missing location ranges");
    if (!(cfg->target_step_size > 0.0) || !(cfg->target_sight_range > 0.0)) return fail(MATE_EINVAL, "target parameters must be positive");
    if (nc > 0 && (!(cfg->camera_min_viewing_angle > 0.0) || cfg->camera_min_viewing_angle > 180.0 || !(cfg->camera_rotation_step > 0.0) ||
                   !(cfg->camera_zooming_step > 0.0) || !(cfg->camera_max_sight_range > 0.0)))
        return fail(MATE_EINVAL, "camera parameters out of range");
    if (cfg->max_episode_steps <= 0) return fail(MATE_EINVAL, "max_episode_steps must be positive");
    if (cfg->num_cargoes_per_target < MATE_NUM_WAREHOUSES) return fail(MATE_EINVAL, "num_cargoes_per_target must be >= 4");
    if (cfg->num_high_capacity_targets < 0 || cfg->num_high_capacity_targets > nt) return fail(MATE_EINVAL, "bad num_high_capacity_targets");
    const double freight_scale = std::ceil(2.0 * kTerrain / cfg->target_step_size);       // environment.py:521
    const double bounty_scale = std::ceil(freight_scale * std::fmax(0.0, cfg->bounty_factor));
    if (2.0 * bounty_scale > 65535.0 || (double)cfg->num_cargoes_per_target * nt > 65535.0)
        return fail(MATE_EINVAL, "bounty/cargo counts exceed the packed 16-bit state fields");

    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(kernel.prepare());
    CUDA_TRY(kernel.prepare_wrappers());
    std::unique_ptr<MateSim> sim(new MateSim());   // frees what is made so far on every early return
    sim->cfg = *cfg;
    sim->config_hash = config_fingerprint(*cfg);
    sim->cfg.camera_location_ranges = sim->cfg.target_location_ranges = sim->cfg.obstacle_location_ranges = nullptr;
    sim->num_envs = num_envs;
    sim->device = device;
    sim->env_index_base = env_index_base;
    sim->kernel = kernel;
    const int bpad = (int)align_up((size_t)num_envs, 256);
    sim->bpad = bpad;

    // one allocation, carved into the SoA arrays
    Params& p = sim->base;
    sim->state_bytes = carve_state(p, nullptr, nc, nt, no, bpad, false);
    if (cudaMalloc(&sim->state_block, sim->state_bytes) != cudaSuccess) return fail(MATE_ENOMEM, "cudaMalloc(state) failed");
    CUDA_TRY(cudaMemset(sim->state_block, 0, sim->state_bytes));
    carve_state(p, (char*)sim->state_block, nc, nt, no, bpad, false);

    // Warp tiles: 32 environments per warp for the batches that give every SM several of those; smaller batches are cut
    // into tiles of 16 or 8 so that the latency-bound launch still has warps to overlap (measured, MATE-4v8-9: 16 384
    // envs 0.0697 / 0.0622 / 0.0685 ms with 32 / 16 / 8, 4096 envs 0.0610 / 0.0468 / 0.0417; from 32 768 envs on 32 wins:
    // MATE-8v8-9 x 32 768 0.129 / 0.178 / 0.218 -- idle lanes still cost issue slots).
    sim->tile_envs = num_envs >= 24576 ? 32 : (num_envs >= 8192 ? 16 : 8);
    if (const char* v = getenv("MATE_B200_TILE")) { const int t = atoi(v); if (t == 8 || t == 16 || t == 32) sim->tile_envs = t; }
    p.tile_envs = sim->tile_envs;

    // location ranges on device (reset)
    std::vector<double> ranges((size_t)4 * (nc + nt + no) + 4, 0.0);
    if (nc) memcpy(ranges.data(), cfg->camera_location_ranges, sizeof(double) * 4 * nc);
    memcpy(ranges.data() + 4 * nc, cfg->target_location_ranges, sizeof(double) * 4 * nt);
    if (no) memcpy(ranges.data() + 4 * (nc + nt), cfg->obstacle_location_ranges, sizeof(double) * 4 * no);
    CUDA_TRY(cudaMalloc(&sim->d_ranges, ranges.size() * sizeof(double)));
    CUDA_TRY(cudaMemcpy(sim->d_ranges, ranges.data(), ranges.size() * sizeof(double), cudaMemcpyHostToDevice));
    p.cam_ranges = sim->d_ranges; p.tgt_ranges = sim->d_ranges + 4 * nc; p.obs_ranges = sim->d_ranges + 4 * (nc + nt);

    p.num_envs = num_envs; p.bpad = bpad; p.env_index_base = env_index_base; p.seed = 0;
    sim->l2_window = l2_keep_acquire(device, no > 0 ? ((size_t)(no - 1) * bpad + (size_t)num_envs) * sizeof(float4) : 0,
                                     (size_t)num_envs * ((size_t)nc * sim->kernel.dc + (size_t)nt * sim->kernel.dt) * sizeof(float));
    p.l2_window_bytes = sim->l2_window;
    p.max_episode_steps = cfg->max_episode_steps; p.num_cargoes_per_target = cfg->num_cargoes_per_target;
    p.num_high_capacity = cfg->num_high_capacity_targets; p.start_with_cargoes = cfg->targets_start_with_cargoes != 0;
    p.shuffle = cfg->shuffle_entities != 0; p.reward_sparse = cfg->reward_sparse != 0;
    p.transmittance = std::fmin(std::fmax(cfg->obstacle_transmittance, 0.0), 1.0);   // environment.py:1470-1476
    p.transmittance_is_one = p.transmittance == 1.0;
    p.freight_scale = (int)freight_scale; p.bounty_scale = (int)bounty_scale; p.reward_scale = (int)(freight_scale + bounty_scale);
    p.cam_radius = cfg->camera_radius; p.cam_min_view = cfg->camera_min_viewing_angle; p.cam_rmax = cfg->camera_max_sight_range;
    p.cam_rot_step = cfg->camera_rotation_step; p.cam_zoom_step = cfg->camera_zooming_step;
    p.cam_area_product = cfg->camera_min_viewing_angle * (cfg->camera_max_sight_range * cfg->camera_max_sight_range);  // entities.py:285
    p.tgt_step_size = cfg->target_step_size; p.tgt_sight_range = cfg->target_sight_range;
    p.obs_r_low = cfg->obstacle_radius_low; p.obs_r_high = cfg->obstacle_radius_high;

    // prepared resets: a second state block of the same layout + first-view masks + the ready tags, addressed by
    // next_base: the scalars and range pointers of the live block with the state pointers of the second block
    sim->refill_mode = 1;
    if (const char* v = getenv("MATE_B200_REFILL")) {
        if (!strcmp(v, "0") || !strcmp(v, "off")) sim->refill_mode = 0;
        else if (!strcmp(v, "sync")) sim->refill_mode = sim->refill_mode ? 2 : 0;
        else if (atoi(v) > 0) sim->refill_period = atoi(v);
    }
    if (sim->refill_mode) {
        Params& n = sim->next_base;
        n = p;
        const size_t block2 = carve_state(n, nullptr, nc, nt, no, bpad, true);
        if (cudaMalloc(&sim->next_block, block2) != cudaSuccess) return fail(MATE_ENOMEM, "cudaMalloc(prepared state) failed");
        CUDA_TRY(cudaMemset(sim->next_block, 0, block2));
        carve_state(n, (char*)sim->next_block, nc, nt, no, bpad, true);
        n.live_env_b = p.env_b;
        p.ready = n.ready;   // the live tags are the second block's
        CUDA_TRY(cudaMalloc(&sim->d_next, sizeof(Params)));
        CUDA_TRY(cudaStreamCreateWithFlags(&sim->side, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&sim->side_event, cudaEventDisableTiming));
        CUDA_TRY(cudaMemcpy(sim->d_next, &sim->next_base, sizeof(Params), cudaMemcpyHostToDevice));
        p.next = sim->d_next;
    }

    // neutral initial state so that a step before reset/set_state is well defined
    {
        std::vector<double> theta((size_t)nc * bpad, cfg->camera_min_viewing_angle > 0 ? cfg->camera_min_viewing_angle : 90.0);
        if (nc) CUDA_TRY(cudaMemcpy(p.cam_theta, theta.data(), theta.size() * sizeof(double), cudaMemcpyHostToDevice));
        std::vector<uint32_t> pack((size_t)nt * bpad, pack_target(0, -1, 0, 1, 0, 0));
        CUDA_TRY(cudaMemcpy(p.tgt_pack, pack.data(), pack.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    *out = sim.release();
    return MATE_OK;
}

extern "C" int mate_b200_destroy(MateSim* sim) {
    if (!sim) return MATE_OK;
    cudaSetDevice(sim->device);
    delete sim;
    return MATE_OK;
}

extern "C" int mate_b200_obs_dims(const MateSim* sim, int32_t* cam_dim, int32_t* tgt_dim) {
    if (!sim) return fail(MATE_EINVAL, "null handle");
    if (cam_dim) *cam_dim = sim->kernel.dc;
    if (tgt_dim) *tgt_dim = sim->kernel.dt;
    return MATE_OK;
}

// bytes of observation rows per environment in the handle's format: region 0 = camera rows, 1 = target rows
static size_t env_row_bytes(const MateSim* sim, int region) {
    const size_t elem = sim->obs_format == MATE_OBS_FORMAT_F16 ? 2 : 4;
    return region == 0 ? elem * sim->cfg.num_cameras * sim->kernel.dc : elem * sim->cfg.num_targets * sim->kernel.dt;
}
// the rows of environment `env` in a buffer of one region's rows (the row pointers are typed float* in the ABI)
static float* env_rows(const MateSim* sim, float* rows, int region, size_t env) {
    return reinterpret_cast<float*>(reinterpret_cast<char*>(rows) + env * env_row_bytes(sim, region));
}

// the kernel launch just enqueued was accepted
static int check_launch(const char* what) {
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(MATE_ECUDA, std::string(what) + " launch: " + cudaGetErrorString(err));
    return MATE_OK;
}

// the observation wrapper codes as an ObsOps (the count has been checked), in the order the reference admits:
// (Enhanced | Shared)* Relative? Rescaled? (MATE_MAX_OBS_OPS, include/mate_b200.h)
static int parse_obs_ops(const MateSim* sim, const int32_t* ops, int32_t num_ops, const float* cam_affine, const float* tgt_affine,
                         ObsOps* o) {
    *o = ObsOps{};
    o->n = num_ops;
    int stage = 0;   // 0 = mask codes, 1 = after MATE_OBS_RELATIVE, 2 = after MATE_OBS_RESCALED
    for (int i = 0; i < num_ops; ++i) {
        if (ops[i] < MATE_OBS_ENHANCED_CAMERA || ops[i] > MATE_OBS_RESCALED) return fail(MATE_EINVAL, "unknown observation wrapper code");
        if (ops[i] == MATE_OBS_RESCALED && (!tgt_affine || (sim->cfg.num_cameras > 0 && !cam_affine)))
            return fail(MATE_EINVAL, "MATE_OBS_RESCALED needs the affine tables");
        const int at = ops[i] == MATE_OBS_RESCALED ? 2 : (ops[i] == MATE_OBS_RELATIVE ? 1 : 0);
        if (at < stage || (at > 0 && at == stage))
            return fail(MATE_EINVAL, "observation wrappers must be stacked as (Enhanced | Shared)* Relative? Rescaled?");
        stage = at;
        o->op[i] = ops[i];
    }
    return MATE_OK;
}

extern "C" int mate_b200_set_observation_format(MateSim* sim, int32_t format) {
    if (!sim) return fail(MATE_EINVAL, "null handle");
    if (format != MATE_OBS_FORMAT_F32 && format != MATE_OBS_FORMAT_F16) return fail(MATE_EINVAL, "unknown observation format code");
    if (sim->rows_written)
        return fail(MATE_ESTATE, "the observation format can only be set before the handle's first reset, step, step_host or observe");
    sim->obs_format = format;
    sim->base.obs_format = format;
    return MATE_OK;
}

extern "C" int mate_b200_fov_range(MateSim* sim, const int32_t* env, const int32_t* camera, const double* angle_deg,
                                   double* out, int64_t n, void* stream) {
    if (!sim || !env || !camera || !angle_deg || !out || n < 0) return fail(MATE_EINVAL, "bad argument");
    if (sim->cfg.num_cameras == 0) return fail(MATE_EINVAL, "the configuration has no cameras");
    if (n == 0) return MATE_OK;
    CUDA_TRY(cudaSetDevice(sim->device));
    sim->kernel.launch_fov(sim->base, env, camera, angle_deg, out, n, (cudaStream_t)stream);
    sim->launches += 1;
    return check_launch("fov_range");
}

extern "C" int mate_b200_render(MateSim* sim, const int32_t* env, int32_t count, int32_t size, uint8_t* out, void* stream) {
    if (!sim || !out) return fail(MATE_EINVAL, "null argument");
    if (count <= 0) return fail(MATE_EINVAL, "count must be positive");
    if (!env && count != sim->num_envs) return fail(MATE_EINVAL, "without an environment list every environment is rendered: count must be num_envs");
    if (size < MATE_RENDER_MIN_SIZE || size > MATE_RENDER_MAX_SIZE) return fail(MATE_EINVAL, "size must lie in [MATE_RENDER_MIN_SIZE, MATE_RENDER_MAX_SIZE]");
    CUDA_TRY(cudaSetDevice(sim->device));
    sim->kernel.launch_render(sim->base, env, count, size, out, (cudaStream_t)stream);
    sim->launches += 1;
    return check_launch("render");
}

extern "C" int64_t mate_b200_launch_count(const MateSim* sim) { return sim ? sim->launches : 0; }
extern "C" int mate_b200_host_leg_info(const MateSim* sim, int32_t* leg, uint64_t* row_bytes_on_link) {
    if (!sim) return fail(MATE_EINVAL, "null handle");
    if (leg) *leg = sim->last_leg;
    if (row_bytes_on_link) *row_bytes_on_link = sim->last_link_bytes;
    return MATE_OK;
}

extern "C" int mate_b200_transform_observations(MateSim* sim, float* cam_obs, float* tgt_obs, const int32_t* ops,
                                                int32_t num_ops, const float* cam_affine, const float* tgt_affine,
                                                void* stream) {
    if (!sim || !tgt_obs || (sim->cfg.num_cameras > 0 && !cam_obs) || (num_ops > 0 && !ops)) return fail(MATE_EINVAL, "null argument");
    if (num_ops < 0 || num_ops > MATE_MAX_OBS_OPS) return fail(MATE_EINVAL, "too many observation wrappers (MATE_MAX_OBS_OPS)");
    if (sim->obs_format != MATE_OBS_FORMAT_F32)
        return fail(MATE_EINVAL, "transform_observations works on float32 rows; register the wrappers (set_observation_ops) on a float16 handle");
    if (num_ops == 0) return MATE_OK;
    if (((uintptr_t)cam_obs & 15) || ((uintptr_t)tgt_obs & 15)) return fail(MATE_EINVAL, "observation buffers must be 16-byte aligned");
    ObsOps o;
    if (int rc = parse_obs_ops(sim, ops, num_ops, cam_affine, tgt_affine, &o)) return rc;
    CUDA_TRY(cudaSetDevice(sim->device));
    Params p = sim->base;
    p.cam_obs = cam_obs; p.tgt_obs = tgt_obs;
    sim->kernel.launch_wrappers(p, o, cam_affine, tgt_affine, sim->num_envs, (cudaStream_t)stream);
    sim->launches += 1;
    return check_launch("wrapper kernel");
}

extern "C" int mate_b200_set_observation_ops(MateSim* sim, const int32_t* ops, int32_t num_ops, const float* cam_affine,
                                             const float* tgt_affine) {
    if (!sim || (num_ops > 0 && !ops)) return fail(MATE_EINVAL, "null argument");
    if (num_ops < 0 || num_ops > MATE_MAX_OBS_OPS) return fail(MATE_EINVAL, "too many observation wrappers (MATE_MAX_OBS_OPS)");
    ObsOps o;
    if (int rc = parse_obs_ops(sim, ops, num_ops, cam_affine, tgt_affine, &o)) return rc;
    // the stack -- (Enhanced | Shared)* Relative? Rescaled?, checked above -- is applied while the rows are composed (FoldOps)
    FoldOps f{};
    int k = 0;
    while (k < num_ops && ops[k] >= MATE_OBS_ENHANCED_CAMERA && ops[k] <= MATE_OBS_SHARED_TARGET) f.mask_op[f.n_mask++] = ops[k++];
    if (k < num_ops && ops[k] == MATE_OBS_RELATIVE) { f.relative = 1; ++k; }
    if (k < num_ops && ops[k] == MATE_OBS_RESCALED) { f.rescaled = 1; ++k; }
    f.fast = num_ops > 0 ? 1 : 0;
    if (f.fast && f.rescaled) {
        CUDA_TRY(cudaSetDevice(sim->device));
        const int nc = sim->cfg.num_cameras;
        const ObsLayout L{nc, sim->cfg.num_targets, sim->cfg.num_obstacles};
        const int dc = L.dc(), dt = L.dt();
        std::vector<float> cam((size_t)2 * std::max(dc, 1), 0.f), tgt((size_t)2 * dt, 0.f);
        if (nc) CUDA_TRY(cudaMemcpy(cam.data(), cam_affine, sizeof(float) * 2 * dc, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(tgt.data(), tgt_affine, sizeof(float) * 2 * dt, cudaMemcpyDeviceToHost));
        auto col = [](const std::vector<float>& t, int c) { return make_float2(t[2 * c], t[2 * c + 1]); };
        auto same = [](float2 a, float2 b) { return a.x == b.x && a.y == b.y; };
        bool uniform = true;
        for (int j = 0; j < ObsLayout::PRESERVED; ++j) { f.pres[j] = col(tgt, j); if (nc) uniform = uniform && same(f.pres[j], col(cam, j)); }
        for (int j = 0; j < ObsLayout::TGT_PRIVATE; ++j) f.tself[j] = col(tgt, ObsLayout::SELF + j);
        for (int j = 0; j < ObsLayout::CAM_PRIVATE && nc; ++j) f.cself[j] = col(cam, ObsLayout::SELF + j);
        // an entry of each kind from the target rows; every entry of a kind has the same bounds in both teams' rows
        // (mate/constants.py:195-254): checked, not assumed
        float2* const entry[3] = {f.tgt, f.obs, f.cam};   // by EntityKind
        for (int kind = KIND_TARGET; kind <= KIND_CAMERA; ++kind) {
            if (L.count(kind) == 0) continue;
            const int w = ObsLayout::width(kind);
            for (int j = 0; j < w; ++j) entry[kind][j] = col(tgt, L.entry_offset(false, kind, 0) + j);
            for (int e = 0; e < L.count(kind); ++e) for (int j = 0; j < w; ++j) {
                uniform = uniform && same(entry[kind][j], col(tgt, L.entry_offset(false, kind, e) + j));
                if (nc) uniform = uniform && same(entry[kind][j], col(cam, L.entry_offset(true, kind, e) + j));
            }
        }
        if (!uniform) f.fast = 0;   // tables of the caller's own: generic path
    }
    if (const char* v = getenv("MATE_B200_FOLD")) { if (v[0] == '0') f.fast = 0; }   // tests: force the generic shared-memory path
    sim->base.obs_ops = o;
    sim->base.cam_affine = cam_affine;
    sim->base.tgt_affine = tgt_affine;
    sim->base.fold = f;
    return MATE_OK;
}

extern "C" int mate_b200_soft_coverage(MateSim* sim, const uint8_t* mask_ct, const uint8_t* done, float* soft_matrix, void* stream) {
    if (!sim || !mask_ct || !soft_matrix) return fail(MATE_EINVAL, "null argument");
    if (sim->cfg.num_cameras == 0) return fail(MATE_EINVAL, "the configuration has no cameras");
    CUDA_TRY(cudaSetDevice(sim->device));
    if (!sim->soft_edges)   // ranges at the two sector edges of every camera, filled by the pre-pass
        CUDA_TRY(cudaMalloc(&sim->soft_edges, sizeof(double) * 2 * (size_t)sim->num_envs * sim->cfg.num_cameras));
    sim->kernel.launch_soft(sim->base, mask_ct, done, sim->soft_edges, soft_matrix, (cudaStream_t)stream);
    sim->launches += 2;
    return check_launch("soft coverage");
}

extern "C" int mate_b200_auxiliary_terms(MateSim* sim, const MateStepAux* aux, const float* rewards, const float* soft_matrix,
                                         float* cam_terms, float* tgt_terms, void* stream) {
    if (!sim || !aux || !rewards || !tgt_terms || (sim->cfg.num_cameras > 0 && !cam_terms)) return fail(MATE_EINVAL, "null argument");
    if (!aux->coverage || !aux->target_dones || !aux->is_colliding || !aux->warehouse_dist || !aux->tgt_goal || !aux->tgt_empty_bits ||
        (sim->cfg.num_cameras > 0 && (!aux->mask_ct || !aux->mask_tc)))
        return fail(MATE_EINVAL, "auxiliary_terms needs mask_ct, mask_tc, coverage, target_dones, is_colliding, warehouse_dist, tgt_goal, tgt_empty_bits");
    CUDA_TRY(cudaSetDevice(sim->device));
    if (((uintptr_t)cam_terms & 15) || ((uintptr_t)tgt_terms & 15) || ((uintptr_t)aux->warehouse_dist & 15))
        return fail(MATE_EINVAL, "term tensors and warehouse_dist must be 16-byte aligned");
    const int threads = 128;
    const long long agents = (long long)sim->num_envs * (sim->cfg.num_cameras + sim->cfg.num_targets);
    aux_terms_kernel<<<(unsigned)((agents + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        *aux, rewards, soft_matrix, cam_terms, tgt_terms, sim->num_envs, sim->cfg.num_cameras, sim->cfg.num_targets);
    sim->launches += 1;
    return check_launch("auxiliary terms");
}

// The registered communication wrappers of team 0 (cameras) or 1 (targets) as the agent kernels take them.
static CommFilter comm_filter(const MateSim* sim, int team) {
    const MateMessageFilter& f = sim->message_filter;
    CommFilter c{};
    c.range_limit = f.range_limit[team];
    // keep / 2^32 is the keep probability rounded down to a multiple of 2^-32; 1 gives 2^32 (every draw passes), 0 gives 0
    c.keep = (unsigned long long)floor(f.keep_probability[team] * 4294967296.0);
    c.seed = sim->seed;
    c.delivered = f.delivered[team];
    c.totals = f.total_edges[team];
    c.pairwise = (!isinf(c.range_limit) || c.keep <= 0xFFFFFFFFull || c.delivered || c.totals) ? 1 : 0;
    return c;
}

extern "C" int mate_b200_set_message_filter(MateSim* sim, const MateMessageFilter* filter) {
    if (!sim) return fail(MATE_EINVAL, "null handle");
    MateMessageFilter f = {{INFINITY, INFINITY}, {1.0, 1.0}, {nullptr, nullptr}, {nullptr, nullptr}};
    if (filter) f = *filter;
    const int team_size[2] = {sim->cfg.num_cameras, sim->cfg.num_targets};
    for (int t = 0; t < 2; ++t) {
        if (!(f.range_limit[t] >= 0.0)) return fail(MATE_EINVAL, "range_limit must be >= 0 or +inf");
        if (!(f.keep_probability[t] >= 0.0 && f.keep_probability[t] <= 1.0)) return fail(MATE_EINVAL, "keep_probability must lie in [0, 1]");
        if ((uintptr_t)f.delivered[t] & 7) return fail(MATE_EINVAL, "delivered must be 8-byte aligned");
        if ((uintptr_t)f.total_edges[t] & 3) return fail(MATE_EINVAL, "total_edges must be 4-byte aligned");
        const bool used = !isinf(f.range_limit[t]) || f.keep_probability[t] < 1.0 || f.delivered[t] || f.total_edges[t];
        if (used && team_size[t] > 8)
            return fail(MATE_EINVAL, "message filters and communication edges cover teams of at most 8 agents (bit 8 s + r)");
    }
    sim->message_filter = f;
    return MATE_OK;
}

extern "C" int mate_b200_greedy_target_actions(MateSim* sim, double* memory, const uint8_t* reset_mask, double noise_scale,
                                               uint64_t seed, uint64_t serial, const MateAgentReplay* replay, float* tgt_act,
                                               void* stream) {
    if (!sim || !memory || !tgt_act) return fail(MATE_EINVAL, "null argument");
    if (((uintptr_t)tgt_act & 7) || ((uintptr_t)memory & 7)) return fail(MATE_EINVAL, "agent buffers must be 8-byte aligned");
    CUDA_TRY(cudaSetDevice(sim->device));
    MateAgentReplay r{};
    if (replay) r = *replay;
    const int threads = 128;
    greedy_target_kernel<<<(sim->num_envs + threads - 1) / threads, threads, 0, (cudaStream_t)stream>>>(
        sim->base, sim->cfg.num_targets, memory, reset_mask, noise_scale, seed, serial, r, comm_filter(sim, 1), tgt_act);
    sim->launches += 1;
    return check_launch("greedy target");
}

extern "C" int mate_b200_greedy_camera_actions(MateSim* sim, double* memory, const uint8_t* tracked, const uint8_t* reset_mask,
                                               uint64_t seed, uint64_t serial, const MateCameraAgentReplay* replay, float* cam_act,
                                               void* stream) {
    if (!sim || !memory || !tracked || !cam_act) return fail(MATE_EINVAL, "null argument");
    if (sim->cfg.num_cameras == 0) return fail(MATE_EINVAL, "the configuration has no cameras");
    if (((uintptr_t)cam_act & 7) || ((uintptr_t)memory & 7)) return fail(MATE_EINVAL, "agent buffers must be 8-byte aligned");
    CUDA_TRY(cudaSetDevice(sim->device));
    MateCameraAgentReplay r{};
    if (replay) r = *replay;
    // one thread per camera agent; a warp's 32 agent memories are staged in shared memory
    const int nc = sim->cfg.num_cameras, nt = sim->cfg.num_targets;
    if (32 % nc != 0) return fail(MATE_EINVAL, "the batched GreedyCameraAgent needs a number of cameras that divides 32");
    const long long agents = (long long)sim->num_envs * nc;
    greedy_camera_kernel<<<(unsigned)((agents + kCameraAgentThreads - 1) / kCameraAgentThreads), kCameraAgentThreads, 0, (cudaStream_t)stream>>>(
        sim->base, nc, nt, memory, tracked, reset_mask, seed, serial, r, comm_filter(sim, 0), cam_act);
    sim->launches += 1;
    return check_launch("greedy camera");
}

extern "C" int mate_b200_exchange_messages(MateSim* sim, const MateMessageExchange* exchange, uint64_t serial, void* stream) {
    if (!sim || !exchange) return fail(MATE_EINVAL, "null argument");
    const MateMessageExchange m = *exchange;
    if (m.team != 0 && m.team != 1) return fail(MATE_EINVAL, "team must be 0 (cameras) or 1 (targets)");
    const int n = m.team == 0 ? sim->cfg.num_cameras : sim->cfg.num_targets;
    if (n < 1 || n > 8) return fail(MATE_EINVAL, "the message exchange covers teams of 1 to 8 agents (bit 8 s + r)");
    if (m.dim < 1 || (long long)n * n * m.dim > 0x7FFFFFFFll) return fail(MATE_EINVAL, "dim must be >= 1 and N * N * dim < 2^31");
    if (m.reduction != MATE_MESSAGES_NONE && m.reduction != MATE_MESSAGES_SUM && m.reduction != MATE_MESSAGES_MEAN)
        return fail(MATE_EINVAL, "reduction must be MATE_MESSAGES_NONE, _SUM or _MEAN");
    if (!m.content || !m.inbox || !m.episode) return fail(MATE_EINVAL, "content, inbox and episode are required");
    if (((uintptr_t)m.content & 3) || ((uintptr_t)m.inbox & 3) || ((uintptr_t)m.episode & 3))
        return fail(MATE_EINVAL, "content, inbox and episode must be 4-byte aligned");
    CUDA_TRY(cudaSetDevice(sim->device));
    const Params& p = sim->base;
    ExchangeArgs a{};
    a.content = m.content; a.recipients = m.recipients; a.inbox = m.inbox; a.delivered = m.delivered; a.episode = m.episode;
    a.x = m.team == 0 ? p.cam_x : p.tgt_x;
    a.y = m.team == 0 ? p.cam_y : p.tgt_y;
    a.env_b = p.env_b;
    a.comm = comm_filter(sim, m.team);
    a.num_envs = sim->num_envs; a.bpad = sim->bpad; a.n = n; a.dim = m.dim; a.reduction = m.reduction;
    a.vec = m.dim % 4 == 0 && !((uintptr_t)m.content & 15) && !((uintptr_t)m.inbox & 15);
    a.team = (uint32_t)m.team; a.serial = (uint32_t)serial; a.env_index_base = p.env_index_base;
    message_exchange_kernel<<<(sim->num_envs + kExchangeWarps - 1) / kExchangeWarps, kExchangeWarps * 32, 0, (cudaStream_t)stream>>>(a);
    sim->launches += 1;
    return check_launch("message exchange");
}

extern "C" int mate_b200_decode_actions(const int64_t* index, const float* table, int32_t table_size, float* out,
                                        int64_t count, void* stream) {
    if (!index || !table || !out || table_size <= 0 || count < 0) return fail(MATE_EINVAL, "bad argument");
    if (count == 0) return MATE_OK;
    if (((uintptr_t)out & 7) || ((uintptr_t)table & 7)) return fail(MATE_EINVAL, "action buffers must be 8-byte aligned");
    decode_actions_kernel<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(index, table, table_size, out, count);
    return check_launch("decode");
}

// CTAs of a step-kernel launch over `count` environments
static int step_grid(const MateSim* sim, int count) {
    const int per_cta = sim->kernel.envs_per_cta / 32 * sim->tile_envs;
    return (count + per_cta - 1) / per_cta;
}

// Launch the fused kernel over envs [begin, begin + count); I/O pointers are for env 0.
static int launch_range(MateSim* sim, Params p, int begin, int count, cudaStream_t stream) {
    const int nc = sim->cfg.num_cameras, nt = sim->cfg.num_targets;
    // SoA rows are indexed [row * bpad + env]: shifting the base pointers selects the sub-range
    for_each_state_array(p, nc, nt, sim->cfg.num_obstacles, [&](auto*& ptr, int) { ptr += begin; });
    if (p.cam_act) p.cam_act += (size_t)begin * nc * 2;
    if (p.tgt_act) p.tgt_act += (size_t)begin * nt * 2;
    if (p.cam_obs) p.cam_obs = env_rows(sim, p.cam_obs, 0, begin);
    if (p.tgt_obs) p.tgt_obs = env_rows(sim, p.tgt_obs, 1, begin);
    if (p.rewards) p.rewards += (size_t)begin * 2;
    if (p.done) p.done += begin;
    if (p.env_mask) p.env_mask += begin;
    if (p.replay_transmit) p.replay_transmit += (size_t)begin * nc * nt;
    if (p.replay_choice) p.replay_choice += (size_t)begin * nt;
    if (p.ready) p.ready += begin;   // the live tags, an array of the second block
    p.next_offset = begin;   // `next` addresses whole-batch arrays
    p.env_index_base += begin;
    p.num_envs = count;
    sim->kernel.launch(p, step_grid(sim, count), stream);
    sim->launches += 1;
    return check_launch("kernel");
}

static int check_obs_alignment(const void* cam_obs, const void* tgt_obs) {
    if (((uintptr_t)cam_obs & 15) || ((uintptr_t)tgt_obs & 15)) return fail(MATE_EINVAL, "observation buffers must be 16-byte aligned");
    return MATE_OK;
}

// the view masks / per-target flags are written with 4-, 8- and 16-byte stores
static int check_aux_alignment(const MateStepAux* aux) {
    if (!aux) return MATE_OK;
    const void* ptrs[] = {aux->mask_ct, aux->mask_cc, aux->mask_co, aux->mask_tc, aux->mask_to, aux->mask_tt, aux->target_dones,
                          aux->is_colliding, aux->warehouse_dist};
    for (const void* ptr : ptrs)
        if ((uintptr_t)ptr & 15) return fail(MATE_EINVAL, "auxiliary output buffers must be 16-byte aligned");
    return MATE_OK;
}

static void fill_aux(Params& p, const MateStepAux* aux, const MateReplay* replay) {
    if (aux) {
        p.aux = *aux; p.has_aux = 1;
        p.has_aux_detail = aux->mask_ct || aux->mask_cc || aux->mask_co || aux->mask_tc || aux->mask_to || aux->mask_tt ||
                           aux->target_dones || aux->is_colliding || aux->warehouse_dist || aux->tgt_goal || aux->tgt_empty_bits;
    } else {
        memset(&p.aux, 0, sizeof(p.aux)); p.has_aux = 0; p.has_aux_detail = 0;
    }
    p.replay_transmit = replay ? replay->transmit : nullptr;
    p.replay_choice = replay ? replay->goal_choice : nullptr;
}

// Launch MODE_PREPARE over the second state block: re-initialises the prepared next episode of every env
// whose tag is stale.  Off the step path: on the side stream, ordered after the work already enqueued on
// `stream` (refill_mode 2: on `stream` itself, used by the tests to make the prepared path deterministic).
static int launch_prepare(MateSim* sim, cudaStream_t stream) {
    if (!sim->refill_mode) return MATE_OK;
    cudaStream_t target = stream;
    if (sim->refill_mode == 1) {
        CUDA_TRY(cudaEventRecord(sim->side_event, stream));
        CUDA_TRY(cudaStreamWaitEvent(sim->side, sim->side_event, 0));
        target = sim->side;
    }
    Params n = sim->next_base;
    n.mode = MODE_PREPARE; n.flags = 0; n.seed = sim->seed; n.l2_window_bytes = 0;
    n.cam_act = n.tgt_act = nullptr; n.cam_obs = n.tgt_obs = n.rewards = nullptr; n.done = nullptr; n.env_mask = nullptr;
    fill_aux(n, nullptr, nullptr);
    sim->kernel.launch(n, step_grid(sim, sim->num_envs), target);
    sim->launches += 1;
    sim->steps_since_refill = 0;
    return check_launch("prepare");
}

// after a step with auto-resets: refill the prepared episodes every refill_period steps (refill_mode 2: every step)
static int refill_after_step(MateSim* sim, uint32_t flags, cudaStream_t stream) {
    if ((flags & MATE_STEP_AUTO_RESET) && sim->refill_mode &&
        (sim->refill_mode == 2 || ++sim->steps_since_refill >= sim->refill_period))
        return launch_prepare(sim, stream);
    return MATE_OK;
}

// the prepared episodes no longer match the live state (explicit reset with a new seed, set_state)
static int invalidate_prepared(MateSim* sim, cudaStream_t stream) {
    if (!sim->refill_mode) return MATE_OK;
    CUDA_TRY(cudaStreamSynchronize(sim->side));
    CUDA_TRY(cudaMemsetAsync(sim->base.ready, 0, sizeof(uint32_t) * sim->bpad, stream));
    return MATE_OK;
}

__global__ void rewind_episode_kernel(int4* __restrict__ env_b, const uint8_t* __restrict__ env_mask, int num_envs) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < num_envs && (env_mask == nullptr || env_mask[e] != 0)) env_b[e].w = 0;
}

extern "C" int mate_b200_seed(MateSim* sim, const uint8_t* env_mask, uint64_t seed, void* stream) {
    if (!sim) return fail(MATE_EINVAL, "null handle");
    CUDA_TRY(cudaSetDevice(sim->device));
    sim->seed = seed;
    if (int rc = invalidate_prepared(sim, (cudaStream_t)stream)) return rc;
    rewind_episode_kernel<<<(sim->num_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(sim->base.env_b, env_mask, sim->num_envs);
    return check_launch("seed");
}

extern "C" int mate_b200_reset(MateSim* sim, const uint8_t* env_mask, uint64_t seed, float* cam_obs,
                               float* tgt_obs, void* stream) {
    if (!sim) return fail(MATE_EINVAL, "null argument");
    if (int rc = check_obs_alignment(cam_obs, tgt_obs)) return rc;
    CUDA_TRY(cudaSetDevice(sim->device));
    sim->seed = seed;
    sim->rows_written = true;
    Params p = sim->base;
    p.mode = MODE_RESET; p.flags = 0; p.seed = seed;
    p.cam_obs = cam_obs; p.tgt_obs = tgt_obs; p.env_mask = env_mask;
    fill_aux(p, nullptr, nullptr);
    if (int rc = invalidate_prepared(sim, (cudaStream_t)stream)) return rc;
    if (int rc = launch_range(sim, p, 0, sim->num_envs, (cudaStream_t)stream)) return rc;
    return launch_prepare(sim, (cudaStream_t)stream);
}

extern "C" int mate_b200_step(MateSim* sim, const float* cam_act, const float* tgt_act, float* cam_obs,
                              float* tgt_obs, float* rewards, uint8_t* done, const MateStepAux* aux,
                              const MateReplay* replay, uint32_t flags, void* stream) {
    if (!sim || !tgt_act || !rewards || !done) return fail(MATE_EINVAL, "null argument");
    if (sim->cfg.num_cameras > 0 && !cam_act) return fail(MATE_EINVAL, "null camera actions");
    if (int rc = check_obs_alignment(cam_obs, tgt_obs)) return rc;
    if (((uintptr_t)cam_act & 7) || ((uintptr_t)tgt_act & 7) || ((uintptr_t)rewards & 7)) return fail(MATE_EINVAL, "action/reward buffers must be 8-byte aligned");
    if (int rc = check_aux_alignment(aux)) return rc;
    CUDA_TRY(cudaSetDevice(sim->device));
    sim->rows_written = true;
    Params p = sim->base;
    p.mode = MODE_STEP; p.flags = flags; p.seed = sim->seed;
    p.cam_act = cam_act; p.tgt_act = tgt_act; p.cam_obs = cam_obs; p.tgt_obs = tgt_obs; p.rewards = rewards; p.done = done;
    fill_aux(p, aux, replay);
    if (int rc = launch_range(sim, p, 0, sim->num_envs, (cudaStream_t)stream)) return rc;
    return refill_after_step(sim, flags, (cudaStream_t)stream);
}

extern "C" int mate_b200_observe(MateSim* sim, float* cam_obs, float* tgt_obs, const MateStepAux* aux,
                                 const MateReplay* replay, void* stream) {
    if (!sim) return fail(MATE_EINVAL, "null argument");
    if (int rc = check_obs_alignment(cam_obs, tgt_obs)) return rc;
    if (int rc = check_aux_alignment(aux)) return rc;
    CUDA_TRY(cudaSetDevice(sim->device));
    sim->rows_written = true;
    Params p = sim->base;
    p.mode = MODE_OBSERVE; p.flags = 0; p.seed = sim->seed;
    p.cam_obs = cam_obs; p.tgt_obs = tgt_obs;
    fill_aux(p, aux, replay);
    return launch_range(sim, p, 0, sim->num_envs, (cudaStream_t)stream);
}

// ---- host-buffer path: chunked H2D -> kernel -> D2H over a few streams ------------------------
// Makes only what is still missing, so that a call after a failed one does not make anything twice.
static int ensure_host_path(MateSim* sim) {
    if (sim->host_ready) return MATE_OK;
    const size_t B = sim->num_envs;
    const int nc = sim->cfg.num_cameras, nt = sim->cfg.num_targets;
    for (int i = 0; i < MateSim::kHostStreams; ++i) {
        if (!sim->hstreams[i]) CUDA_TRY(cudaStreamCreateWithFlags(&sim->hstreams[i], cudaStreamNonBlocking));
        if (!sim->hevents[i]) CUDA_TRY(cudaEventCreateWithFlags(&sim->hevents[i], cudaEventDisableTiming));
    }
    if (!sim->h_cam_act) CUDA_TRY(cudaMalloc(&sim->h_cam_act, sizeof(float) * (B * nc * 2 + 4)));
    if (!sim->h_tgt_act) CUDA_TRY(cudaMalloc(&sim->h_tgt_act, sizeof(float) * B * nt * 2));
    if (!sim->h_cam_obs) CUDA_TRY(cudaMalloc(&sim->h_cam_obs, sizeof(float) * (B * nc * sim->kernel.dc + 4)));
    if (!sim->h_tgt_obs) CUDA_TRY(cudaMalloc(&sim->h_tgt_obs, sizeof(float) * B * nt * sim->kernel.dt));
    if (!sim->h_rewards) CUDA_TRY(cudaMalloc(&sim->h_rewards, sizeof(float) * B * 2));
    if (!sim->h_done) CUDA_TRY(cudaMalloc(&sim->h_done, B));
    // Compacted device -> host leg (mate_hostpath.cuh): what bounds it is the number of host threads that rebuild the dense
    // rows (measured with 15: 9.3 - 9.6e6 env-steps/s against 8.6 - 8.7e6 for the dense copy, with 10: 8.3e6, with 6: 6.4e6,
    // profiles/r2v_hostpath.md), so it is used when this process has at least 14 of them to itself -- all host threads the
    // process may run on but the caller's, divided among the processes that share the host (one per GPU) -- and the rows
    // are whole 16-byte chunks.  MATE_B200_HOST_COMPACT=0 / 1 forces the choice, MATE_B200_HOST_THREADS the pool size.
    int threads = (int)std::thread::hardware_concurrency();
    {
        cpu_set_t set;
        if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) threads = std::min(threads > 0 ? threads : CPU_COUNT(&set), CPU_COUNT(&set));
    }
    int sharers = 1;
    if (const char* v = getenv("LOCAL_WORLD_SIZE")) sharers = std::max(1, atoi(v));
    threads = std::max(1, threads / sharers - 1);
    if (const char* v = getenv("MATE_B200_HOST_THREADS")) threads = std::max(1, atoi(v));
    threads = std::min(threads, 64);
    // 1: every call takes the compacted leg (rebuilding all rows needs >= 14 threads to beat the dense copy); 2: only the calls
    // that patch changes into kept rows do (5 threads are enough for those: 1.02e7 against 8.5e6; 3 when four or more
    // processes share the host, whose memory system then bounds the dense copies: 8 x B200 1.74e7 against 1.49e7), the others
    // copy densely
    sim->compact_mode = threads >= 14 ? 1 : ((threads >= 5 || (threads >= 3 && sharers >= 4)) ? 2 : 0);
    if (const char* v = getenv("MATE_B200_HOST_COMPACT")) sim->compact_mode = v[0] == '1' ? 1 : (v[0] == '2' ? 2 : 0);
    if (env_row_bytes(sim, 0) % 16 || env_row_bytes(sim, 1) % 16) sim->compact_mode = 0;
    if (sim->compact_mode) {
        const size_t region_bytes[2] = {B * env_row_bytes(sim, 0), B * env_row_bytes(sim, 1)};
        bool ok = true;
        for (int r = 0; r < 2 && ok; ++r) {
            if (region_bytes[r] == 0) continue;
            const size_t chunks = region_bytes[r] / 16 + 8, blocks = chunks / kCompactBlock + MateSim::kMaxHostChunks + 1;
            ok = cudaMalloc(&sim->d_compact[r], chunks * 16) == cudaSuccess && cudaMalloc(&sim->d_table[r], blocks * sizeof(CompactEntry)) == cudaSuccess &&
                 cudaMallocHost(&sim->p_compact[r], chunks * 16) == cudaSuccess && cudaMallocHost(&sim->p_table[r], blocks * sizeof(CompactEntry)) == cudaSuccess &&
                 cudaMalloc(&sim->h_rows2[r], region_bytes[r] + 16) == cudaSuccess;
        }
        ok = ok && cudaMalloc(&sim->d_count, sizeof(unsigned int) * MateSim::kMaxHostChunks * 2) == cudaSuccess &&
             cudaMallocHost(&sim->p_count, sizeof(unsigned int) * MateSim::kMaxHostChunks * 2) == cudaSuccess &&
             cudaHostGetDevicePointer(reinterpret_cast<void**>(&sim->p_count_dev), sim->p_count, 0) == cudaSuccess &&
             cudaStreamCreateWithFlags(&sim->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
        for (int i = 0; i < MateSim::kMaxHostChunks && ok; ++i)
            ok = cudaEventCreateWithFlags(&sim->e_tables[i], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&sim->e_counts[i], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&sim->e_stream[i], cudaEventDisableTiming) == cudaSuccess;
        if (ok) sim->pool.reset(new ExpandPool(threads, sim->device));
        else {   // not enough pinned host memory or device memory for the second copy of the rows: the dense leg needs neither
            cudaGetLastError();
            sim->compact_mode = 0;
            for (int r = 0; r < 2; ++r) { cudaFree(sim->h_rows2[r]); sim->h_rows2[r] = nullptr; }
        }
    }
    sim->host_ready = true;
    return MATE_OK;
}

// one launch chunk of a step_host call, enqueued on `s`: its actions to the device, then the step over its environments
static int step_chunk(MateSim* sim, const Params& p, const float* cam_act, const float* tgt_act, int begin, int count, cudaStream_t s) {
    const int nc = sim->cfg.num_cameras, nt = sim->cfg.num_targets;
    if (nc) CUDA_TRY(cudaMemcpyAsync(sim->h_cam_act + (size_t)begin * nc * 2, cam_act + (size_t)begin * nc * 2, sizeof(float) * count * nc * 2, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(sim->h_tgt_act + (size_t)begin * nt * 2, tgt_act + (size_t)begin * nt * 2, sizeof(float) * count * nt * 2, cudaMemcpyHostToDevice, s));
    return launch_range(sim, p, begin, count, s);
}

// the rewards and done flags of a launch chunk to the caller's buffers, enqueued on `s`
static int copy_rewards_done(MateSim* sim, float* rewards, uint8_t* done, int begin, int count, cudaStream_t s) {
    CUDA_TRY(cudaMemcpyAsync(rewards + (size_t)begin * 2, sim->h_rewards + (size_t)begin * 2, sizeof(float) * count * 2, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(done + begin, sim->h_done + begin, count, cudaMemcpyDeviceToHost, s));
    return MATE_OK;
}

// ---- dense device -> host leg: every chunk's rows are copied as they are
static int dense_leg(MateSim* sim, const Params& p, int chunk, const float* cam_act, const float* tgt_act, float* cam_obs,
                     float* tgt_obs, float* rewards, uint8_t* done) {
    const int B = sim->num_envs;
    int k = 0;
    for (int begin = 0; begin < B; begin += chunk, ++k) {
        const int count = std::min(chunk, B - begin);
        cudaStream_t s = sim->hstreams[k % MateSim::kHostStreams];
        if (int rc = step_chunk(sim, p, cam_act, tgt_act, begin, count, s)) return rc;
        if (sim->cfg.num_cameras && cam_obs) CUDA_TRY(cudaMemcpyAsync(env_rows(sim, cam_obs, 0, begin), env_rows(sim, p.cam_obs, 0, begin), count * env_row_bytes(sim, 0), cudaMemcpyDeviceToHost, s));
        if (tgt_obs) CUDA_TRY(cudaMemcpyAsync(env_rows(sim, tgt_obs, 1, begin), env_rows(sim, p.tgt_obs, 1, begin), count * env_row_bytes(sim, 1), cudaMemcpyDeviceToHost, s));
        if (int rc = copy_rewards_done(sim, rewards, done, begin, count, s)) return rc;
    }
    for (int i = 0; i < MateSim::kHostStreams; ++i) CUDA_TRY(cudaStreamSynchronize(sim->hstreams[i]));
    sim->last_leg = 0; sim->last_link_bytes = (unsigned long long)B * ((cam_obs ? env_row_bytes(sim, 0) : 0) + (tgt_obs ? env_row_bytes(sim, 1) : 0));
    return MATE_OK;
}

// ---- compacted device -> host leg (mate_hostpath.cuh): every launch chunk's rows are compacted on the device, the
//      compact streams cross the link one after the other, host threads expand them into the caller's buffers
//      (`delta`: the changes against `rows_before` are patched into the rows the caller's buffers still hold)
static int compact_leg(MateSim* sim, const Params& p, int chunk, bool delta, const float* const rows_before[2],
                       const float* cam_act, const float* tgt_act, float* cam_obs, float* tgt_obs, float* rewards, uint8_t* done) {
    static const bool trace = getenv("MATE_B200_HOST_TRACE") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count(); };
    double t_enq = 0, t_counts = 0, t_last_stream = 0;
    const int B = sim->num_envs;
    const int num_chunks = (B + chunk - 1) / chunk;
    float* const host_rows[2] = {cam_obs, tgt_obs};
    // a team without a buffer is a region of no rows: no compaction, no table, no stream, no expansion
    const size_t per_env[2] = {cam_obs ? env_row_bytes(sim, 0) : 0, tgt_obs ? env_row_bytes(sim, 1) : 0};
    const float* const dev_rows[2] = {p.cam_obs, p.tgt_obs};
    std::vector<long long> table_base(2 * (num_chunks + 1), 0);
    CUDA_TRY(cudaMemsetAsync(sim->d_count, 0, sizeof(unsigned int) * MateSim::kMaxHostChunks * 2, sim->hstreams[0]));
    CUDA_TRY(cudaEventRecord(sim->hevents[1], sim->hstreams[0]));
    for (int i = 1; i < MateSim::kHostStreams; ++i) CUDA_TRY(cudaStreamWaitEvent(sim->hstreams[i], sim->hevents[1], 0));
    int kc = 0;
    for (int begin = 0; begin < B; begin += chunk, ++kc) {
        const int count = std::min(chunk, B - begin);
        cudaStream_t s = sim->hstreams[kc % MateSim::kHostStreams];
        if (int rc = step_chunk(sim, p, cam_act, tgt_act, begin, count, s)) return rc;
        for (int r = 0; r < 2; ++r) {
            table_base[2 * (kc + 1) + r] = table_base[2 * kc + r];
            if (per_env[r] == 0) continue;
            const size_t first = (size_t)begin * per_env[r] / 16;            // B % 4 == 0 and chunk % 4 == 0: whole chunks
            const long long nchunks = (long long)((size_t)count * per_env[r] / 16);
            const long long nblocks = (nchunks + kCompactBlock - 1) / kCompactBlock;
            CompactEntry* table = sim->d_table[r] + table_base[2 * kc + r];
            table_base[2 * (kc + 1) + r] += nblocks;
            if (delta) compact_changes_kernel<<<1184, 128, 0, s>>>(reinterpret_cast<const uint4*>(dev_rows[r]) + first, reinterpret_cast<const uint4*>(rows_before[r]) + first,
                                                                   nchunks, sim->d_compact[r] + first, table, sim->d_count + 2 * kc + r);
            else compact_chunks_kernel<<<1184, 128, 0, s>>>(reinterpret_cast<const uint4*>(dev_rows[r]) + first, nchunks,
                                                            sim->d_compact[r] + first, table, sim->d_count + 2 * kc + r);
            sim->launches += 1;
        }
        // The sizes of the chunk's compact streams go to the host by a store into pinned memory, not by a copy: a copy
        // would queue behind the compact streams of earlier chunks on the copy engine, and the next stream could only be
        // enqueued after the previous one had crossed the link (a bubble per chunk).
        publish_counts_kernel<<<1, 32, 0, s>>>(sim->d_count + 2 * kc, sim->p_count_dev + 2 * kc);
        CUDA_TRY(cudaEventRecord(sim->e_counts[kc], s));
        for (int r = 0; r < 2; ++r) {
            const long long nblocks = table_base[2 * (kc + 1) + r] - table_base[2 * kc + r];
            if (nblocks > 0) CUDA_TRY(cudaMemcpyAsync(sim->p_table[r] + table_base[2 * kc + r], sim->d_table[r] + table_base[2 * kc + r], sizeof(CompactEntry) * nblocks, cudaMemcpyDeviceToHost, s));
        }
        if (int rc = copy_rewards_done(sim, rewards, done, begin, count, s)) return rc;
        CUDA_TRY(cudaEventRecord(sim->e_tables[kc], s));
    }
    t_enq = since();
    // the sizes are known once a chunk's kernels have run: its compact streams go on the copy stream in chunk order
    const int pieces = std::max(1, sim->pool->size());
    kc = 0;
    for (int begin = 0; begin < B; begin += chunk, ++kc) {
        CUDA_TRY(cudaEventSynchronize(sim->e_counts[kc]));
        CUDA_TRY(cudaStreamWaitEvent(sim->copy_stream, sim->e_tables[kc], 0));   // a chunk's stream event then covers its tables too
        for (int r = 0; r < 2; ++r) {
            if (per_env[r] == 0 || sim->p_count[2 * kc + r] == 0) continue;
            const size_t first = (size_t)begin * per_env[r] / 16;
            CUDA_TRY(cudaMemcpyAsync(sim->p_compact[r] + first, sim->d_compact[r] + first, (size_t)sim->p_count[2 * kc + r] * 16,
                                     cudaMemcpyDeviceToHost, sim->copy_stream));
        }
        CUDA_TRY(cudaEventRecord(sim->e_stream[kc], sim->copy_stream));
        // expansion: the pool's threads wait for the chunk's stream themselves, so the caller's thread goes on to the next sizes
        const int count = std::min(chunk, B - begin);
        for (int r = 0; r < 2; ++r) {
            if (per_env[r] == 0) continue;
            const size_t first = (size_t)begin * per_env[r] / 16;
            const long long nchunks = (long long)((size_t)count * per_env[r] / 16);
            const long long nblocks = (nchunks + kCompactBlock - 1) / kCompactBlock;
            const long long per_piece = (nblocks + pieces - 1) / pieces;
            __m128i* dst = reinterpret_cast<__m128i*>(host_rows[r]) + first;
            const bool aligned = (((uintptr_t)dst) & 15) == 0;
            for (long long b0 = 0; b0 < nblocks; b0 += per_piece)
                sim->pool->submit(ExpandPool::Work{sim->p_table[r] + table_base[2 * kc + r], delta, reinterpret_cast<const __m128i*>(sim->p_compact[r] + first),
                                                   dst, nchunks, b0, std::min(nblocks, b0 + per_piece), aligned, sim->e_stream[kc]});
        }
    }
    t_counts = since();
    CUDA_TRY(cudaStreamSynchronize(sim->copy_stream));
    t_last_stream = since();
    sim->pool->wait();
    for (int i = 0; i < MateSim::kHostStreams; ++i) CUDA_TRY(cudaStreamSynchronize(sim->hstreams[i]));
    {
        unsigned long long link = 0;
        for (int i = 0; i < 2 * num_chunks; ++i) link += (unsigned long long)sim->p_count[i] * 16ull;
        link += (unsigned long long)(table_base[2 * num_chunks] + table_base[2 * num_chunks + 1]) * sizeof(CompactEntry);
        sim->last_leg = delta ? 2 : 1; sim->last_link_bytes = link;
    }
    if (trace) {
        unsigned long long kept = 0;
        for (int i = 0; i < 2 * num_chunks; ++i) kept += sim->p_count[i];
        fprintf(stderr, "step_host compact: enqueued %.2f ms, sizes known + copies enqueued %.2f, last stream arrived %.2f, expanded %.2f; kept %.1f MB of %.1f MB, %d threads, changes only %d\n",
                t_enq, t_counts, t_last_stream, since(), kept * 16 / 1e6, (per_env[0] + per_env[1]) * (double)B / 1e6, sim->pool->size(), (int)delta);
    }
    return MATE_OK;
}

extern "C" int mate_b200_step_host(MateSim* sim, const float* cam_act, const float* tgt_act, float* cam_obs,
                                   float* tgt_obs, float* rewards, uint8_t* done, uint32_t flags) {
    if (!sim || !tgt_act || !rewards || !done) return fail(MATE_EINVAL, "null argument");
    const int nc = sim->cfg.num_cameras;
    if (nc > 0 && !cam_act) return fail(MATE_EINVAL, "null camera actions");
    CUDA_TRY(cudaSetDevice(sim->device));
    sim->rows_written = true;
    if (int rc = ensure_host_path(sim)) return rc;
    const int B = sim->num_envs;
    // chunk size: a multiple of the CTA tile, ~16 chunks so copies and kernels overlap
    int chunk = (B + 15) / 16;
    const int tile = sim->kernel.envs_per_cta * 8;
    chunk = (int)align_up((size_t)std::max(chunk, 1), (size_t)tile);
    Params p = sim->base;
    p.mode = MODE_STEP; p.flags = flags; p.seed = sim->seed;
    // the rows of this call and of the previous one take turns in two pairs of device buffers (compacted leg only)
    const bool two_buffers = sim->compact_mode && sim->h_rows2[1] != nullptr && (nc == 0 || sim->h_rows2[0] != nullptr);
    float* const rows_now[2] = {two_buffers && sim->row_parity ? sim->h_rows2[0] : sim->h_cam_obs, two_buffers && sim->row_parity ? sim->h_rows2[1] : sim->h_tgt_obs};
    float* const rows_before[2] = {two_buffers && !sim->row_parity ? sim->h_rows2[0] : sim->h_cam_obs, two_buffers && !sim->row_parity ? sim->h_rows2[1] : sim->h_tgt_obs};
    // a team without a host buffer has no rows composed on the device either
    p.cam_act = sim->h_cam_act; p.tgt_act = sim->h_tgt_act; p.cam_obs = cam_obs ? rows_now[0] : nullptr; p.tgt_obs = tgt_obs ? rows_now[1] : nullptr;
    p.rewards = sim->h_rewards; p.done = sim->h_done;
    fill_aux(p, nullptr, nullptr);
    // work queued earlier on the legacy default stream (torch's default) or on blocking streams is finished first;
    // callers that use non-blocking streams of their own synchronise them before this call (include/mate_b200.h)
    CUDA_TRY(cudaEventRecord(sim->hevents[0], nullptr));
    for (int i = 0; i < MateSim::kHostStreams; ++i) CUDA_TRY(cudaStreamWaitEvent(sim->hstreams[i], sim->hevents[0], 0));
    const int num_chunks = (B + chunk - 1) / chunk;
    // MATE_STEP_HOST_ROWS_KEPT: the caller's row buffers still hold the rows of the previous call (same buffers, not
    // modified since) and the device still holds them too: only the 64-byte groups that differ cross the link and are
    // rewritten.  Otherwise the all-zero chunks are dropped and every byte of the caller's buffers is written.
    const bool delta = two_buffers && (flags & MATE_STEP_HOST_ROWS_KEPT) && sim->kept_valid && sim->kept_rows[0] == cam_obs && sim->kept_rows[1] == tgt_obs;
    const bool compact = (sim->compact_mode == 1 || (sim->compact_mode == 2 && delta)) && num_chunks <= MateSim::kMaxHostChunks && B % 4 == 0 &&
                         !((uintptr_t)cam_obs & 3) && !((uintptr_t)tgt_obs & 3);
    sim->kept_valid = false;
    if (int rc = compact ? compact_leg(sim, p, chunk, delta, rows_before, cam_act, tgt_act, cam_obs, tgt_obs, rewards, done)
                         : dense_leg(sim, p, chunk, cam_act, tgt_act, cam_obs, tgt_obs, rewards, done))
        return rc;
    if (compact || two_buffers) {   // the caller's buffers and the device hold this call's rows: the next call may send changes only
        sim->kept_rows[0] = cam_obs; sim->kept_rows[1] = tgt_obs; sim->kept_valid = true;
    }
    if (two_buffers) sim->row_parity ^= 1;
    // the prepared episodes are refilled on the side stream like on the device path
    return refill_after_step(sim, flags, nullptr);
}

// ---- state get / set (host arrays, synchronous) --------------------------------------------------
// Both move the whole state block through its host copy (MateSim::host) and convert each field between the
// struct-of-arrays values [row * bpad + env] and the batched rows [B][rows][comps] of a MateStateView.
// The host copy is carved like the device block, so host code reads and writes the state at the device's offsets.  It is
// pinned, since pageable copies of the block made both calls slower than the per-array copies they replace, and made on
// first use, since pinning it in create made create + destroy 17 times as long (MATE-4v8-9 x 65 536, one B200).
static int ensure_host_copy(MateSim* sim) {
    if (sim->host_block) return MATE_OK;
    if (cudaMallocHost(&sim->host_block, sim->state_bytes) != cudaSuccess) {
        cudaGetLastError();
        sim->host_block = nullptr;
        return fail(MATE_ENOMEM, "cudaMallocHost(state copy) failed");
    }
    carve_state(sim->host, (char*)sim->host_block, sim->cfg.num_cameras, sim->cfg.num_targets, sim->cfg.num_obstacles, sim->bpad, false);
    return MATE_OK;
}

extern "C" int mate_b200_get_state(MateSim* sim, MateStateView* v) {
    if (!sim || !v) return fail(MATE_EINVAL, "null argument");
    CUDA_TRY(cudaSetDevice(sim->device));
    CUDA_TRY(cudaDeviceSynchronize());
    if (int rc = ensure_host_copy(sim)) return rc;
    const Params& h = sim->host;
    CUDA_TRY(cudaMemcpy(sim->host_block, sim->state_block, sim->state_bytes, cudaMemcpyDeviceToHost));
    const int nc = sim->cfg.num_cameras, nt = sim->cfg.num_targets, no = sim->cfg.num_obstacles;
    const size_t bp = sim->bpad, B = sim->num_envs;
    for (size_t e = 0; e < B; ++e) {
        for (int r = 0; r < nc; ++r) {
            const size_t s = r * bp + e, i = e * nc + r;
            if (v->cam_xy) { v->cam_xy[2 * i] = h.cam_x[s]; v->cam_xy[2 * i + 1] = h.cam_y[s]; }
            if (v->cam_phi) v->cam_phi[i] = h.cam_phi[s];
            if (v->cam_theta) v->cam_theta[i] = h.cam_theta[s];
        }
        for (int r = 0; r < nt; ++r) {
            const size_t s = r * bp + e, i = e * nt + r;
            if (v->tgt_xy) { v->tgt_xy[2 * i] = h.tgt_x[s]; v->tgt_xy[2 * i + 1] = h.tgt_y[s]; }
            const uint32_t q = h.tgt_pack[s];
            if (v->tgt_capacity) v->tgt_capacity[i] = tp_capacity(q);
            if (v->tgt_goal) v->tgt_goal[i] = tp_goal(q);
            if (v->tgt_weight) v->tgt_weight[i] = tp_weight(q);
            if (v->tgt_bounty) v->tgt_bounty[i] = tp_bounty(q);
            if (v->tgt_empty_bits) v->tgt_empty_bits[i] = tp_empty(q);
        }
        for (int r = 0; r < no; ++r) {
            const size_t s = r * bp + e, i = e * no + r;
            if (v->obs_xyr) { v->obs_xyr[3 * i] = h.obs_x[s]; v->obs_xyr[3 * i + 1] = h.obs_y[s]; v->obs_xyr[3 * i + 2] = h.obs_r[s]; }
        }
        const uint4 c0 = h.cargo[e], c1 = h.cargo[bp + e], a = h.env_a[e];
        const int4 b = h.env_b[e];
        const uint32_t words[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
        if (v->remaining) for (int k = 0; k < 16; ++k) v->remaining[e * 16 + k] = (int32_t)((words[k >> 1] >> ((k & 1) * 16)) & 0xFFFF);
        if (v->awaiting) { v->awaiting[e * 4 + 0] = a.x & 0xFFFF; v->awaiting[e * 4 + 1] = a.x >> 16; v->awaiting[e * 4 + 2] = a.y & 0xFFFF; v->awaiting[e * 4 + 3] = a.y >> 16; }
        if (v->episode_step) v->episode_step[e] = (int32_t)a.z;
        if (v->num_delivered) v->num_delivered[e] = (int32_t)a.w;
        if (v->episode_reward) { v->episode_reward[e * 2] = (double)b.x; v->episode_reward[e * 2 + 1] = (double)b.y; }
        if (v->episode_id) v->episode_id[e] = b.w;
    }
    return MATE_OK;
}

extern "C" int mate_b200_set_state(MateSim* sim, const MateStateView* v) {
    if (!sim || !v) return fail(MATE_EINVAL, "null argument");
    CUDA_TRY(cudaSetDevice(sim->device));
    CUDA_TRY(cudaDeviceSynchronize());
    if (int rc = ensure_host_copy(sim)) return rc;
    const Params& h = sim->host;
    CUDA_TRY(cudaMemcpy(sim->host_block, sim->state_block, sim->state_bytes, cudaMemcpyDeviceToHost));
    const int nc = sim->cfg.num_cameras, nt = sim->cfg.num_targets, no = sim->cfg.num_obstacles;
    const size_t bp = sim->bpad, B = sim->num_envs;
    if (v->cam_theta)
        for (size_t i = 0; i < B * nc; ++i)
            if (!(v->cam_theta[i] > 0.0) || v->cam_theta[i] > 180.0) return fail(MATE_EINVAL, "cam_theta out of (0, 180]");
    // Until the upload below only the host copy changes (each call downloads it afresh): a view refused on the way leaves
    // the handle as it was.
    for (size_t e = 0; e < B; ++e) {
        for (int r = 0; r < nc; ++r) {
            const size_t s = r * bp + e, i = e * nc + r;
            if (v->cam_xy) { h.cam_x[s] = v->cam_xy[2 * i]; h.cam_y[s] = v->cam_xy[2 * i + 1]; }
            if (v->cam_phi) h.cam_phi[s] = v->cam_phi[i];
            if (v->cam_theta) h.cam_theta[s] = v->cam_theta[i];
        }
        for (int r = 0; r < nt; ++r) {
            const size_t s = r * bp + e, i = e * nt + r;
            if (v->tgt_xy) { h.tgt_x[s] = v->tgt_xy[2 * i]; h.tgt_y[s] = v->tgt_xy[2 * i + 1]; }
            const uint32_t q = h.tgt_pack[s];
            const int capacity = v->tgt_capacity ? v->tgt_capacity[i] : tp_capacity(q);
            const int goal = v->tgt_goal ? v->tgt_goal[i] : tp_goal(q);
            const int weight = v->tgt_weight ? v->tgt_weight[i] : tp_weight(q);
            const int bounty = v->tgt_bounty ? v->tgt_bounty[i] : tp_bounty(q);
            const int empty = v->tgt_empty_bits ? v->tgt_empty_bits[i] : tp_empty(q);
            if (capacity < 1 || capacity > 2 || goal < -1 || goal > 3 || weight < 0 || weight > 3 || bounty < 0 || bounty > 65535)
                return fail(MATE_EINVAL, "target integer state out of range");
            h.tgt_pack[s] = pack_target(bounty, goal, weight, capacity, empty, tp_colliding(q));
        }
        for (int r = 0; r < no; ++r) {
            const size_t s = r * bp + e, i = e * no + r;
            if (v->obs_xyr) {
                h.obs_x[s] = v->obs_xyr[3 * i]; h.obs_y[s] = v->obs_xyr[3 * i + 1]; h.obs_r[s] = v->obs_xyr[3 * i + 2];
                h.obs_f4[s] = make_float4((float)h.obs_x[s], (float)h.obs_y[s], (float)h.obs_r[s], 0.f);   // fp32 shadow read by the prefilters and the observation packer
            }
        }
        if (v->cam_xy || v->obs_xyr) h.cc_clear[e] = 0;   // geometry changed: invalidate the per-episode camera line-of-sight cache
        uint4& a = h.env_a[e];
        int4& b = h.env_b[e];
        if (v->remaining) {
            uint32_t words[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            for (int k = 0; k < 16; ++k) words[k >> 1] |= ((uint32_t)v->remaining[e * 16 + k] & 0xFFFF) << ((k & 1) * 16);
            h.cargo[e] = make_uint4(words[0], words[1], words[2], words[3]);
            h.cargo[bp + e] = make_uint4(words[4], words[5], words[6], words[7]);
        }
        if (v->awaiting) {
            a.x = ((uint32_t)v->awaiting[e * 4 + 0] & 0xFFFF) | ((uint32_t)v->awaiting[e * 4 + 1] << 16);
            a.y = ((uint32_t)v->awaiting[e * 4 + 2] & 0xFFFF) | ((uint32_t)v->awaiting[e * 4 + 3] << 16);
        }
        if (v->episode_step) a.z = (uint32_t)v->episode_step[e];
        if (v->num_delivered) a.w = (uint32_t)v->num_delivered[e];
        if (v->episode_reward) { b.x = (int)std::lrint(v->episode_reward[e * 2]); b.y = (int)std::lrint(v->episode_reward[e * 2 + 1]); b.z = 0; }
        if (v->episode_id) b.w = v->episode_id[e];
    }
    CUDA_TRY(cudaMemcpy(sim->state_block, sim->host_block, sim->state_bytes, cudaMemcpyHostToDevice));
    if (sim->refill_mode) CUDA_TRY(cudaMemset(sim->base.ready, 0, sizeof(uint32_t) * sim->bpad));   // prepared episodes may no longer match
    return launch_prepare(sim, nullptr);   // prepare the next episodes of the new state right away
}

// ---- device-side snapshots (mate_snapshot.cuh) ----------------------------------------------------------------------
// The payload of `count` environments: every array of for_each_state_array as rows x count elements ([row * count + i]),
// each section 256-byte aligned, then the 16 floats of `stats`.  With a table the sections are bound to the handle's live
// arrays and to `payload`; table->n counts the arrays even past kSnapMaxArrays.  Returns the payload bytes.
static size_t snapshot_layout(const MateSim* sim, size_t count, char* payload, SnapTable* table) {
    Params p = sim->base;
    size_t off = 0;
    if (table) { *table = SnapTable{}; table->bpad = sim->bpad; table->num_envs = sim->num_envs; table->count = (int)count; table->stats = p.stats; }
    for_each_state_array(p, sim->cfg.num_cameras, sim->cfg.num_targets, sim->cfg.num_obstacles, [&](auto*& ptr, int rows) {
        const size_t elem = sizeof(*ptr);
        if (table && rows > 0) {
            if (table->n < kSnapMaxArrays)
                table->a[table->n] = SnapArray{reinterpret_cast<char*>(ptr), payload + off, rows, (int)elem};
            table->n += 1;
            table->rows += rows;
        }
        off = align_up(off + elem * rows * count, 256);
    });
    if (table) table->payload_stats = reinterpret_cast<float*>(payload + off);
    return off + sizeof(float) * 16;
}

extern "C" int mate_b200_snapshot_bytes(const MateSim* sim, int32_t count, uint64_t* bytes) {
    if (!sim || !bytes) return fail(MATE_EINVAL, "null argument");
    if (count <= 0) return fail(MATE_EINVAL, "count must be positive");
    *bytes = snapshot_layout(sim, (size_t)count, nullptr, nullptr);
    return MATE_OK;
}

extern "C" int mate_b200_save_state(MateSim* sim, const int32_t* env, int32_t count, void* payload, MateSnapshotInfo* info,
                                    void* stream) {
    if (!sim || !payload || !info) return fail(MATE_EINVAL, "null argument");
    if (count <= 0) return fail(MATE_EINVAL, "count must be positive");
    if (!env && count != sim->num_envs) return fail(MATE_EINVAL, "without an environment list the snapshot holds every environment: count must be num_envs");
    if ((uintptr_t)payload & 15) return fail(MATE_EINVAL, "the snapshot payload must be 16-byte aligned");
    SnapTable t;
    const size_t bytes = snapshot_layout(sim, (size_t)count, static_cast<char*>(payload), &t);
    if (t.n > kSnapMaxArrays) return fail(MATE_EINVAL, "more state arrays than the snapshot table holds (kSnapMaxArrays)");
    CUDA_TRY(cudaSetDevice(sim->device));
    snapshot_gather_kernel<<<snapshot_grid(t, count), kSnapThreads, 0, (cudaStream_t)stream>>>(t, env);
    sim->launches += 1;
    if (int rc = check_launch("snapshot gather")) return rc;
    *info = MateSnapshotInfo{};
    info->version = MATE_SNAPSHOT_VERSION;
    info->num_cameras = sim->cfg.num_cameras; info->num_targets = sim->cfg.num_targets; info->num_obstacles = sim->cfg.num_obstacles;
    info->count = count;
    info->config_hash = sim->config_hash;
    info->seed = sim->seed;
    info->payload_bytes = bytes;
    return MATE_OK;
}

extern "C" int mate_b200_load_state(MateSim* sim, const void* payload, const MateSnapshotInfo* info, const int32_t* src,
                                    uint32_t flags, void* stream) {
    if (!sim || !payload || !info) return fail(MATE_EINVAL, "null argument");
    if (info->version != MATE_SNAPSHOT_VERSION) return fail(MATE_EINVAL, "snapshot version " + std::to_string(info->version) + ", this library reads version " + std::to_string(MATE_SNAPSHOT_VERSION));
    if (info->num_cameras != sim->cfg.num_cameras || info->num_targets != sim->cfg.num_targets || info->num_obstacles != sim->cfg.num_obstacles)
        return fail(MATE_EINVAL, "the snapshot is of another shape (cameras, targets, obstacles)");
    if (info->config_hash != sim->config_hash) return fail(MATE_EINVAL, "the snapshot was saved by a handle with another configuration");
    if (info->count <= 0) return fail(MATE_EINVAL, "the snapshot's count must be positive");
    if (flags & ~MATE_LOAD_STATE_RESUME) return fail(MATE_EINVAL, "unknown load flags");
    const bool resume = (flags & MATE_LOAD_STATE_RESUME) != 0;
    if (resume && src) return fail(MATE_EINVAL, "MATE_LOAD_STATE_RESUME restores the whole batch: it takes no map");
    if (!src && info->count != sim->num_envs) return fail(MATE_EINVAL, "without a map the snapshot must hold num_envs environments");
    if ((uintptr_t)payload & 15) return fail(MATE_EINVAL, "the snapshot payload must be 16-byte aligned");
    SnapTable t;
    const size_t bytes = snapshot_layout(sim, (size_t)info->count, static_cast<char*>(const_cast<void*>(payload)), &t);
    if (info->payload_bytes != bytes) return fail(MATE_EINVAL, "the snapshot's payload_bytes do not match its count");
    if (t.n > kSnapMaxArrays) return fail(MATE_EINVAL, "more state arrays than the snapshot table holds (kSnapMaxArrays)");
    t.copy_stats = resume;
    t.ready = sim->refill_mode ? sim->base.ready : nullptr;
    CUDA_TRY(cudaSetDevice(sim->device));
    const cudaStream_t s = (cudaStream_t)stream;
    if (sim->refill_mode == 1) {   // a prepare still running on the side stream writes the tags this load clears
        CUDA_TRY(cudaEventRecord(sim->side_event, sim->side));
        CUDA_TRY(cudaStreamWaitEvent(s, sim->side_event, 0));
    }
    snapshot_scatter_kernel<<<snapshot_grid(t, sim->num_envs), kSnapThreads, 0, s>>>(t, src);
    sim->launches += 1;
    if (int rc = check_launch("snapshot scatter")) return rc;
    if (resume) sim->seed = info->seed;
    return launch_prepare(sim, s);   // fresh prepared episodes for the loaded environments
}

extern "C" int mate_b200_episode_stats(MateSim* sim, float* out16, int32_t reset_after, void* stream) {
    if (!sim || !out16) return fail(MATE_EINVAL, "null argument");
    CUDA_TRY(cudaSetDevice(sim->device));
    CUDA_TRY(cudaMemcpyAsync(out16, sim->base.stats, sizeof(float) * 16, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    if (reset_after) CUDA_TRY(cudaMemsetAsync(sim->base.stats, 0, sizeof(float) * 16, (cudaStream_t)stream));
    return MATE_OK;
}

#ifdef MATE_DEV_TIMELINE   // development builds only (profiles/tools/timeline.py): per-tile phase time stamps of the last step launch
extern "C" int mate_b200_debug_timeline(unsigned long long* out, int32_t count) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpyFromSymbol(out, mate::g_timeline, sizeof(unsigned long long) * (size_t)count));
    return MATE_OK;
}
#endif
