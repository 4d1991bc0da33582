// mate_wrappers.cuh -- the reference's observation wrappers as ONE in-place pass over the joint
// observation tensors (SURVEY.md section 8f, N1).  Restated behaviour (reference root):
//   mate/wrappers/enhanced_observation.py:72-123 (EnhancedObservation.observation),
//   mate/wrappers/shared_field_of_view.py:74-145 (SharedFieldOfView.observation),
//   mate/agents/utils.py:40-94 (convert_coordinates, used by RelativeCoordinates),
//   mate/agents/utils.py:97-127 (normalize_observation, used by RescaledObservation).
//
// The reference applies each wrapper as NumPy slicing on the [N, D] joint observation of ONE environment.
// Here a warp loads the 6 KB block of one environment into shared memory (16-byte coalesced loads),
// applies the requested wrappers in the reference's order, lanes = (observer row, entity slot) pairs, and
// stores the block back: one read and one write of the observation tensors whatever the number of
// stacked wrappers.  The kernel is HBM bound (2 x 407 MB for MATE-4v8-9 x 65 536).
#pragma once

#include <type_traits>

#include "mate_common.cuh"

namespace mate {

template <int NC, int NT, int NO>
struct WShape {
    static constexpr int DC = ObsLayout{NC, NT, NO}.dc(), DT = ObsLayout{NC, NT, NO}.dt();
    static constexpr int CAM_ROW = NC * DC, TGT_ROW = NT * DT;
    static constexpr int BLOCK = CAM_ROW + TGT_ROW;            // floats per environment
    static constexpr int E = NT + NO + NC;                     // entity slots per observer row
    static constexpr int R = NC + NT;
    static constexpr int SCR = 4 * (NO > 0 ? NO : 1) + 2 * E + 8 + 4 * E + 2;   // obstacle entries, shared masks, shared empty bits, fp64 locations
    static constexpr int WARP_FLOATS = ((BLOCK + SCR + 3) / 4) * 4;
    static constexpr int WARPS = 4;
    static constexpr int SMEM_BYTES = (WARPS * WARP_FLOATS + 2 * (DC + DT)) * 4;
    static constexpr bool VEC = (CAM_ROW % 4 == 0) && (TGT_ROW % 4 == 0);
};

// The registered observation wrappers applied IN PLACE to the rows of one environment that a warp holds in shared
// memory: B = camera rows [NC][DC], T = target rows [NT][DT]; `scr` = S::SCR floats of scratch (8-byte aligned).
// Called by all 32 lanes.  Used by obs_transform_kernel (a pass over observation tensors) and by the step kernel's
// packer (mate_step.cuh: the wrappers registered with mate_b200_set_observation_ops cost no extra pass at all).
template <int NC, int NT, int NO>
__device__ __forceinline__ void apply_obs_ops(const Params& p, const ObsOps& ops, const int env, float* B, float* T, float* scr,
                                              const float* aff_cam, const float* aff_tgt) {
    using S = WShape<NC, NT, NO>;
    constexpr int DC = S::DC, DT = S::DT, E = S::E, R = S::R;
    // Entry offsets are L.entry_offset(observer is a camera, kind, index), written as block start + width * index with the
    // block starts as compile-time constants: the call with run-time arguments compiles to different code.
    constexpr ObsLayout L{NC, NT, NO};
    const int lane = threadIdx.x & 31;
    float* ob = scr;                                           // [NO][4] obstacle_states_flagged
    float* shm = ob + 4 * (NO > 0 ? NO : 1);                   // [2][E] shared view masks (camera team, target team)
    float* she = shm + 2 * E;                                  // [4] shared empty bits
    double* pos = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(she + 8) + 7) & ~(uintptr_t)7);   // [E][2] fp64 locations: targets, obstacles, cameras
    for (int o = lane; o < NO; o += 32) {
        const float4 f = p.obs_f4[(size_t)o * p.bpad + env];
        ob[4 * o] = f.x; ob[4 * o + 1] = f.y; ob[4 * o + 2] = f.z; ob[4 * o + 3] = 1.f;
    }
    bool relative_op = false;
    for (int i = 0; i < ops.n; ++i) relative_op = relative_op || ops.op[i] == MATE_OBS_RELATIVE;
    if (relative_op) {
        for (int k = lane; k < E; k += 32) {   // RelativeCoordinates subtracts in fp64 (fp32 would lose ~1e-4 to cancellation)
            const size_t bp = p.bpad;
            double x, y;
            if (k < NT) { x = p.tgt_x[(size_t)k * bp + env]; y = p.tgt_y[(size_t)k * bp + env]; }
            else if (k < NT + NO) { x = p.obs_x[(size_t)(k - NT) * bp + env]; y = p.obs_y[(size_t)(k - NT) * bp + env]; }
            else { x = p.cam_x[(size_t)(k - NT - NO) * bp + env]; y = p.cam_y[(size_t)(k - NT - NO) * bp + env]; }
            pos[2 * k] = x; pos[2 * k + 1] = y;
        }
    }
    __syncwarp();
    auto row_ptr = [&](int r) { return r < NC ? B + r * DC : T + (r - NC) * DT; };
    // Entity kinds with compile-time widths: 0 = target (x, y, sight range, loaded | flag), 1 = obstacle
    // (x, y, r | flag), 2 = camera (x, y, r, Rs cos, Rs sin, theta | flag).  `pairs<K>(r0, n, f)` spreads the
    // (observer row in [r0, r0 + n), entity of kind K) pairs over the lanes and calls
    // f(row pointer, row, entity index, slot offset in that row).
    auto pairs = [&](auto k, const int r0, const int n, auto&& f) {
        constexpr int K = decltype(k)::value;
        constexpr int N = L.count(K), W = ObsLayout::width(K), OC = L.block(true, K), OT = L.block(false, K);
        if constexpr (N > 0) {
        for (int q = lane; q < n * N; q += 32) {
            const int r = r0 + q / (N > 0 ? N : 1), idx = q % (N > 0 ? N : 1);
            const int off = r < NC ? OC + W * idx : OT + W * idx;
            f(row_ptr(r), r, idx, off);
        }
        }
    };
    using K0 = std::integral_constant<int, KIND_TARGET>;
    using K1 = std::integral_constant<int, KIND_OBSTACLE>;
    using K2 = std::integral_constant<int, KIND_CAMERA>;
    // write the public state (+ flag 1) of entity `idx` of kind K, or zeros
    auto fill = [&](auto k, float* dst, const int idx, const bool on) {
        constexpr int K = decltype(k)::value;
        constexpr int W = ObsLayout::width(K);
        const float* src = K == 0 ? T + idx * DT + ObsLayout::SELF : (K == 1 ? ob + 4 * idx : B + idx * DC + ObsLayout::SELF);
#pragma unroll
        for (int j = 0; j < W - 1; ++j) dst[j] = on ? src[j] : 0.f;
        dst[W - 1] = on ? 1.f : 0.f;
    };
    // shm layout: targets [0, NT), obstacles [NT, NT + NO), cameras [NT + NO, E)  (same as `pos`)
    constexpr int SH0 = 0, SH1 = NT, SH2 = NT + NO;

#pragma unroll 1
    for (int i = 0; i < ops.n; ++i) {
        const int op = ops.op[i];
        if (op == MATE_OBS_ENHANCED_CAMERA || op == MATE_OBS_ENHANCED_TARGET || op == MATE_OBS_SHARED_CAMERA || op == MATE_OBS_SHARED_TARGET) {
            const bool cam_team = op == MATE_OBS_ENHANCED_CAMERA || op == MATE_OBS_SHARED_CAMERA;
            const bool shared = op == MATE_OBS_SHARED_CAMERA || op == MATE_OBS_SHARED_TARGET;
            const int r0 = cam_team ? 0 : NC, nrows = cam_team ? NC : NT;
            if (nrows == 0) continue;
            if (shared) {   // "or" of the team's view masks (flag entries), and of the targets' empty bits
                for (int k = lane; k < E; k += 32) {
                    const int kind = k < NT ? 0 : (k < NT + NO ? 1 : 2);
                    const int idx = k < NT ? k : (k < NT + NO ? k - NT : k - NT - NO);
                    constexpr int C0 = L.block(true, KIND_TARGET), C1 = L.block(true, KIND_OBSTACLE), C2 = L.block(true, KIND_CAMERA);
                    constexpr int T0 = L.block(false, KIND_TARGET), T1 = L.block(false, KIND_OBSTACLE), T2 = L.block(false, KIND_CAMERA);
                    const int w = kind == 0 ? ObsLayout::TGT_ENTRY : (kind == 1 ? ObsLayout::OBS_ENTRY : ObsLayout::CAM_ENTRY);
                    const int off = cam_team ? (kind == 0 ? C0 : (kind == 1 ? C1 : C2)) + w * idx
                                             : (kind == 2 ? T2 : (kind == 1 ? T1 : T0)) + w * idx;
                    bool any = cam_team ? kind == 2 : kind == 0;   // teammates are always shared (flag 1)
                    for (int r = 0; r < nrows; ++r) any = any || row_ptr(r0 + r)[off + w - 1] != 0.f;
                    shm[k] = any ? 1.f : 0.f;
                }
                if (!cam_team && lane < NW) {
                    bool any = false;
                    for (int t = 0; t < NT; ++t) any = any || row_ptr(NC + t)[ObsLayout::TGT_EMPTY + lane] != 0.f;
                    she[lane] = any ? 1.f : 0.f;
                }
            } else if (!cam_team && lane < NW) {   // np.logical_not(remaining_cargoes).all(axis=-1)
                const uint4 c0 = p.cargo[env], c1 = p.cargo[(size_t)p.bpad + env];
                const uint32_t w0 = lane == 0 ? c0.x : (lane == 1 ? c0.z : (lane == 2 ? c1.x : c1.z));
                const uint32_t w1 = lane == 0 ? c0.y : (lane == 1 ? c0.w : (lane == 2 ? c1.y : c1.w));
                she[lane] = (w0 | w1) == 0u ? 1.f : 0.f;
            }
            __syncwarp();
            pairs(K0{}, r0, nrows, [&](float* row, int, int idx, int off) { fill(K0{}, row + off, idx, !shared || shm[SH0 + idx] != 0.f); });
            pairs(K1{}, r0, nrows, [&](float* row, int, int idx, int off) { fill(K1{}, row + off, idx, !shared || shm[SH1 + idx] != 0.f); });
            pairs(K2{}, r0, nrows, [&](float* row, int, int idx, int off) { fill(K2{}, row + off, idx, !shared || shm[SH2 + idx] != 0.f); });
            if (!cam_team) {
                for (int q = lane; q < NT * NW; q += 32) row_ptr(NC + q / NW)[ObsLayout::TGT_EMPTY + (q % NW)] = she[q % NW];
            }
            __syncwarp();
        } else if (op == MATE_OBS_RELATIVE) {
            // locations still hold the simulator's values unless a rescale came first: subtract in fp64 from
            // the state (entity - observer), else in place on whatever the entries hold now.  parse_obs_ops refuses
            // RESCALED before RELATIVE, so `exact` always holds; the in-place branch stays only because removing it
            // changes the register allocation of every step kernel, wrapper-free launches included (measured 0.15 -
            // 0.3 % slower on a B200 at 1000 W)
            bool exact = true;
            for (int j = 0; j < i; ++j) exact = exact && ops.op[j] != MATE_OBS_RESCALED;
            auto relative = [&](auto k, float* row, const int r, const int idx, const int off) {
                constexpr int K = decltype(k)::value;
                constexpr int W = ObsLayout::width(K);
                if (row[off + W - 1] == 0.f) return;
                if (exact) {
                    const int ke = (K == 0 ? SH0 : (K == 1 ? SH1 : SH2)) + idx, ko = r < NC ? SH2 + r : r - NC;
                    row[off] = (float)(pos[2 * ke] - pos[2 * ko]); row[off + 1] = (float)(pos[2 * ke + 1] - pos[2 * ko + 1]);
                } else {
                    row[off] -= row[ObsLayout::SELF]; row[off + 1] -= row[ObsLayout::SELF + 1];
                }
            };
            pairs(K0{}, 0, R, [&](float* row, int r, int idx, int off) { relative(K0{}, row, r, idx, off); });
            pairs(K1{}, 0, R, [&](float* row, int r, int idx, int off) { relative(K1{}, row, r, idx, off); });
            pairs(K2{}, 0, R, [&](float* row, int r, int idx, int off) { relative(K2{}, row, r, idx, off); });
            for (int q = lane; q < R * 2 * NW; q += 32) {   // the warehouse locations in the preserved block
                const int r = q / (2 * NW), j = q % (2 * NW);
                float* row = row_ptr(r);
                const int ko = r < NC ? SH2 + r : r - NC;
                constexpr int WH = ObsLayout::WAREHOUSE;
                if (exact) row[WH + j] = (float)((double)row[WH + j] - pos[2 * ko + (j & 1)]);
                else row[WH + j] -= row[ObsLayout::SELF + (j & 1)];
            }
            __syncwarp();
        } else if (op == MATE_OBS_RESCALED) {
            // a lane keeps its columns' (scale, shift) in registers and walks down the rows of a team
            for (int col = lane; col < DC; col += 32) {
                const float sc = aff_cam[2 * col], sh = aff_cam[2 * col + 1];
#pragma unroll
                for (int r = 0; r < NC; ++r) B[r * DC + col] = B[r * DC + col] * sc + sh;
            }
            for (int col = lane; col < DT; col += 32) {
                const float sc = aff_tgt[2 * col], sh = aff_tgt[2 * col + 1];
#pragma unroll
                for (int t = 0; t < NT; ++t) T[t * DT + col] = T[t * DT + col] * sc + sh;
            }
            __syncwarp();
        }
    }
}

template <int NC, int NT, int NO>
__global__ void __launch_bounds__(WShape<NC, NT, NO>::WARPS * 32)
obs_transform_kernel(const __grid_constant__ Params p, const ObsOps ops, const float* __restrict__ cam_affine,
                     const float* __restrict__ tgt_affine) {
    using S = WShape<NC, NT, NO>;
    constexpr int DC = S::DC, DT = S::DT;
    extern __shared__ __align__(16) float wsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* aff = wsm + S::WARPS * S::WARP_FLOATS;              // [DC + DT][2] scale, shift (RescaledObservation)
    bool rescale = false;
    for (int i = 0; i < ops.n; ++i) rescale = rescale || ops.op[i] == MATE_OBS_RESCALED;
    if (rescale) {
        for (int k = threadIdx.x; k < 2 * DC; k += blockDim.x) aff[k] = NC > 0 ? cam_affine[k] : 0.f;
        for (int k = threadIdx.x; k < 2 * DT; k += blockDim.x) aff[2 * DC + k] = tgt_affine[k];
    }
    __syncthreads();
    const int env = blockIdx.x * S::WARPS + warp;
    if (env >= p.num_envs) return;
    float* B = wsm + warp * S::WARP_FLOATS;                    // cam rows, then target rows
    float* cam_g = p.cam_obs + (size_t)env * S::CAM_ROW;
    float* tgt_g = p.tgt_obs + (size_t)env * S::TGT_ROW;
    // ---- load
    if (S::VEC) {
        // all 16-byte loads of the block are issued before the first one is stored to shared memory
        const float4* c4 = reinterpret_cast<const float4*>(cam_g);
        const float4* t4 = reinterpret_cast<const float4*>(tgt_g) - S::CAM_ROW / 4;
        float4* b4 = reinterpret_cast<float4*>(B);
        constexpr int NV = S::BLOCK / 4, NIT = (NV + 31) / 32;
        float4 v[NIT];
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int k = it * 32 + lane;
            if (it * 32 + 32 <= NV || k < NV) v[it] = __ldcs((k < S::CAM_ROW / 4 ? c4 : t4) + k);
        }
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int k = it * 32 + lane;
            if (it * 32 + 32 <= NV || k < NV) b4[k] = v[it];
        }
    } else {
        for (int k = lane; k < S::CAM_ROW; k += 32) B[k] = cam_g[k];
        for (int k = lane; k < S::TGT_ROW; k += 32) B[S::CAM_ROW + k] = tgt_g[k];
    }
    __syncwarp();
    apply_obs_ops<NC, NT, NO>(p, ops, env, B, B + S::CAM_ROW, B + S::BLOCK, aff, aff + 2 * DC);
    // ---- store
    if (S::VEC) {
        float4* c4 = reinterpret_cast<float4*>(cam_g);
        float4* t4 = reinterpret_cast<float4*>(tgt_g) - S::CAM_ROW / 4;
        const float4* b4 = reinterpret_cast<const float4*>(B);
        constexpr int NV = S::BLOCK / 4, NIT = (NV + 31) / 32;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int k = it * 32 + lane;
            if (it * 32 + 32 <= NV || k < NV) (k < S::CAM_ROW / 4 ? c4 : t4)[k] = b4[k];
        }
    } else {
        for (int k = lane; k < S::CAM_ROW; k += 32) cam_g[k] = B[k];
        for (int k = lane; k < S::TGT_ROW; k += 32) tgt_g[k] = B[S::CAM_ROW + k];
    }
}

// DiscreteCamera / DiscreteTarget (mate/wrappers/discrete_action_spaces.py:98-117, 204-228): grid index ->
// continuous action through the wrapper's action table [levels * levels][2]
__global__ void decode_actions_kernel(const int64_t* __restrict__ index, const float* __restrict__ table, int table_size,
                                      float* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long k = index[i];
    k = k < 0 ? 0 : (k >= table_size ? table_size - 1 : k);
    reinterpret_cast<float2*>(out)[i] = reinterpret_cast<const float2*>(table)[k];
}

// Per-agent terms of AuxiliaryCameraRewards / AuxiliaryTargetRewards / MoreTrainingInformation
// (mate/wrappers/auxiliary_camera_rewards.py:140-149, auxiliary_target_rewards.py:135-177,
// more_training_information.py:61-82) from the auxiliary outputs of the last step.  One thread per AGENT (first all
// cameras, then all targets, so that a warp holds one kind): an agent's 8 / 16 output floats leave as two / four
// 16-byte stores, neighbouring threads read neighbouring mask rows.  (Round 1: one thread per environment wrote its
// 160 floats with scalar stores 640 bytes apart.)
__global__ void aux_terms_kernel(const MateStepAux ax, const float* __restrict__ rewards, const float* __restrict__ soft,
                                 float* __restrict__ cam_terms, float* __restrict__ tgt_terms, int num_envs, int nc, int nt) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long num_cam = (long long)num_envs * nc, num_tgt = (long long)num_envs * nt;
    if (i >= num_cam + num_tgt) return;
    if (i < num_cam) {
        const int e = (int)(i / nc), c = (int)(i - (long long)e * nc);
        int num_tracked = 0, sensed = 0;
        float soft_sum = 0.f, soft_max = -3.0e38f;   // auxiliary_camera_rewards.py:130-138
        for (int t = 0; t < nt; ++t) {
            const int seen = ax.mask_ct[(size_t)i * nt + t] != 0;
            num_tracked += seen;
            sensed |= ax.mask_tc[((size_t)e * nt + t) * nc + c] != 0;
            if (soft) {
                const float v = soft[(size_t)i * nt + t];
                soft_sum += seen ? v : 0.f;
                soft_max = fmaxf(soft_max, v);
            }
        }
        float4* q = reinterpret_cast<float4*>(cam_terms + (size_t)i * MATE_CAM_TERMS);
        q[0] = make_float4(rewards[(size_t)e * 2], ax.coverage[(size_t)e * 3], ax.coverage[(size_t)e * 3 + 1], ax.coverage[(size_t)e * 3 + 2]);
        q[1] = make_float4(soft ? (num_tracked > 0 ? soft_sum : tanhf(soft_max)) : 0.f, (float)num_tracked, 1.f, (float)sensed);
        return;
    }
    const long long k = i - num_cam;          // (environment, target)
    const int e = (int)(k / nt), t = (int)(k - (long long)e * nt);
    bool tracked = false;                     // some camera sees target t
    float soft_sum = 0.f, soft_max = -3.0e38f;
    for (int c = 0; c < nc; ++c) {
        const size_t j = ((size_t)e * nc + c) * nt + t;
        const bool seen = ax.mask_ct[j] != 0;
        tracked = tracked || seen;
        if (soft) {
            const float v = soft[j];
            soft_sum += seen ? v : 0.f;
            soft_max = fmaxf(soft_max, v);
        }
    }
    const int goal = ax.tgt_goal[k], empty = ax.tgt_empty_bits[k];
    const float4 dist = reinterpret_cast<const float4*>(ax.warehouse_dist)[k];
    float wd[NW] = {fmaxf(dist.x - (float)kWarehouseRadius, 0.f), fmaxf(dist.y - (float)kWarehouseRadius, 0.f),
                    fmaxf(dist.z - (float)kWarehouseRadius, 0.f), fmaxf(dist.w - (float)kWarehouseRadius, 0.f)};
    float nearest_open = (float)kTerrain;     // TERRAIN_WIDTH / 2 when every warehouse is known to be empty
    bool any_open = false;
    float at_goal = 0.f;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        if (!((empty >> w) & 1)) { nearest_open = any_open ? fminf(nearest_open, wd[w]) : wd[w]; any_open = true; }
        at_goal = goal == w ? wd[w] : at_goal;
    }
    const float goal_distance = goal >= 0 ? at_goal : nearest_open;               // auxiliary_target_rewards.py:143-149
    const float info_goal_distance = goal >= 0 ? at_goal : (float)kTerrain;       // more_training_information.py:72
    const float soft_t = (soft && nc > 0) ? (tracked ? soft_sum : tanhf(soft_max)) : 0.f;   // auxiliary_target_rewards.py:151-162
    float4* q = reinterpret_cast<float4*>(tgt_terms + (size_t)k * MATE_TGT_TERMS);
    q[0] = make_float4(rewards[(size_t)e * 2 + 1], ax.coverage[(size_t)e * 3], ax.coverage[(size_t)e * 3 + 1], ax.coverage[(size_t)e * 3 + 2]);
    q[1] = make_float4(goal_distance / (float)(2.0 * kTerrain), (float)(ax.target_dones[k] != 0), soft_t, (float)tracked);
    q[2] = make_float4((float)(ax.is_colliding[k] != 0), 1.f, (float)goal, info_goal_distance);
    q[3] = make_float4(wd[0], wd[1], wd[2], wd[3]);
}

// =============================================================================================
// AuxiliaryCameraRewards.compute_soft_coverage_scores (mate/wrappers/auxiliary_camera_rewards.py:182-233):
// signed distance of every target to the boundary of the camera's field of view, in units of the radius of the
// sector's inscribed circle.  The boundary is the OUTER sampled polyline of the camera
// (Camera.add_obstacles / boundary_between(outer=True), mate/entities.py:362-479, 484-511) restricted to the
// current sector, plus the two sector edges (end points from the inner polyline, 16 points along each edge).
// Like the inner polyline it is never materialised: one warp per (environment, camera) enumerates the sample rays
// (integer-degree grid; per obstacle the lattice at max_rho and the two 21-point edge segments), one per lane, keeps
// those inside the sector, cuts each at the FAR side of the discs it crosses (Obstacle.obstruct(outer=True),
// entities.py:158-184; the discs sit in shared memory, a bearing test rejects the ones a ray cannot cross) and keeps,
// per target, the minimum squared distance in registers.
// Exactly tangent rays are not cut by their own disc (the reference decides them by rounding noise, DESIGN.md
// "Tangent rays").  Environments that were auto-reset in the last step get zeros (their state already belongs to
// the next episode).
// =============================================================================================
// Pre-pass of the soft coverage: the ranges of the inner polyline at the two sector edges of every camera
// (boundary_between uses sight_range_at for its first and last point, entities.py:507-511, 536-541), one THREAD per
// (environment, camera, side).  Inside the warp-per-camera kernel below this scalar routine (~3000 dependent fp64
// instructions) was executed by all 32 lanes for two values and set the kernel's time: 5.9 ms at 65 536 environments.
template <int NC, int NO>
__global__ void soft_edges_kernel(const Params p, const uint8_t* __restrict__ done, double* __restrict__ edges) {
    constexpr int NCX = NC > 0 ? NC : 1;
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // ((environment, camera), side)
    if (q >= (long long)p.num_envs * NCX * 2) return;
    const int side = (int)(q & 1);
    const long long item = q >> 1;
    const int e = (int)(item / NCX), c = (int)(item - (long long)e * NCX);
    if (done != nullptr && done[e] != 0) { edges[q] = 0.0; return; }
    const size_t bp = p.bpad;
    const double cx = p.cam_x[(size_t)c * bp + e], cy = p.cam_y[(size_t)c * bp + e];
    const double phi = p.cam_phi[(size_t)c * bp + e], theta = p.cam_theta[(size_t)c * bp + e];
    const double left = normalize_angle(phi - theta * 0.5);
    const double a = normalize_angle(side ? left + theta : left);
    double rho = p.cam_rmax;
    if (NO > 0) {
        bool collapsed = false;   // the camera inside a disc of its set: every ray has norm 0 (entities.py:378-388)
        for (int o = 0; o < NO; ++o) {
            const double ox = p.obs_x[(size_t)o * bp + e] - cx, oy = p.obs_y[(size_t)o * bp + e] - cy, orad = p.obs_r[(size_t)o * bp + e];
            const double od = sqrt(ox * ox + oy * oy);
            collapsed = collapsed || (od < p.cam_rmax + orad && orad > od);
        }
        double sn, cs;
        sincospi(a * (1.0 / 180.0), &sn, &cs);
        rho = collapsed ? 0.0 : sight_range_at<NO>(ObsRef{p.obs_x + e, p.obs_y + e, p.obs_r + e, bp}, cx, cy, p.cam_rmax, a, cs, sn);
    }
    edges[q] = rho;
}

// Far side of disc (rx, ry, R, d) on the ray of bearing `a` (degrees), exactly as the reference evaluates it
// (Obstacle.obstruct(outer=True), entities.py:158-184) in fp64; < 0: the ray is not cut.  Only reached by the rays the
// fp32 evaluation below finds within 1e-4 R of tangency.
__device__ __noinline__ double soft_cut_exact(double rx, double ry, double R, double d, double a) {
    double sn, cs;
    sincospi(a * (1.0 / 180.0), &sn, &cs);
    const double proj = rx * cs + ry * sn;
    if (proj < 0.0) return -1.0;
    const double cosv = fmin(1.0, proj / d);
    const double perp = d * sqrt(fmax(1.0 - cosv * cosv, 0.0));
    if (!(R > perp * (1.0 + 1e-9))) return -1.0;
    return fmax(0.0, d * cosv + sqrt(fmax(R * R - perp * perp, 0.0)));
}

// Round 2: every sample is classified in fp64 (its bearing, the sector test: a handful of adds and compares) but
// EVALUATED in fp32.  A cut is computed from the ray's bearing RELATIVE to the disc (beta = a - bearing of the disc, an
// exact fp64 difference of a few degrees: perp = d sin(beta), proj = d cos(beta)), which keeps the relative precision
// of fp32 where the absolute formulation (ray direction against a centre 1000 units away) loses the near-tangent
// chords; rays within 1e-4 R of tangency take the fp64 expression of the reference.  Only the discs whose angular
// extent meets the sector can cut a sample inside the sector: the cut loop walks that compact list (1-3 discs instead
// of the 9 of the obstacle set), behind an fp32 bearing test.  The three kinds of samples (grid rays, per-disc lattice
// rays / edge points, sector-edge points) share one dense index space: 32 per pass whatever their kind.
template <int NC, int NT, int NO>
__global__ void __launch_bounds__(128, 8)
soft_coverage_kernel(const Params p, const uint8_t* __restrict__ mask_ct, const uint8_t* __restrict__ done,
                     const double* __restrict__ edges, float* __restrict__ out) {
    constexpr int NCX = NC > 0 ? NC : 1, NOX = NO > 0 ? NO : 1;
    constexpr uint32_t FULL = 0xffffffffu;
    constexpr int WARPS = 4;   // launch: 128 threads per block
    // per warp: the RELEVANT discs of the camera's obstacle set (those whose angular extent meets the sector), compacted,
    // relative to the camera; read by all lanes (mostly broadcast)
    __shared__ double sdisc64[WARPS][NOX][6];    // x, y, R, distance, bearing (deg), half opening angle (deg)
    __shared__ float sdisc32[WARPS][NOX][13];    // distance, R, half opening angle, near_rho, {near x, near y, far x, far y} x {left, right}, bearing
    __shared__ int soffs[WARPS][NOX + 1];        // prefix sums of their sample counts
    const int lane = threadIdx.x & 31, wslot = (threadIdx.x >> 5) & (WARPS - 1);
    double (*disc)[6] = sdisc64[wslot];
    float (*fdisc)[13] = sdisc32[wslot];
    int* offs = soffs[wslot];
    const long long item = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // (environment, camera)
    if (item >= (long long)p.num_envs * NCX) return;
    const int e = (int)(item / NCX), c = (int)(item - (long long)e * NCX);
    float* const row = out + ((size_t)e * NCX + c) * NT;
    if (done != nullptr && done[e] != 0) {
        if (lane < NT) row[lane] = 0.f;
        return;
    }
    const size_t bp = p.bpad;
    const double cx = p.cam_x[(size_t)c * bp + e], cy = p.cam_y[(size_t)c * bp + e];
    const double phi = p.cam_phi[(size_t)c * bp + e], theta = p.cam_theta[(size_t)c * bp + e];
    const double rmax = p.cam_rmax;
    const float rmax32 = (float)rmax;
    // sector (boundary_between, entities.py:484-511)
    const double left = normalize_angle(phi - theta * 0.5), right = left + theta;
    const bool wraps = right > 180.0;
    auto in_sector = [&](const double a) {
        return wraps ? (a > left || a < right - 360.0 || a == -180.0) : (a > left && a < right);
    };
    // the camera's obstacle set (entities.py:363-368), one disc per lane; its samples: lattice rays at max_rho and the
    // two 21-point edge segments (entities.py:419-448), only for the discs that reach into the sector
    bool member = false, inside_disc = false;
    int my_count = 0;
    double ox = 0.0, oy = 0.0, orad = 0.0, od = 0.0, ang = 0.0, half = 0.0;
    if (lane < NO) {
        ox = p.obs_x[(size_t)lane * bp + e] - cx; oy = p.obs_y[(size_t)lane * bp + e] - cy; orad = p.obs_r[(size_t)lane * bp + e];
        od = sqrt(ox * ox + oy * oy);
        member = od < rmax + orad;
        inside_disc = member && orad > od;
        // cheap rejection before the fp64 atan2 / asin: a disc farther than 90 + theta / 2 degrees from the sector axis (+ its
        // own half opening angle, at most 90 where the camera is outside) cannot meet the sector when its centre lies behind
        if (member && !inside_disc) {
            ang = atan2(oy, ox) * kRad2Deg; half = asin(orad / od) * kRad2Deg;
            // angular distance between the disc's bearing and the sector axis vs. the two half widths (+ slack)
            if (!(fabs(normalize_angle(ang - phi)) > half + theta * 0.5 + 0.02)) {
                const int two_half = (int)(2.0 * half);
                my_count = (two_half > 16 ? two_half : 16) + 1 + 42;
            }
        }
    }
    const bool collapsed = __any_sync(FULL, inside_disc);   // entities.py:378-388: every ray has norm 0
    if (collapsed) my_count = 0;
    const uint32_t relevant = __ballot_sync(FULL, my_count > 0);
    const int nrel = __popc(relevant);
    int incl = my_count;    // inclusive scan over the lanes
#pragma unroll
    for (int sh = 1; sh < 32; sh <<= 1) {
        const int up = __shfl_up_sync(FULL, incl, sh);
        if (lane >= sh) incl += up;
    }
    if (my_count > 0) {
        const int r = __popc(relevant & ((1u << lane) - 1u));
        offs[r] = incl - my_count;
        disc[r][0] = ox; disc[r][1] = oy; disc[r][2] = orad; disc[r][3] = od; disc[r][4] = ang; disc[r][5] = half;
        float* fd = fdisc[r];
        fd[0] = (float)od; fd[1] = (float)orad; fd[2] = (float)half; fd[12] = (float)ang;
        // the two edge segments: from near_rho on the tangent to rmax 0.01 degrees beside it
        const float near_rho = (float)fmin(rmax, sqrt(od * od + orad * orad));
        fd[3] = near_rho;
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const double edge = side ? ang + half : ang - half, far_angle = side ? ang + half + 0.01 : ang - half - 0.01;
            float ns, nc_, fs, fc;
            sincospif((float)(normalize_angle(edge) * (1.0 / 180.0)), &ns, &nc_);
            sincospif((float)(normalize_angle(far_angle) * (1.0 / 180.0)), &fs, &fc);
            fd[4 + 4 * side] = near_rho * nc_; fd[5 + 4 * side] = near_rho * ns;
            fd[6 + 4 * side] = rmax32 * fc; fd[7 + 4 * side] = rmax32 * fs;
        }
    }
    const int total_disc = __shfl_sync(FULL, incl, 31);
    __syncwarp();
    // the boundary points and the distances of the targets to them (relative to the camera, at most ~4000 units) in
    // fp32: the score is a float32 and loses < 1e-5 of dist_max here
    float tx[NT], ty[NT], best[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        tx[t] = (float)(p.tgt_x[(size_t)t * bp + e] - cx); ty[t] = (float)(p.tgt_y[(size_t)t * bp + e] - cy);
        best[t] = 3.0e38f;
    }
    const float rho_l = (float)edges[item * 2], rho_r = (float)edges[item * 2 + 1];   // soft_edges_kernel
    // (a) the integer-degree grid (entities.py:339-342): only the degrees inside the sector are enumerated
    const int k_first = (int)floor(left) - 1;                 // a little more than the open interval (left, right); in_sector decides
    int count_grid = (int)ceil(theta) + 3;
    if (count_grid > 360) count_grid = 360;                   // every degree at most once
    // (c) the two sector edges: 16 points from the camera to the end point + the end point, per side
    const int total = count_grid + total_disc + 34;
    constexpr float kTan = 1.7453292431e-4f;   // tan(0.01 deg): the 0.01 degrees between the two ends of an edge segment
    for (int s0 = 0; s0 < total; s0 += 32) {
        const int s = s0 + lane;
        bool live = s < total;
        double a = 0.0;            // bearing of the sample, degrees in [-180, 180)
        float n = 0.f, cs = 1.f, sn = 0.f;
        int skip = -1;             // the disc a tangent ray / an edge point belongs to: it does not cut its own samples
        bool cut = true;
        if (s < count_grid) {
            int k = k_first + s;                                   // integer degree, may run past +180
            if (k >= 180) k -= 360;
            a = (double)k;
            live = live && in_sector(a);
            sincospif((float)k * (1.0f / 180.0f), &sn, &cs);
            n = rmax32;
        } else if (s < count_grid + total_disc) {
            const int sidx = s - count_grid;
            int o = 0;
            while (o + 1 < nrel && offs[o + 1] <= sidx) ++o;
            const int j = sidx - offs[o];
            const double ang_o = disc[o][4], half_o = disc[o][5];
            const double aL = ang_o - half_o, aR = ang_o + half_o;
            const int two_half = (int)(2.0 * half_o);
            const int nlat = two_half > 16 ? two_half : 16;
            const float* fd = fdisc[o];
            if (j <= nlat) {        // lattice ray
                const double step = (aR - aL) / (double)nlat;   // np.linspace
                a = normalize_angle(j >= nlat ? aR : ((double)j * step + aL));
                sincospif((float)(a * (1.0 / 180.0)), &sn, &cs);
                n = fminf(rmax32, fd[0] + fd[1]);
                if (j == 0 || j == nlat) skip = o;               // exactly tangent to its own disc
            } else {                // point k of an edge segment
                const int q = j - nlat - 1;
                const int side = q >= 21 ? 1 : 0, k = side ? q - 21 : q;
                const float t = k >= 20 ? 1.0f : (float)k * 0.05f;
                const float vx = (1.0f - t) * fd[4 + 4 * side] + t * fd[6 + 4 * side];
                const float vy = (1.0f - t) * fd[5 + 4 * side] + t * fd[7 + 4 * side];
                const float inv = rsqrtf(vx * vx + vy * vy);
                n = 1.0f / inv;
                cs = vx * inv; sn = vy * inv;
                // bearing of the point: the tangent's bearing plus the (tiny) angle between the segment's near end and the
                // point, t rmax sin(0.01 deg) / ((1 - t) near_rho + t rmax cos(0.01 deg)) radians to 1e-8 relative
                const float delta = __fdividef(t * rmax32 * kTan, (1.0f - t) * fd[3] + t * rmax32) * (float)kRad2Deg;
                a = normalize_angle(side ? aR + (double)delta : aL - (double)delta);
                skip = o;
            }
            live = live && in_sector(a);
        } else {
            const int q = s - count_grid - total_disc;
            const bool is_right = q >= 17;
            const int k = is_right ? q - 17 : q;          // k = 16: the end point itself
            const float rho = is_right ? rho_r : rho_l;
            sincospif((float)((is_right ? right : left) * (1.0 / 180.0)), &sn, &cs);
            n = k >= 16 ? rho : (float)k * (rho * 0.0625f);
            cut = false;
        }
        if (!live) continue;
        if (collapsed && cut) n = 0.f;
        // cut at the far side of the discs the ray crosses (Obstacle.obstruct(outer=True))
        if (cut && n > 0.f) {
            const float a32 = (float)a;
#pragma unroll 1
            for (int o = 0; o < nrel; ++o) {
                const float* fd = fdisc[o];
                float coarse = fabsf(a32 - fd[12]);
                coarse = coarse > 180.f ? 360.f - coarse : coarse;
                if (coarse > fd[2] + 2e-3f || o == skip) continue;      // the ray passes beside the disc
                const float d = fd[0], R = fd[1];
                if (d >= n + R) continue;
                double beta = fabs(a - disc[o][4]);
                beta = beta > 180.0 ? 360.0 - beta : beta;
                float sb, cb;
                sincospif((float)beta * (1.0f / 180.0f), &sb, &cb);
                const float perp = d * sb, proj = d * cb;
                if (proj < 0.f) continue;
                const float margin = R - perp;
                float far_side;
                if (fabsf(margin) < 1e-4f * R) {
                    const double f64 = soft_cut_exact(disc[o][0], disc[o][1], disc[o][2], disc[o][3], a);
                    if (f64 < 0.0) continue;
                    far_side = (float)f64;
                } else {
                    if (!(margin > 0.f)) continue;
                    far_side = proj + sqrtf(margin * (R + perp));
                }
                n = fminf(n, far_side);
            }
        }
        const float px = n * cs, py = n * sn;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const float dx = tx[t] - px, dy = ty[t] - py;
            best[t] = fminf(best[t], dx * dx + dy * dy);
        }
    }
#pragma unroll
    for (int t = 0; t < NT; ++t) {
#pragma unroll
        for (int sh = 16; sh >= 1; sh >>= 1) best[t] = fminf(best[t], __shfl_xor_sync(FULL, best[t], sh));
    }
    // one target per lane: the signed distance in units of the radius of the sector's inscribed circle
    if (lane < NT) {
        const double sight_range = sqrt(p.cam_area_product / theta);
        double sn_h, cs_h;
        sincospi(theta * (0.5 / 180.0), &sn_h, &cs_h);
        const double dist_max = theta < 180.0 ? sight_range / (1.0 + 1.0 / sn_h) : sight_range * 0.5;
        float mine = best[0];
#pragma unroll
        for (int t = 1; t < NT; ++t) mine = lane == t ? best[t] : mine;
        const double dist = (double)sqrtf(mine);
        const bool tracked = mask_ct[((size_t)e * NCX + c) * NT + lane] != 0;
        row[lane] = (float)((tracked ? dist : -dist) / dist_max);
    }
}

}  // namespace mate
