// mate_step.cuh -- fused per-step kernel of the B200-native MultiAgentTracking simulator
// (second generation: one LANE per environment for the simulation, one WARP per environment
// for the observation rows).
//
// One launch per env.step.  Reference behaviour being restated (paths relative to the
// reference root): mate/environment.py:590-676 (step), :1271-1388 (_assign_goals / _simulate /
// _update_view), :908-983 (joint_observation), :679-834 (reset); mate/entities.py:158-184
// (obstruct), :347-360 (Camera.simulate), :362-511 (FOV polyline + perceive), :645-668
// (Target.simulate).
//
// Mapping (sm_100a; nothing here is a contraction, so no tensor cores):
//   * A warp owns 32 consecutive environments and never synchronises with other warps.
//   * SIMULATE / VIEW / GOALS: lane l owns environment env0 + l.  With struct-of-arrays state
//     every warp-wide load or store of one field is one fully used 256-byte segment, and the
//     ~250 distance / sector predicates of an environment run without a single idle lane (the
//     first generation gave a group of 8 lanes to an environment and idled half of them).
//     Predicates are decided in fp32 on squares with a guard band; inside the band the fp64
//     expression of the reference decides (out of line, state re-read from HBM/L2).
//   * Divergent work is not executed where it arises but queued and executed densely:
//       - (camera, target) pairs that pass the range + sector test go to a per-warp queue in
//         shared memory; the warp then processes 32 pairs at a time, one per lane (transmittance
//         draw, conservative occlusion classification, exact polyline only when undecided);
//       - targets whose step may touch a disc are re-simulated in fp64 after the fast loop;
//       - targets standing in a warehouse are handled one per lane and iteration.
//   * OBSERVATIONS: the warp walks over its 32 environments; for each, the lanes are (observer row,
//     entity) PAIRS: a pair writes the entity's public state + flag into the staged row if the observer's
//     mask bit is set and zeros otherwise, every float of the block exactly once, and the finished block
//     leaves the SM with 16-byte streaming stores (bulk copies were slower here, see DESIGN.md).  Masks (one or
//     two words per observer row) and the fp32 entity values are handed from the simulation phase to this phase
//     through shared memory.
#pragma once

#include <cuda_fp16.h>

#include <type_traits>

#include "mate_common.cuh"
#include "mate_wrappers.cuh"

namespace mate {

constexpr int kRollCamerasFrom = 5;   // from this many cameras on, the loop over the observing camera of Camera.perceive stays rolled (instruction cache)
constexpr int kStepMinCtas = 8;       // caps registers at 128 (4 warps per SM sub-partition); 65 536 envs = 2048 warp tiles = 13.8 per SM -> one wave

#ifdef MATE_DEV_TIMELINE   // development builds only: per-tile phase time stamps (profiles/tools/timeline.py)
__device__ unsigned long long g_timeline[4096 * 8];
__device__ __forceinline__ void tl_mark(const int env0, const int k) {
    if ((threadIdx.x & 31) == 0 && (env0 >> 5) < 4096) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        g_timeline[(env0 >> 5) * 8 + k] = t;
    }
}
#define TL_MARK(k) tl_mark(env0, k)
#else
#define TL_MARK(k)
#endif

template <int NC, int NT, int NO>
struct Shape2 {
    static constexpr int DC = ObsLayout{NC, NT, NO}.dc(), DT = ObsLayout{NC, NT, NO}.dt();
    static constexpr int CAM_ROW = NC * DC, TGT_ROW = NT * DT; // floats per environment
    static constexpr int R = NC + NT;                          // observer rows per environment
    // mask words per observer row: word 0 = cameras (bits 0-7), targets (bits 8-15) and, when
    // they fit, obstacles (bits 16-31); otherwise obstacles take a second word
    static constexpr int MW = NO <= 16 ? 1 : 2;
    static constexpr int MSTRIDE = (R * MW) | 1;               // odd stride: lane-per-env access is conflict free
    // fp32 values per environment: targets {x, y, packed state}, cameras {x, y, theta, Rs cos phi, Rs sin phi}
    // (the observation packer and the fp32 prefilters read the same entries)
    static constexpr int CV = 5;
    static constexpr int V_T = 0, V_C = 3 * NT, VN = 3 * NT + CV * NC;
    static constexpr int VSTRIDE = VN | 1;
    // Camera rows whose length is a multiple of 32 floats (MATE-4v2-9: 96) would all start at the same shared-memory bank
    // and every scatter store of the packer would be a 4-way conflict: such rows are staged 4 floats apart (plain packer)
    static constexpr int CAM_SKEW = (NC > 1 && DC % 32 == 0) ? 4 : 0;
    static constexpr int STAGE_CAM = ((NC * (DC + CAM_SKEW) + 3) / 4) * 4;
    static constexpr int STAGE_FLOATS = STAGE_CAM + ((TGT_ROW + 3) / 4) * 4;
    static constexpr bool DENSE16 = (CAM_ROW % 4 == 0) && (TGT_ROW % 4 == 0);   // both teams' float32 rows of an env are 16-byte multiples
    static constexpr int E = NT + NO + NC;                     // entity slots (lanes of the scatter)
    // Obstacle slots of the packer: a slot is 4 floats, a row's slots are contiguous, and scalar stores of lanes 16 bytes
    // apart are 4-way bank conflicts.  Observer rows are therefore grouped by the ALIGNMENT of their obstacle block
    // (16 bytes / 8 bytes / odd) into rounds of 32 / NO rows, and a round stores with the widest aligned type
    // (1, 2 or 3 instructions instead of 4) -- unless the grouping needs more than one round more than plain row order.
    // Only the observer rows [r0, r1) that the launch composes take part.
    struct ORounds { int n; int grouped; int row[40][4]; int cls[40]; };   // cls: 0 = 16-byte aligned, 2 = 8-byte, 1 = odd, -1 = mixed (scalar stores)
    __host__ __device__ static constexpr int o_offset(int row) {
        return (row < NC ? row * (DC + CAM_SKEW) : STAGE_CAM + (row - NC) * DT) + ObsLayout{NC, NT, NO}.block(row < NC, KIND_OBSTACLE);
    }
    __host__ __device__ static constexpr ORounds make_orounds(const int r0, const int r1) {
        ORounds r{};
        const int rpr = NO > 0 ? 32 / NO : 1, plain = (r1 - r0 + rpr - 1) / rpr;
        for (int i = 0; i < 40; ++i) { r.cls[i] = -1; for (int j = 0; j < 4; ++j) r.row[i][j] = -1; }
        if (NO == 0) { r.n = 0; return r; }
        const int order[3] = {0, 2, 1};
        int n = 0;
        for (int k = 0; k < 3; ++k) {
            int fill = 0;
            for (int row = r0; row < r1; ++row) {
                const int al = o_offset(row) & 3, cls = al == 0 ? 0 : (al == 2 ? 2 : 1);
                if (cls != order[k]) continue;
                if (fill == 0) r.cls[n] = cls;
                r.row[n][fill++] = row;
                if (fill == rpr) { fill = 0; ++n; }
            }
            if (fill > 0) ++n;
        }
        if (n <= plain + 1) { r.n = n; r.grouped = 1; return r; }
        for (int i = 0; i < 40; ++i) { r.cls[i] = -1; for (int j = 0; j < 4; ++j) r.row[i][j] = -1; }
        for (int row = r0; row < r1; ++row) r.row[(row - r0) / rpr][(row - r0) % rpr] = row;
        r.n = plain;
        return r;
    }
    static constexpr int WARPS = 2;   // warps per CTA (warps are independent; this only sets the CTA granularity)
    static constexpr int ENVS_PER_CTA = WARPS * 32;
    static constexpr int QCAP = 64;
    static constexpr int OFF_STAGE = 0;
    static constexpr int OFF_MASK = OFF_STAGE + STAGE_FLOATS * 4;
    static constexpr int OFF_VAL = OFF_MASK + 32 * MSTRIDE * 4;
    static constexpr int OFF_Q = OFF_VAL + 32 * VSTRIDE * 4;
    static constexpr int OFF_Q2 = OFF_Q + QCAP * 2;             // second queue: pairs that need the exact polyline
    static constexpr int WARP_BYTES = ((OFF_Q2 + QCAP * 2 + 15) / 16) * 16;
    // scratch of the observation wrappers folded into the packer (apply_obs_ops), behind the block, only when some are registered
    static constexpr int FOLD_SCR = 4 * (NT + NO + NC) + R * MW + 1 + 2 * ObsLayout::AFF_COLS;   // fp64 locations, mask words, (scale, shift) of the own-row columns
    static constexpr int OPS_FLOATS = WShape<NC, NT, NO>::SCR > FOLD_SCR ? WShape<NC, NT, NO>::SCR : FOLD_SCR;
    static constexpr int OPS_BYTES = ((OPS_FLOATS * 4 + 15) / 16) * 16;
    static constexpr int SMEM_BYTES = WARPS * WARP_BYTES;
};

// mask bit positions inside an observer row
__device__ __forceinline__ constexpr uint32_t bit_cam(int c) { return 1u << c; }
__device__ __forceinline__ constexpr uint32_t bit_tgt(int t) { return 1u << (8 + t); }

// The exact (fp64) paths read the discs of an environment from arrays nobody else touches in a step: a
// DRAM round trip for a handful of lanes.  The lines are requested as soon as it is known that an
// environment will take such a path (a target within reach of a disc, a pair the classification left open).
template <int NO>
__device__ __forceinline__ void prefetch_discs64(const Params& p, int er) {
    const size_t bp = p.bpad;
#pragma unroll
    for (int o = 0; o < NO; ++o) {
        const size_t i = (size_t)o * bp + er;
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p.obs_x + i));
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p.obs_y + i));
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p.obs_r + i));
    }
}

// ---- out-of-line exact (fp64) decisions, state re-read from global memory -------------------
// ||a - b|| <= thr (or <), entities a / b given by their SoA rows.  The sum of squares is not contracted into an FMA, like
// fov_reach_test: a partner exactly at the sight range is decided by the rounding of the C oracle.
__device__ __noinline__ bool sense_exact(const double* ax, const double* ay, const double* bx, const double* by,
                                         double thr, bool strict) {
    const double ex = *ax - *bx, ey = *ay - *by;
    const double d2 = __dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), t2 = thr * thr;
    return strict ? dist_lt(d2, thr, t2 * (1.0 - 1e-12), t2 * (1.0 + 1e-12)) : dist_le(d2, thr, t2 * (1.0 - 1e-12), t2 * (1.0 + 1e-12));
}

// Camera.perceive range + sector test in the reference's arithmetic for camera c of env `er`
__device__ __noinline__ int fov_reach_global(const Params& p, int er, int c, const double* qx, const double* qy) {
    const size_t i = (size_t)c * p.bpad + er;
    const double theta = p.cam_theta[i];
    return fov_reach_exact(p.cam_x[i], p.cam_y[i], p.cam_phi[i], theta, sqrt(p.cam_area_product / theta), *qx, *qy);
}

// fp32 prefilter of the same test: 0 = no, 1 = yes, 2 = inside the guard band (ask the fp64 version).
// (hx, hy) = Rs (cos phi, sin phi) is the heading scaled by the sensing radius, rs2 = Rs^2, ch2 = cos^2(theta/2);
// every term of the sector test is scaled by Rs^2, which leaves the decisions unchanged.
__device__ __forceinline__ int fov_reach32(float cx, float cy, float rs2, float hx, float hy, float ch2, float qx, float qy) {
    const float relx = qx - cx, rely = qy - cy;
    const float d2 = relx * relx + rely * rely;
    if (d2 > rs2 * (1.0f + 4e-5f)) return 0;
    const float dot = relx * hx + rely * hy;
    const float sq = dot >= 0.0f ? dot * dot : -(dot * dot);
    const float diff = sq - d2 * ch2 * rs2;       // >= 0  <=>  angle(rel, heading) <= theta / 2
    const float band = (4e-5f * d2 + 1e-3f) * rs2;
    if (diff < -band) return 0;
    if (diff > band && d2 < rs2 * (1.0f - 4e-5f)) return 1;
    return 2;
}

// Target.simulate (entities.py:645-668) in fp64 for the queued targets whose step may touch a disc:
// 32 (environment, target) items at a time, one per lane.  An fp32 segment-to-centre distance test picks
// the discs that can modify the step (Obstacle.obstruct changes a ray only if the ray meets the disc, i.e.
// the disc centre is within R of the segment); only those go through the fp64 Obstacle.obstruct.
template <int NC, int NT, int NO, class S>
__device__ __noinline__ void process_slow_targets(const Params& p, int env0, float* val, const uint16_t* queue, int base, int n,
                                                  const uint32_t (&near)[NT]) {
    const int lane = threadIdx.x & 31;
    const bool live = lane < n;
    const uint32_t item = live ? queue[base + lane] : 0u;
    const int src = item >> 8, t = item & 0xFF;
    // the discs within reach of this target's step, from the lane that owns its environment (called by all 32 lanes)
    constexpr bool REACH_MASKS = NO > 16 && NO + NC <= 32;
    uint32_t reach_set = 0xffffffffu;
    if (REACH_MASKS) {
        reach_set = 0u;
#pragma unroll
        for (int k = 0; k < NT; ++k) { const uint32_t m = __shfl_sync(0xffffffffu, near[k], src); if (k == t) reach_set = m; }
    }
    if (!live) return;
    const int env = env0 + src;
    const bool env_ok = env < p.num_envs;
    const int er = env_ok ? env : p.num_envs - 1;
    float* v = val + src * S::VSTRIDE;
    const float* camv = v + S::V_C;
    uint32_t tpack = __float_as_uint(v[S::V_T + 3 * t + 2]);
    const size_t bp = p.bpad;
    const float4* const obs_f4 = p.obs_f4 + er;
    const double* const obs_x = p.obs_x + er; const double* const obs_y = p.obs_y + er; const double* const obs_r = p.obs_r + er;
    const double* const cam_x = p.cam_x + er; const double* const cam_y = p.cam_y + er;
    const double cam_radius = p.cam_radius;
    const double tx = p.tgt_x[(size_t)t * bp + er], ty = p.tgt_y[(size_t)t * bp + er];
    const float2 a = reinterpret_cast<const float2*>(p.tgt_act)[(size_t)er * NT + t];
    const double step_size = p.tgt_step_size / (double)tp_capacity(tpack);
    StepVec s{(double)a.x, (double)a.y, 0.0, 0.0, step_size, false, false};
    const double n2 = s.vx * s.vx + s.vy * s.vy;
    if (n2 > step_size * step_size * (1.0 - 1e-12)) {
        s.n = sqrt(n2); s.has_n = true;
        if (s.n > step_size) {   // Vector2D.norm setter (utils.py:223-229), see DESIGN.md
            const double k = step_size / s.n;
            s.vx *= k; s.vy *= k; s.n = step_size;
        }
        s.bound = s.n * (1.0 + 1e-12);
    }
    const double desx = tx + s.vx, desy = ty + s.vy;
    // fp32 candidates: discs (obstacles, then cameras) whose centre lies within R (+ slack) of the segment
    // [origin, origin + v] -- a necessary condition for Obstacle.obstruct to change the step (the origin inside the
    // disc, or the ray entering it within its length)
    const float ftx = (float)tx, fty = (float)ty;
    auto candidates = [&](const double vx, const double vy) {
        unsigned long long cand = 0ull;
        const float fvx = (float)vx, fvy = (float)vy;
        const float vv = fvx * fvx + fvy * fvy, inv_vv = vv > 0.f ? 1.0f / vv : 0.f;
        auto near_segment = [&](const float cx, const float cy, const float R) {
            const float rx = cx - ftx, ry = cy - fty;
            const float tt = fminf(fmaxf((rx * fvx + ry * fvy) * inv_vv, 0.f), 1.f);
            const float ex = rx - tt * fvx, ey = ry - tt * fvy;
            const float reach = R * 1.0001f + 0.02f;
            return !(ex * ex + ey * ey > reach * reach);
        };
        if (REACH_MASKS) {   // only the discs within reach of the step (a bent step is never longer than the straight one)
            uint32_t rm = reach_set;
#pragma unroll 1
            while (rm != 0u) {
                const int d = __ffs(rm) - 1;
                rm &= rm - 1u;
                bool hit;
                if (d < NO) { const float4 ob = obs_f4[(size_t)d * bp]; hit = near_segment(ob.x, ob.y, ob.z); }
                else hit = near_segment(camv[S::CV * (d - NO)], camv[S::CV * (d - NO) + 1], (float)cam_radius);
                cand |= (unsigned long long)hit << d;
            }
            return cand;
        }
        float4 nxt = make_float4(0.f, 0.f, 0.f, 0.f);
        if (NO > 0) nxt = obs_f4[0];
#pragma unroll 4
        for (int o = 0; o < NO; ++o) {
            const float4 ob = nxt;
            if (o + 1 < NO) nxt = obs_f4[(size_t)(o + 1) * bp];
            cand |= (unsigned long long)near_segment(ob.x, ob.y, ob.z) << o;
        }
#pragma unroll
        for (int c = 0; c < NC; ++c)
            cand |= (unsigned long long)near_segment(camv[S::CV * c], camv[S::CV * c + 1], (float)cam_radius) << (NO + c);
        return cand;
    };
    // Discs in the reference's order.  A disc that is not a candidate cannot change the step; once a disc has bent
    // it, the candidates among the LATER discs are those of the bent step (re-classified in fp32: the reference walks
    // all of them through Obstacle.obstruct, 32 fp64 evaluations per bent step in the Navigation preset).  Every lane
    // walks its OWN candidates (most targets have exactly one), so the warp pays one round trip for the fp64 disc per
    // candidate rank instead of one per disc index.
    unsigned long long cand = candidates(s.vx, s.vy);
#pragma unroll 1
    while (cand != 0ull) {
        const int d = __ffsll((long long)cand) - 1;
        const double ovx = s.vx, ovy = s.vy;
        if (d < NO) obstruct_step(s, tx, ty, obs_x[(size_t)d * bp], obs_y[(size_t)d * bp], obs_r[(size_t)d * bp]);
        else obstruct_step(s, tx, ty, cam_x[(size_t)(d - NO) * bp], cam_y[(size_t)(d - NO) * bp], cam_radius);
        const unsigned long long later = ~((2ull << d) - 1ull);
        if (s.vx != ovx || s.vy != ovy) cand = candidates(s.vx, s.vy) & later;
        else cand &= later;
    }
    const double nx = fmin(fmax(tx + s.vx, -kTerrain), kTerrain);
    const double ny = fmin(fmax(ty + s.vy, -kTerrain), kTerrain);
    const int colliding = !(fabs(nx - desx) <= 1e-6 && fabs(ny - desy) <= 1e-6);
    tpack = (tpack & ~(1u << 27)) | ((uint32_t)colliding << 27);
    if (env_ok) { p.tgt_x[(size_t)t * bp + env] = nx; p.tgt_y[(size_t)t * bp + env] = ny; }
    v[S::V_T + 3 * t + 0] = (float)nx; v[S::V_T + 3 * t + 1] = (float)ny;
    v[S::V_T + 3 * t + 2] = __uint_as_float(tpack);
}

// occlusion of the segment camera c -> point q of env `er`: fast classification, exact polyline if undecided
template <int NO>
__device__ __forceinline__ bool line_of_sight(const Params& p, int er, int c, float fcx, float fcy, float fqx, float fqy,
                                              const double* qxp, const double* qyp) {
    const size_t bp = p.bpad;
    const int fast = occlusion_fast<NO>(p.obs_f4 + er, bp, fcx, fcy, fqx - fcx, fqy - fcy, (float)p.cam_rmax);
    if (fast != 2) return fast == 1;
    const double cx = p.cam_x[(size_t)c * bp + er], cy = p.cam_y[(size_t)c * bp + er];
    const double relx = *qxp - cx, rely = *qyp - cy;
    return occlusion_exact<NO>(ObsRef{p.obs_x + er, p.obs_y + er, p.obs_r + er, bp}, cx, cy, relx, rely,
                               sqrt(relx * relx + rely * rely), p.cam_rmax);
}

// per-episode cache of the static camera -> camera lines of sight (bit 8 j + c: camera c has a clear
// line of sight to camera j; bit 63: valid)
template <int NC, int NO>
__device__ __noinline__ unsigned long long build_cc_cache(const Params& p, int er) {
    const size_t bp = p.bpad;
    unsigned long long w = 1ull << 63;
    for (int c = 0; c < NC; ++c)
        for (int j = 0; j < NC; ++j) {
            if (j == c) continue;
            bool clear = true;
            if (NO > 0 && !p.transmittance_is_one) {
                const double* qx = p.cam_x + (size_t)j * bp + er;
                const double* qy = p.cam_y + (size_t)j * bp + er;
                clear = line_of_sight<NO>(p, er, c, (float)p.cam_x[(size_t)c * bp + er], (float)p.cam_y[(size_t)c * bp + er],
                                          (float)*qx, (float)*qy, qx, qy);
            }
            w |= (unsigned long long)clear << (8 * j + c);
        }
    return w;
}

// MultiAgentTracking.reset for one environment (one lane): new geometry and cargo table, written
// straight to the state arrays.  Returns the capacity-2 bit set; cargo goes to `cargo`.
template <int NC, int NT, int NO>
__device__ __noinline__ uint32_t reset_env_global(const Params& p, int e, RngKey key, Cargo* cargo) {
    double Ecam[(NC > 0 ? NC : 1) * 5], Etgt[NT * 2], Eobs[(NO > 0 ? NO : 1) * 3];
    uint32_t scr[16];
    ResetCfg rc;
    rc.cam_radius = p.cam_radius; rc.cam_min_view = p.cam_min_view; rc.cam_rot_step = p.cam_rot_step;
    rc.cam_area_product = p.cam_area_product; rc.tgt_step_size = p.tgt_step_size;
    rc.obs_r_low = p.obs_r_low; rc.obs_r_high = p.obs_r_high;
    rc.cam_ranges = p.cam_ranges; rc.tgt_ranges = p.tgt_ranges; rc.obs_ranges = p.obs_ranges;
    rc.shuffle = p.shuffle; rc.num_high_capacity = p.num_high_capacity;
    rc.num_cargoes_per_target = p.num_cargoes_per_target;
    env_reset<NC, NT, NO, 5>(rc, key, Ecam, Etgt, Eobs, scr);
    const size_t bp = p.bpad;
    for (int c = 0; c < NC; ++c) {
        p.cam_x[(size_t)c * bp + e] = Ecam[c * 5 + 0]; p.cam_y[(size_t)c * bp + e] = Ecam[c * 5 + 1];
        p.cam_phi[(size_t)c * bp + e] = Ecam[c * 5 + 2]; p.cam_theta[(size_t)c * bp + e] = Ecam[c * 5 + 3];
    }
    for (int t = 0; t < NT; ++t) { p.tgt_x[(size_t)t * bp + e] = Etgt[2 * t]; p.tgt_y[(size_t)t * bp + e] = Etgt[2 * t + 1]; }
    for (int o = 0; o < NO; ++o) {
        p.obs_x[(size_t)o * bp + e] = Eobs[3 * o]; p.obs_y[(size_t)o * bp + e] = Eobs[3 * o + 1]; p.obs_r[(size_t)o * bp + e] = Eobs[3 * o + 2];
        p.obs_f4[(size_t)o * bp + e] = make_float4((float)Eobs[3 * o], (float)Eobs[3 * o + 1], (float)Eobs[3 * o + 2], 0.f);
    }
    for (int k = 0; k < 8; ++k) cargo->rem[k] = scr[k];
    cargo->aw[0] = scr[8]; cargo->aw[1] = scr[9];
    return scr[10];
}

// One view mask of one environment ([ROWS][COLS] uint8 in the caller's tensor): the rows' bits are concatenated
// into a bit string, four bits at a time become four bytes with one multiply ((x & 15) * 0x00204081 & 0x01010101
// puts bit j into byte j), and the bytes leave with the widest store the row length allows -- instead of one
// byte store per mask entry (a lane owns an environment, so every store of the warp touches 32 sectors).
template <int ROWS, int COLS>
struct MaskBytes {
    static constexpr int L = ROWS * COLS, NB = (L + 31) / 32 > 0 ? (L + 31) / 32 : 1;
    uint32_t w[NB];
    __device__ __forceinline__ MaskBytes() {
#pragma unroll
        for (int i = 0; i < NB; ++i) w[i] = 0u;
    }
    __device__ __forceinline__ void row(const int r, uint32_t bits) {   // r must be a compile-time constant after unrolling
        if (COLS < 32) bits &= (1u << (COLS & 31)) - 1u;
        const int off = r * COLS, word = off >> 5, sh = off & 31;
        w[word] |= bits << sh;
        if (sh + COLS > 32) w[word + 1] |= bits >> (32 - sh);
    }
    __device__ __forceinline__ uint32_t bytes4(const int j) const {   // bytes 4 j .. 4 j + 3 of the row-major byte array
        const uint32_t nib = (w[(4 * j) >> 5] >> ((4 * j) & 31)) & 15u;
        return (nib * 0x00204081u) & 0x01010101u;
    }
    __device__ __forceinline__ void store(uint8_t* base, const size_t e) const {
        if (L == 0) return;
        uint8_t* dst = base + e * L;
        if (L % 16 == 0) {
#pragma unroll
            for (int i = 0; i < L / 16; ++i)
                reinterpret_cast<uint4*>(dst)[i] = make_uint4(bytes4(4 * i), bytes4(4 * i + 1), bytes4(4 * i + 2), bytes4(4 * i + 3));
        } else if (L % 8 == 0) {
#pragma unroll
            for (int i = 0; i < L / 8; ++i) reinterpret_cast<uint2*>(dst)[i] = make_uint2(bytes4(2 * i), bytes4(2 * i + 1));
        } else if (L % 4 == 0) {
#pragma unroll
            for (int i = 0; i < L / 4; ++i) reinterpret_cast<uint32_t*>(dst)[i] = bytes4(i);
        } else {
#pragma unroll
            for (int i = 0; i < L; ++i) dst[i] = (uint8_t)((w[i >> 5] >> (i & 31)) & 1u);
        }
    }
};

// aux outputs = the reference's public per-step attributes (environment.py:634-661); one lane = one env
template <int NC, int NT, int NO, class S>
__device__ __noinline__ void write_aux_env(const Params& p, int e, const uint32_t* mrow, const float* vrow, uint32_t tdone_bits,
                                           float cov_now, float cov_real, float transport, int delivered, int episode_step) {
    const MateStepAux& ax = p.aux;
    constexpr int MW = S::MW;
    auto obs_bits = [&](int row) -> uint32_t { return MW == 1 ? (mrow[row] >> 16) : mrow[row * MW + 1]; };
    {
        MaskBytes<NC, NT> ct; MaskBytes<NC, NC> cc; MaskBytes<NC, NO> co;
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const uint32_t w = mrow[c * MW];
            ct.row(c, w >> 8); cc.row(c, w); co.row(c, obs_bits(c));
        }
        if (ax.mask_ct) ct.store(ax.mask_ct, (size_t)e);
        if (ax.mask_cc) cc.store(ax.mask_cc, (size_t)e);
        if (ax.mask_co) co.store(ax.mask_co, (size_t)e);
    }
    {
        MaskBytes<NT, NC> tc; MaskBytes<NT, NT> tt; MaskBytes<NT, NO> to;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const uint32_t w = mrow[(NC + t) * MW];
            tc.row(t, w); tt.row(t, w >> 8); to.row(t, obs_bits(NC + t));
        }
        if (ax.mask_tc) tc.store(ax.mask_tc, (size_t)e);
        if (ax.mask_tt) tt.store(ax.mask_tt, (size_t)e);
        if (ax.mask_to) to.store(ax.mask_to, (size_t)e);
    }
    {   // per-target flags and integers
        MaskBytes<1, NT> dones, colliding;
        uint32_t coll = 0;
#pragma unroll
        for (int t = 0; t < NT; ++t) coll |= (uint32_t)tp_colliding(__float_as_uint(vrow[S::V_T + 3 * t + 2])) << t;
        dones.row(0, tdone_bits); colliding.row(0, coll);
        if (ax.target_dones) dones.store(ax.target_dones, (size_t)e);
        if (ax.is_colliding) colliding.store(ax.is_colliding, (size_t)e);
    }
    for (int t = 0; t < NT; ++t) {
        const uint32_t tp = __float_as_uint(vrow[S::V_T + 3 * t + 2]);
        if (ax.tgt_goal) ax.tgt_goal[(size_t)e * NT + t] = tp_goal(tp);
        if (ax.tgt_empty_bits) ax.tgt_empty_bits[(size_t)e * NT + t] = (uint8_t)tp_empty(tp);
        if (ax.warehouse_dist) {
            const double tx = p.tgt_x[(size_t)t * p.bpad + e], ty = p.tgt_y[(size_t)t * p.bpad + e];
            float wd[NW];
#pragma unroll
            for (int w4 = 0; w4 < NW; ++w4) {
                const double wx = (w4 == 0 || w4 == 3) ? kWarehouseCoord : -kWarehouseCoord;
                const double wy = (w4 < 2) ? kWarehouseCoord : -kWarehouseCoord;
                wd[w4] = (float)norm2(tx - wx, ty - wy);
            }
            reinterpret_cast<float4*>(ax.warehouse_dist)[(size_t)e * NT + t] = make_float4(wd[0], wd[1], wd[2], wd[3]);
        }
    }
    if (ax.coverage) {   // coverage statistics (environment.py:966-979)
        ax.coverage[(size_t)e * 3 + 0] = cov_now; ax.coverage[(size_t)e * 3 + 1] = cov_real; ax.coverage[(size_t)e * 3 + 2] = transport;
    }
    if (ax.num_delivered) ax.num_delivered[e] = delivered;
    if (ax.episode_step) ax.episode_step[e] = episode_step;
}

// Camera.simulate's derived quantities (entities.py:334,360) -> the fp32 entries of one camera
__device__ __forceinline__ void store_camera(float* v, double x, double y, double phi, double theta, double area_product) {
    const double rs = sqrt(area_product / theta);
    double sn, cs;
    sincospi(phi * (1.0 / 180.0), &sn, &cs);
    v[0] = (float)x; v[1] = (float)y; v[2] = (float)theta; v[3] = (float)(rs * cs); v[4] = (float)(rs * sn);
}

// ---- guard-band resolution (rare): the fp32 test fell inside its band, the fp64 expression decides.
// One call site per loop nest; `band` has one bit per partner entity, the result has the bits that pass.
// kind: 0 = partner targets, 1 = partner cameras; (ax, ay) is the fixed entity.
__device__ __noinline__ uint32_t resolve_band(const Params& p, int er, const double* ax, const double* ay, uint32_t band, int kind,
                                              double thr, bool strict) {
    uint32_t out = 0;
    while (band) {
        const int k = __ffs(band) - 1;
        band &= band - 1;
        const size_t i = (size_t)k * p.bpad + er;
        const double* bx = kind == 0 ? p.tgt_x + i : p.cam_x + i;
        const double* by = kind == 0 ? p.tgt_y + i : p.cam_y + i;
        if (sense_exact(ax, ay, bx, by, thr, strict)) out |= 1u << k;
    }
    return out;
}
// same for the range + sector test of camera c against partner targets (kind 0) / cameras (kind 1)
__device__ __noinline__ uint32_t resolve_fov_band(const Params& p, int er, int c, uint32_t band, int kind) {
    uint32_t out = 0;
    while (band) {
        const int k = __ffs(band) - 1;
        band &= band - 1;
        const size_t i = (size_t)k * p.bpad + er;
        if (fov_reach_global(p, er, c, kind == 0 ? p.tgt_x + i : p.cam_x + i, kind == 0 ? p.tgt_y + i : p.cam_y + i)) out |= 1u << k;
    }
    return out;
}

// Exact evaluation of the sampled FOV polyline for the queued (camera, target) pairs whose occlusion the
// conservative classification could not decide.  A warp tile has ~7 such pairs per step: one pair per lane would
// leave 25 lanes idle through the longest dependent chain of the kernel, so a QUAD of lanes evaluates one pair
// (sight_range_quad: each lane owns a quarter of the discs, in registers) and the warp takes 8 pairs per pass.
// Called by all 32 lanes.
template <int NC, int NT, int NO, class S>
__device__ __noinline__ void process_exact(const Params& p, int env0, uint32_t* mk, const uint16_t* queue2, int base, int n) {
    const int lane = threadIdx.x & 31, q = lane & 3, slot = lane >> 2;
    const size_t bp = p.bpad;
#pragma unroll 1
    for (int i0 = 0; i0 < n; i0 += 8) {
        const bool live = i0 + slot < n;
        const uint32_t item = queue2[base + (live ? i0 + slot : 0)];   // idle quads shadow pair 0 (results discarded)
        const int src = item >> 8, b = item & 0xFF;
        const int c = b / NT, t = b - c * NT;
        const int envr = min(env0 + src, p.num_envs - 1);
        const double cx = p.cam_x[(size_t)c * bp + envr], cy = p.cam_y[(size_t)c * bp + envr];
        const double relx = p.tgt_x[(size_t)t * bp + envr] - cx, rely = p.tgt_y[(size_t)t * bp + envr] - cy;
        const double dist = sqrt(relx * relx + rely * rely);
        const double ang = normalize_angle(atan2_deg(rely, relx));
        const double range = sight_range_quad<NO>(ObsRef{p.obs_x + envr, p.obs_y + envr, p.obs_r + envr, bp}, cx, cy, p.cam_rmax, ang,
                                                  relx / dist, rely / dist, q);
        if (live && q == 0 && dist <= range * (1.0 + 1e-6)) atomicOr(&mk[src * S::MSTRIDE + c * S::MW], bit_tgt(t));   // entities.py:505
    }
}

// Prepared resets.  MultiAgentTracking.reset costs tens of thousands of dependent instructions for ONE lane
// (rejection placement, cargo table, camera lines of sight, first view) while the other 31 lanes of the
// warp wait, and the launch ends with its slowest warp.  A reset depends only on (seed, env, episode id),
// so it is computed ahead of time: mate_step_kernel2 in MODE_PREPARE runs on a second state block (its
// Params address that block) for every env whose prepared state is not valid for episode id + 1, on a side
// stream, off the step path.  When an episode ends, the step kernel checks the `ready` tag and simply
// copies the prepared state and first-view masks; if the tag does not match it runs the reset in place
// (identical result, same counter-based draws).
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* ptr) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ptr) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* ptr, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(ptr), "r"(v) : "memory");
}

// The time limit announces a reset one step ahead: pull the prepared state of env e into L2 now, so that the
// copy in the next step does not pay one DRAM round trip per group of loads.
template <int NC, int NT, int NO, class S>
__device__ __noinline__ void prefetch_prepared(const Params& nx, int e) {
    const size_t bp = nx.bpad;
    // evict_last: 450 MB of observation rows stream through the L2 before the copy reads these lines
    auto pf = [](const void* ptr) { asm volatile("prefetch.global.L2::evict_last [%0];" :: "l"(ptr)); };
    pf(nx.ready + e);
#pragma unroll 1
    for (int c = 0; c < NC; ++c) { const size_t i = (size_t)c * bp + e; pf(nx.cam_x + i); pf(nx.cam_y + i); pf(nx.cam_phi + i); pf(nx.cam_theta + i); }
#pragma unroll 1
    for (int t = 0; t < NT; ++t) { const size_t i = (size_t)t * bp + e; pf(nx.tgt_x + i); pf(nx.tgt_y + i); }
#pragma unroll 1
    for (int k = 0; k < S::VN; ++k) pf(nx.vals + (size_t)k * bp + e);
#pragma unroll 1
    for (int o = 0; o < NO; ++o) { const size_t i = (size_t)o * bp + e; pf(nx.obs_x + i); pf(nx.obs_y + i); pf(nx.obs_r + i); pf(nx.obs_f4 + i); }
#pragma unroll 1
    for (int w = 0; w < S::R * S::MW; ++w) pf(nx.masks + (size_t)w * bp + e);
    pf(nx.cargo + e); pf(nx.cargo + bp + e); pf(nx.env_a + e); pf(nx.cc_clear + e);
}

// Copy the prepared initial state of the adopting environments (bit set `adopting`) from block `nx` into the live
// block `p`, the fp32 entries and the first-view masks into shared memory.  The whole warp copies: one lane copying
// ~180 scattered words that nobody has touched for an episode needs three to four dependent round trips while its
// warp (and, at the end of the launch, the whole grid) waits; spread over the 32 lanes every lane has 4-5 loads in
// flight and the copy is one round trip.  Cargo, the awaiting counts and the line-of-sight cache go to registers of
// the adopting lane and are loaded by that lane itself.
template <int NC, int NT, int NO, class S>
__device__ __noinline__ void adopt_prepared_warp(const Params& p, const Params& nx, const int env0, uint32_t adopting,
                                                 float* val, uint32_t* mk) {
    const int noff = p.next_offset;   // index shift between this launch's (offset) live arrays and the whole-batch prepared arrays
    __syncwarp();   // the lanes are about to overwrite shared-memory rows their owners read and wrote a moment ago (racecheck)
    constexpr int ND = 4 * NC + 2 * NT + 3 * NO, NV = S::VN, NM = S::R * S::MW;
    constexpr int JD = (ND + 31) / 32, JV = (NV + 31) / 32, JM = (NM + 31) / 32, JF = (NO + 31) / 32 > 0 ? (NO + 31) / 32 : 1;
    const int lane = threadIdx.x & 31;
    const size_t bp = p.bpad;
    while (adopting != 0u) {
        const int src = __ffs(adopting) - 1;
        adopting &= adopting - 1u;
        const int e = env0 + src;
        auto field = [&](const Params& q, const int k, const int e) -> double* {   // k-th double of an environment's state
            if (k < 4 * NC) {
                const int f = k / (NC > 0 ? NC : 1), c = k - f * NC;
                double* base = f == 0 ? q.cam_x : (f == 1 ? q.cam_y : (f == 2 ? q.cam_phi : q.cam_theta));
                return base + (size_t)c * bp + e;
            }
            if (k < 4 * NC + 2 * NT) {
                const int r = k - 4 * NC, f = r / NT, t = r - f * NT;
                return (f == 0 ? q.tgt_x : q.tgt_y) + (size_t)t * bp + e;
            }
            const int r = k - 4 * NC - 2 * NT, f = r / (NO > 0 ? NO : 1), o = r - f * NO;
            return (f == 0 ? q.obs_x : (f == 1 ? q.obs_y : q.obs_r)) + (size_t)o * bp + e;
        };
        double d[JD]; float v[JV]; uint32_t m[JM]; float4 f4[JF];
#pragma unroll
        for (int j = 0; j < JD; ++j) { const int k = lane + 32 * j; d[j] = k < ND ? *field(nx, k, e + noff) : 0.0; }
#pragma unroll
        for (int j = 0; j < JV; ++j) { const int k = lane + 32 * j; v[j] = k < NV ? nx.vals[(size_t)k * bp + e + noff] : 0.f; }
#pragma unroll
        for (int j = 0; j < JM; ++j) { const int k = lane + 32 * j; m[j] = k < NM ? nx.masks[(size_t)k * bp + e + noff] : 0u; }
#pragma unroll
        for (int j = 0; j < JF; ++j) { const int k = lane + 32 * j; f4[j] = k < NO ? nx.obs_f4[(size_t)k * bp + e + noff] : make_float4(0.f, 0.f, 0.f, 0.f); }
#pragma unroll
        for (int j = 0; j < JD; ++j) { const int k = lane + 32 * j; if (k < ND) *field(p, k, e) = d[j]; }
#pragma unroll
        for (int j = 0; j < JV; ++j) { const int k = lane + 32 * j; if (k < NV) val[src * S::VSTRIDE + k] = v[j]; }
#pragma unroll
        for (int j = 0; j < JM; ++j) { const int k = lane + 32 * j; if (k < NM) mk[src * S::MSTRIDE + k] = m[j]; }
#pragma unroll
        for (int j = 0; j < JF; ++j) { const int k = lane + 32 * j; if (k < NO) p.obs_f4[(size_t)k * bp + e] = f4[j]; }
    }
}

// =============================================================================================
// joint_observation (environment.py:908-983) for the warp's environments [env0, env0 + nvalid).
// Out of line on purpose: the packer gets its own register allocation.
// =============================================================================================
// the registered observation wrappers on the staged rows of one environment; out of line: the common case has none
template <int NC, int NT, int NO>
__device__ __noinline__ void fold_obs_ops(const Params& p, const int env, float* stage, float* scratch) {
    using S = Shape2<NC, NT, NO>;
    apply_obs_ops<NC, NT, NO>(p, p.obs_ops, env, stage, stage + S::STAGE_CAM, scratch, p.cam_affine, p.tgt_affine);
}

// two fp32 values rounded to float16 (nearest even), `lo` at the lower address
__device__ __forceinline__ uint32_t half2_bits(const float lo, const float hi) {
    const __half2 h = __float22half2_rn(make_float2(lo, hi));
    return *reinterpret_cast<const uint32_t*>(&h);
}

// One team's rows of an environment -> HBM: N values, staged in shared memory as float32 with rows of ROW values SKEW
// floats apart (camera rows, Shape2::CAM_SKEW).  Each lane stores with the widest type whose size divides the part: 16, 8
// or 4 bytes for float32, 16, 8, 4 or 2 bytes for float16 (the caller's buffers are 16-byte aligned, so the part of
// environment i starts at a multiple of gcd(16, part bytes); MATE-4v2-9: 2 x 101 floats of target rows leave with 8-byte
// stores).  float16 values are rounded from the staged ones in pairs (__float22half2_rn, nearest even).
template <class OutT, int N, int ROW, int SKEW>
__device__ __forceinline__ void store_team_rows(OutT* dst, const float* src) {
    constexpr bool F16 = std::is_same<OutT, __half>::value;
    constexpr int W = (F16 && N % 8 == 0) ? 8 : (N % 4 == 0 ? 4 : (N % 2 == 0 ? 2 : 1));   // values per store
    static_assert(SKEW == 0 || (ROW % W == 0 && SKEW % 4 == 0), "a store must not straddle two skewed rows");
    // staged index of chunk c of the part, in chunks of v floats.  The float32 loads index whole 16- / 8-byte chunks, the
    // float16 loads single floats: the same addresses, but each form gives its format's packers the code they were
    // measured with (ptxas allocates registers across all packers of a kernel, so one form for both changes the others)
    auto at = [](const int c, const int v) { return SKEW ? c + (c / (ROW / v)) * (SKEW / v) : c; };
    const float4* const src4 = reinterpret_cast<const float4*>(src);
    const float2* const src2 = reinterpret_cast<const float2*>(src);
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int it = 0; it < (N / W + 31) / 32; ++it) {
        const int k = it * 32 + lane;
        if (k < N / W) {
            if constexpr (W == 8) {
                // lanes 4-7 of every quarter-warp read their two 16-byte halves in the other order: each of the
                // two loads then covers eight distinct 16-byte bank groups per quarter-warp
                const int sw = (lane >> 2) & 1;
                const float4 a = *reinterpret_cast<const float4*>(src + at(8 * k + 4 * sw, 1));
                const float4 b = *reinterpret_cast<const float4*>(src + at(8 * k + 4 - 4 * sw, 1));
                const float4 lo = sw ? b : a, hi = sw ? a : b;
                __stcs(reinterpret_cast<uint4*>(dst) + k, make_uint4(half2_bits(lo.x, lo.y), half2_bits(lo.z, lo.w),
                                                                     half2_bits(hi.x, hi.y), half2_bits(hi.z, hi.w)));
            } else if constexpr (W == 4) {
                if constexpr (F16) {
                    const float4 a = *reinterpret_cast<const float4*>(src + at(4 * k, 1));
                    __stcs(reinterpret_cast<uint2*>(dst) + k, make_uint2(half2_bits(a.x, a.y), half2_bits(a.z, a.w)));
                } else {
                    __stcs(reinterpret_cast<float4*>(dst) + k, src4[at(k, 4)]);
                }
            } else if constexpr (W == 2) {
                if constexpr (F16) {
                    const float2 a = *reinterpret_cast<const float2*>(src + at(2 * k, 1));
                    __stcs(reinterpret_cast<unsigned int*>(dst) + k, half2_bits(a.x, a.y));
                } else {
                    __stcs(reinterpret_cast<float2*>(dst) + k, src2[at(k, 2)]);
                }
            } else if constexpr (F16) {
                __stcs(reinterpret_cast<unsigned short*>(dst) + k, __half_as_ushort(__float2half_rn(src[at(k, 1)])));
            } else {
                dst[k] = src[at(k, 1)];   // odd float32 parts (MATE-1v1-x, 1v2-x): plain stores, the streaming hint is not measured there
            }
        }
    }
}

// The observer rows a launch composes and stores: the camera rows [0, NC), the target rows [NC, NC + NT) or both
// (a NULL row pointer of the call drops its team, DESIGN.md section 7j)
enum : int { ROWS_CAM = 1, ROWS_TGT = 2, ROWS_BOTH = 3 };

// FOLD = the instantiation that also applies the registered observation wrappers (FoldOps, mate_common.cuh) while
// the rows are composed; the common case (no wrappers) runs the FOLD = false instantiation, which has none of it.
// OutT = element type of the rows in HBM (Params::obs_format): float, or __half rounded once from the staged fp32 rows
// while they leave the SM.  Everything before the copy-out is the same for both.
// ROWS = the observer rows composed (ROWS_*): a row outside the set gets no pair scatter, no own-row block and no
// store, and the rounds of the scatter cover only the rows inside it.  The wrappers outside the canonical form
// (fold_obs_ops) still run over the whole staged block; EnhancedObservation copies entity states from the own-row
// blocks of the other team, so on that path the own-row blocks of every row are composed.
template <int NC, int NT, int NO, bool FOLD, class OutT, int ROWS>
__device__ __noinline__ void pack_rows(const Params& p, const int env0, const int nvalid, float* stage,
                                       const uint32_t* mk, const float* val, float* ops_scratch) {
    using S = Shape2<NC, NT, NO>;
    constexpr bool F16 = std::is_same<OutT, __half>::value;
    static_assert(F16 || std::is_same<OutT, float>::value, "observation rows are float or __half");
    static_assert(ROWS == ROWS_BOTH || ((ROWS == ROWS_CAM || ROWS == ROWS_TGT) && NC > 0), "a single team's rows need cameras");
    constexpr int R = S::R, MW = S::MW, DC = S::DC, DT = S::DT, CV = S::CV;
    constexpr bool WANT_C = (ROWS & ROWS_CAM) != 0, WANT_T = (ROWS & ROWS_TGT) != 0;
    constexpr int R0 = WANT_C ? 0 : NC, R1 = WANT_T ? R : NC;   // the composed rows [R0, R1)
    constexpr int NCX = NC > 0 ? NC : 1;
    constexpr uint32_t FULLMASK = 0xffffffffu;
    constexpr ObsLayout L{NC, NT, NO};
    const int lane = threadIdx.x & 31;
    // ---- folded wrappers: which ones, and the scratch they use (behind the warp's block, present when wrappers are registered)
    const bool fast = FOLD && p.fold.fast != 0;
    const bool f_rel = fast && p.fold.relative != 0, f_resc = fast && p.fold.rescaled != 0, f_mask = fast && p.fold.n_mask > 0;
    constexpr int EALL = NT + NO + NC;
    double* const fpos = reinterpret_cast<double*>(ops_scratch);                       // [EALL][2] fp64 locations: targets, obstacles, cameras
    uint32_t* const mmod = reinterpret_cast<uint32_t*>(ops_scratch) + 4 * EALL;       // [R * MW] mask words after the mask wrappers
    float2* const aff_own = reinterpret_cast<float2*>(ops_scratch + 4 * EALL + R * MW + ((R * MW) & 1));   // [ObsLayout::AFF_COLS] (scale, shift)
    if (FOLD && f_resc) {   // staged once per tile: the parameter block is only reachable through slow generic loads here
        using A = ObsLayout;
        for (int k = lane; k < A::AFF_COLS; k += 32)
            aff_own[k] = k < A::AFF_TSELF ? p.fold.pres[k - A::AFF_PRES]
                       : (k < A::AFF_CSELF ? p.fold.tself[k - A::AFF_TSELF]
                       : (k < A::AFF_TGT ? p.fold.cself[k - A::AFF_CSELF]
                       : (k < A::AFF_OBS ? p.fold.tgt[k - A::AFF_TGT]
                       : (k < A::AFF_CAM ? p.fold.obs[k - A::AFF_OBS] : p.fold.cam[k - A::AFF_CAM]))));
    }
    // launch parameters used inside the loop, read once (a reference to the parameter block is a generic
    // pointer: the compiler would re-load through it after every store)
    const size_t bp = p.bpad;
    OutT* const cam_obs0 = reinterpret_cast<OutT*>(p.cam_obs) + (size_t)env0 * S::CAM_ROW;
    OutT* const tgt_obs0 = reinterpret_cast<OutT*>(p.tgt_obs) + (size_t)env0 * S::TGT_ROW;
    const float4* const obs_f4 = p.obs_f4;
    // The warp walks over its environments and assembles the 6 KB block of observation rows of one
    // environment in shared memory, every float written exactly once and without branches:
    //   * (observer row, entity) PAIRS are spread over the lanes, one entity kind at a time (a lane keeps
    //     the same entity for all rounds of a kind); a pair writes the entity's public state and flag if
    //     the observer's mask bit is set and zeros otherwise (masked-out entries are all-zero);
    //   * lanes 0..R-1 write the preserved block and the private state of "their" observer row.
    // first columns of the entity lists in a camera (C_*) / target (T_*) row, as constants (see apply_obs_ops)
    constexpr int C_TGT = L.block(true, KIND_TARGET), C_OBS = L.block(true, KIND_OBSTACLE), C_CAM = L.block(true, KIND_CAMERA);
    constexpr int T_TGT = L.block(false, KIND_TARGET), T_OBS = L.block(false, KIND_OBSTACLE), T_CAM = L.block(false, KIND_CAMERA);
    constexpr int NOX = NO > 0 ? NO : 1;
    constexpr int RPR_T = 32 / NT, RPR_O = 32 / NOX, RPR_C = 32 / NCX;          // observer rows per round
    constexpr typename S::ORounds ORND = S::make_orounds(R0, R1);
    constexpr int RW = R1 - R0;
    constexpr int RND_T = (RW + RPR_T - 1) / RPR_T, RND_O = NO > 0 ? ORND.n : 1, RND_C = (RW + RPR_C - 1) / RPR_C;
    const float f_sr = (float)p.tgt_sight_range, f_crad = (float)p.cam_radius;
    const float f_rmax = (float)p.cam_rmax, f_rot = (float)p.cam_rot_step, f_zoom = (float)p.cam_zoom_step;
    const float f_step1 = (float)p.tgt_step_size, f_step2 = (float)(p.tgt_step_size / 2.0);
    // per-lane constants of the scatter, hoisted out of the environment loop: for every round the address of
    // this lane's slot in the staged block, the mask word that decides it, and whether the lane has a pair in
    // that round at all (its stores are predicated off otherwise)
    constexpr int NRND = RND_T + (NO > 0 ? RND_O : 0) + (NC > 0 ? RND_C : 0);
    const int t_idx = lane % NT, t_sub = lane / NT;
    const int o_idx = lane % NOX, o_sub = lane / NOX;
    const int c_idx = lane % NCX, c_sub = lane / NCX;
    constexpr int DCS = DC + (FOLD ? 0 : S::CAM_SKEW);   // stride of the staged camera rows (the wrappers' code expects dense rows)
    auto row_base = [&](const int row) { return row < NC ? row * DCS : S::STAGE_CAM + (row - NC) * DT; };
    float* q_ptr[NRND];   // this lane's slot in the staged block, per round
    int m_idx[NRND];      // and the mask word that decides it
    uint32_t on_bits = 0; // bit rd: the lane has a pair in round rd
#pragma unroll
    for (int rd = 0; rd < RND_T; ++rd) {
        const int row = R0 + rd * RPR_T + t_sub;
        const bool on = t_sub < RPR_T && row < R1;
        q_ptr[rd] = stage + (on ? row_base(row) + (row < NC ? C_TGT : T_TGT) + ObsLayout::TGT_ENTRY * t_idx : 0);
        m_idx[rd] = on ? row * MW : 0;
        on_bits |= (uint32_t)on << rd;
    }
    if (NO > 0) {
#pragma unroll
        for (int rd = 0; rd < RND_O; ++rd) {
            int row = R0 + rd * RPR_O + o_sub;
            bool on = o_sub < RPR_O && row < R1;
            if (ORND.grouped) {
                row = -1;
#pragma unroll
                for (int j = 0; j < 4; ++j) row = (j < RPR_O && o_sub == j) ? ORND.row[rd][j] : row;
                on = row >= 0;
            }
            q_ptr[RND_T + rd] = stage + (on ? row_base(row) + (row < NC ? C_OBS : T_OBS) + ObsLayout::OBS_ENTRY * o_idx : 0);
            m_idx[RND_T + rd] = on ? row * MW + (MW - 1) : 0;
            on_bits |= (uint32_t)on << (RND_T + rd);
        }
    }
    if (NC > 0) {
#pragma unroll
        for (int rd = 0; rd < RND_C; ++rd) {
            const int row = R0 + rd * RPR_C + c_sub;
            const bool on = c_sub < RPR_C && row < R1;
            q_ptr[NRND - RND_C + rd] = stage + (on ? row_base(row) + (row < NC ? C_CAM : T_CAM) + ObsLayout::CAM_ENTRY * c_idx : 0);
            m_idx[NRND - RND_C + rd] = on ? row * MW : 0;
            on_bits |= (uint32_t)on << (NRND - RND_C + rd);
        }
    }
    const uint32_t t_bit = bit_tgt(t_idx), o_bit = MW == 1 ? (1u << (16 + o_idx)) : (1u << o_idx), c_bit = bit_cam(c_idx);
    // the own-row entries that never change are staged once per tile: preserved block (environment.py:921-934)
    // and the constant entries of the private state -- unless observation wrappers are folded in, which rewrite
    // them in place for every environment
    const bool has_ops = FOLD && !fast && p.obs_ops.n > 0;   // a stack outside the canonical form: generic shared-memory path
    if (FOLD && f_resc) __syncwarp();   // aff_own is read below
    // (with RescaledObservation folded in, the constants are staged already rescaled; RelativeCoordinates rewrites the
    //  eight warehouse coordinates of a row for every environment, everything else here stays)
    auto stage_constants = [&]() {
        if (lane < R && (ROWS == ROWS_BOTH || has_ops || (lane >= R0 && lane < R1))) {
            const int row = lane;
            float* q = stage + row_base(row);
            auto put = [&](const int col, const float x, const int aff) { q[col] = (FOLD && f_resc) ? fmaf(x, aff_own[aff].x, aff_own[aff].y) : x; };
            static_assert(ObsLayout::PRESERVED == 13 && ObsLayout::WAREHOUSE == 4, "the preserved block is written column by column");
            auto pres = [&](const int col, const float x) { put(col, x, ObsLayout::AFF_PRES + col); };
            pres(0, (float)NC); pres(1, (float)NT); pres(2, (float)NO); pres(3, (float)(row < NC ? row : row - NC));
            pres(4, 925.f); pres(5, 925.f); pres(6, -925.f); pres(7, 925.f); pres(8, -925.f); pres(9, -925.f); pres(10, 925.f); pres(11, -925.f);   // warehouses
            pres(12, 75.f);
            constexpr int C = ObsLayout::SELF, AC = ObsLayout::AFF_CSELF;
            if (row < NC) { put(C + 2, f_crad, AC + 2); put(C + 6, f_rmax, AC + 6); put(C + 7, f_rot, AC + 7); put(C + 8, f_zoom, AC + 8); }
            else put(C + 2, f_sr, ObsLayout::AFF_TSELF + 2);
        }
    };
    stage_constants();
    float* const self_t = stage + S::STAGE_CAM + t_idx * DT + ObsLayout::SELF;   // used by lanes 0..NT-1
    float* const self_c = stage + c_idx * DCS + ObsLayout::SELF;                 // used by the NC lanes from NT on
    // obstacle entries are fetched two environments ahead (an L2 round trip is longer than one iteration)
    const float4* ob_ptr = obs_f4 + (size_t)o_idx * bp + env0;
    float4 ob_next = make_float4(0.f, 0.f, 0.f, 0.f), ob_next2 = ob_next;
    if (NO > 0) { ob_next = ob_ptr[0]; if (nvalid > 1) ob_next2 = ob_ptr[1]; }
    // RelativeCoordinates: the fp64 locations of the next environment's entities are fetched one environment ahead
    constexpr int FJ = (EALL + 31) / 32;
    double fx_next[FJ] = {}, fy_next[FJ] = {};
    // this lane's entities (targets, obstacles, cameras in that order): the addresses of their coordinates in the tile's first
    // environment are worked out once, an environment's fetch is then two loads per entity
    const double* loc_x[FJ];
    const double* loc_y[FJ];
#pragma unroll
    for (int j = 0; j < FJ; ++j) {
        const int k = lane + 32 * j;
        const double *bx = p.tgt_x, *by = p.tgt_y;
        int idx = k < NT ? k : 0;
        if (NO > 0 && k >= NT && k < NT + NO) { bx = p.obs_x; by = p.obs_y; idx = k - NT; }
        if (NC > 0 && k >= NT + NO && k < EALL) { bx = p.cam_x; by = p.cam_y; idx = k - NT - NO; }
        loc_x[j] = bx + (size_t)idx * bp + env0; loc_y[j] = by + (size_t)idx * bp + env0;
    }
    auto load_locations = [&](const int i_env) {
#pragma unroll
        for (int j = 0; j < FJ; ++j)
            if (lane + 32 * j < EALL) { fx_next[j] = loc_x[j][i_env]; fy_next[j] = loc_y[j][i_env]; }
    };
    if (FOLD && f_rel) load_locations(0);
    // the mask wrappers in their order, four bits each (read once: the parameter block is only reachable through generic loads)
    uint32_t mask_ops = 0;
    const int n_mask = FOLD ? p.fold.n_mask : 0;
    if (FOLD && f_mask) { for (int k = 0; k < n_mask; ++k) mask_ops |= (uint32_t)p.fold.mask_op[k] << (4 * k); }
    __syncwarp();
#pragma unroll 1
    for (int i = 0; i < nvalid; ++i) {
        const float* v = val + i * S::VSTRIDE;
        const uint32_t* m = mk + i * S::MSTRIDE;
        const float4 ob = ob_next;
        ob_next = ob_next2;
        if (NO > 0 && i + 2 < nvalid) ob_next2 = ob_ptr[i + 2];
        int empty_fold = 0;   // lanes < NT: the empty bits of "their" target after the mask wrappers
        if (FOLD && fast) {
            const int env = env0 + i;
            if (f_rel) {   // fp64 locations of all entities (RelativeCoordinates subtracts in fp64: fp32 would lose 1e-4 to cancellation)
#pragma unroll
                for (int j = 0; j < FJ; ++j) {
                    const int k = lane + 32 * j;
                    if (k < EALL) { fpos[2 * k] = fx_next[j]; fpos[2 * k + 1] = fy_next[j]; }
                }
                if (i + 1 < nvalid) load_locations(i + 1);   // in flight while this environment is packed
            }
            if (f_mask) {
                // lane r < R owns observer row r: its mask words go through the mask wrappers in their order;
                // lanes < NT also carry target t's empty bits (EnhancedObservation / SharedFieldOfView rewrite them)
                constexpr uint32_t CAMS = NC > 0 ? ((1u << NC) - 1u) : 0u, TGTS = ((1u << NT) - 1u) << 8;
                constexpr uint32_t OBS0 = MW == 1 ? (NO > 0 ? (((1u << NO) - 1u) << 16) : 0u) : 0u;
                constexpr uint32_t OBS1 = MW == 2 ? (NO >= 32 ? 0xffffffffu : ((1u << (NO & 31)) - 1u)) : 0u;
                constexpr uint32_t CAM_LANES = NC > 0 ? ((1u << NC) - 1u) : 0u, TGT_LANES = ((1u << NT) - 1u) << NC, TLOW = (1u << NT) - 1u;
                uint32_t w0 = lane < R ? m[lane * MW] : 0u, w1 = (MW == 2 && lane < R) ? m[lane * MW + 1] : 0u;
                int emp = lane < NT ? tp_empty(__float_as_uint(v[S::V_T + 3 * lane + 2])) : 0;
                const bool cam_lane = lane < NC, tgt_lane = lane >= NC && lane < R;
                for (int k = 0; k < n_mask; ++k) {   // warp-uniform
                    const int op = (int)((mask_ops >> (4 * k)) & 15u);
                    if (op == MATE_OBS_ENHANCED_CAMERA) { if (cam_lane) { w0 = CAMS | TGTS | OBS0; w1 = OBS1; } }
                    else if (op == MATE_OBS_ENHANCED_TARGET) {
                        if (tgt_lane) { w0 = CAMS | TGTS | OBS0; w1 = OBS1; }
                        // np.logical_not(remaining_cargoes).all(axis=-1) (enhanced_observation.py:107-109)
                        const uint4 c0 = p.cargo[env], c1 = p.cargo[bp + env];
                        emp = (int)((c0.x | c0.y) == 0u) | ((int)((c0.z | c0.w) == 0u) << 1) | ((int)((c1.x | c1.y) == 0u) << 2) | ((int)((c1.z | c1.w) == 0u) << 3);
                    } else if (op == MATE_OBS_SHARED_CAMERA) {
                        if (NC > 0 && cam_lane) {   // "or" over the team's rows, teammates always (shared_field_of_view.py:90-110)
                            w0 = __reduce_or_sync(CAM_LANES, w0) | CAMS;
                            if (MW == 2) w1 = __reduce_or_sync(CAM_LANES, w1);
                        }
                    } else if (op == MATE_OBS_SHARED_TARGET) {
                        if (tgt_lane) {
                            w0 = __reduce_or_sync(TGT_LANES, w0) | TGTS;
                            if (MW == 2) w1 = __reduce_or_sync(TGT_LANES, w1);
                        }
                        if (lane < NT) emp = (int)__reduce_or_sync(TLOW, (uint32_t)emp);
                    }
                }
                if (lane < R) { mmod[lane * MW] = w0; if (MW == 2) mmod[lane * MW + 1] = w1; }
                empty_fold = emp;
                m = mmod;
            }
            __syncwarp();
        }
        // Target.state public part (entities.py:631-637), Camera.state public part (entities.py:313-324)
        const uint32_t tpk = __float_as_uint(v[S::V_T + 3 * t_idx + 2]);
        const float t0 = v[S::V_T + 3 * t_idx], t1 = v[S::V_T + 3 * t_idx + 1];
        const int goal = tp_goal(tpk), weight = tp_weight(tpk);
        const float t3 = (goal >= 0 && weight > 0) ? 1.f : 0.f;
        float c0 = 0.f, c1 = 0.f, c3 = 0.f, c4 = 0.f, c5 = 0.f;
        if (NC > 0) {
            const float* cv = v + S::V_C + CV * c_idx;
            c0 = cv[0]; c1 = cv[1]; c3 = cv[3]; c4 = cv[4]; c5 = cv[2];
        }
        const bool plain = !(FOLD && fast);
        // own rows, the entries that change: lane t < NT holds target t, lane c < NC holds camera c
        const int capacity = tp_capacity(tpk), empty = (FOLD && f_mask) ? empty_fold : tp_empty(tpk);
        float sg[NW], se[NW];
#pragma unroll
        for (int w = 0; w < NW; ++w) { sg[w] = (goal == w) ? (float)weight : 0.f; se[w] = (float)((empty >> w) & 1); }
        const float s_step = capacity == 1 ? f_step1 : f_step2, s_cap = (float)capacity;

        if constexpr (FOLD) {
            if (fast) {
                // one entity kind at a time (values -> wrappers -> staged rows): fewer live registers than the plain path
                auto observer = [&](const int midx) { const int row = midx / MW; return row < NC ? NT + NO + row : row - NC; };
                uint32_t mw[NRND];   // all mask words first: the loads are in flight together
#pragma unroll
                for (int rd = 0; rd < NRND; ++rd) mw[rd] = m[m_idx[rd]];
                {   // targets + flag
                    float2 a[5];
#pragma unroll
                    for (int j = 0; j < 5; ++j) a[j] = f_resc ? aff_own[ObsLayout::AFF_TGT + j] : make_float2(1.f, 0.f);
                    double ex = 0.0, ey = 0.0;
                    if (f_rel) { ex = fpos[2 * t_idx]; ey = fpos[2 * t_idx + 1]; }
                    // the lane keeps its entity for all rounds: the entries are rescaled once per environment, a round selects
                    // between them and the image of zero (only relative locations depend on the observer)
                    const float e_in[5] = {t0, t1, f_sr, t3, 1.f};
                    float sv[5];
#pragma unroll
                    for (int j = 0; j < 5; ++j) sv[j] = f_resc ? fmaf(e_in[j], a[j].x, a[j].y) : e_in[j];
#pragma unroll
                    for (int rd = 0; rd < RND_T; ++rd) {
                        const bool hit = (mw[rd] & t_bit) != 0u;
                        float x[5];
#pragma unroll
                        for (int j = 0; j < 5; ++j) x[j] = hit ? sv[j] : a[j].y;
                        if (f_rel && hit) {
                            const int ko = observer(m_idx[rd]);
                            const float rx = (float)(ex - fpos[2 * ko]), ry = (float)(ey - fpos[2 * ko + 1]);
                            x[0] = f_resc ? fmaf(rx, a[0].x, a[0].y) : rx; x[1] = f_resc ? fmaf(ry, a[1].x, a[1].y) : ry;
                        }
                        if ((on_bits >> rd) & 1u) {
                            float* q = q_ptr[rd];
#pragma unroll
                            for (int j = 0; j < 5; ++j) q[j] = x[j];
                        }
                    }
                }
                if (NO > 0) {   // obstacles + flag
                    float2 a[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) a[j] = f_resc ? aff_own[ObsLayout::AFF_OBS + j] : make_float2(1.f, 0.f);
                    double ex = 0.0, ey = 0.0;
                    if (f_rel) { ex = fpos[2 * (NT + o_idx)]; ey = fpos[2 * (NT + o_idx) + 1]; }
                    const float e_in[4] = {ob.x, ob.y, ob.z, 1.f};
                    float sv[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) sv[j] = f_resc ? fmaf(e_in[j], a[j].x, a[j].y) : e_in[j];
#pragma unroll
                    for (int rd = 0; rd < RND_O; ++rd) {
                        const bool hit = (mw[RND_T + rd] & o_bit) != 0u;
                        float x[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) x[j] = hit ? sv[j] : a[j].y;
                        if (f_rel && hit) {
                            const int ko = observer(m_idx[RND_T + rd]);
                            const float rx = (float)(ex - fpos[2 * ko]), ry = (float)(ey - fpos[2 * ko + 1]);
                            x[0] = f_resc ? fmaf(rx, a[0].x, a[0].y) : rx; x[1] = f_resc ? fmaf(ry, a[1].x, a[1].y) : ry;
                        }
                        if ((on_bits >> (RND_T + rd)) & 1u) {
                            float* q = q_ptr[RND_T + rd];
#pragma unroll
                            for (int j = 0; j < 4; ++j) q[j] = x[j];
                        }
                    }
                }
                if (NC > 0) {   // cameras + flag
                    float2 a[7];
#pragma unroll
                    for (int j = 0; j < 7; ++j) a[j] = f_resc ? aff_own[ObsLayout::AFF_CAM + j] : make_float2(1.f, 0.f);
                    double ex = 0.0, ey = 0.0;
                    if (f_rel) { ex = fpos[2 * (NT + NO + c_idx)]; ey = fpos[2 * (NT + NO + c_idx) + 1]; }
                    const float e_in[7] = {c0, c1, f_crad, c3, c4, c5, 1.f};
                    float sv[7];
#pragma unroll
                    for (int j = 0; j < 7; ++j) sv[j] = f_resc ? fmaf(e_in[j], a[j].x, a[j].y) : e_in[j];
#pragma unroll
                    for (int rd = 0; rd < RND_C; ++rd) {
                        const bool hit = (mw[NRND - RND_C + rd] & c_bit) != 0u;
                        float x[7];
#pragma unroll
                        for (int j = 0; j < 7; ++j) x[j] = hit ? sv[j] : a[j].y;
                        if (f_rel && hit) {
                            const int ko = observer(m_idx[NRND - RND_C + rd]);
                            const float rx = (float)(ex - fpos[2 * ko]), ry = (float)(ey - fpos[2 * ko + 1]);
                            x[0] = f_resc ? fmaf(rx, a[0].x, a[0].y) : rx; x[1] = f_resc ? fmaf(ry, a[1].x, a[1].y) : ry;
                        }
                        if ((on_bits >> (NRND - RND_C + rd)) & 1u) {
                            float* q = q_ptr[NRND - RND_C + rd];
#pragma unroll
                            for (int j = 0; j < 7; ++j) q[j] = x[j];
                        }
                    }
                }
            }
        }
        if (plain) {
        float vt[RND_T][5], vo[NO > 0 ? RND_O : 1][4], vc[NC > 0 ? RND_C : 1][7];
#pragma unroll
            for (int rd = 0; rd < RND_T; ++rd) {   // targets + flag
                const bool hit = (m[m_idx[rd]] & t_bit) != 0u;
                vt[rd][0] = hit ? t0 : 0.f; vt[rd][1] = hit ? t1 : 0.f; vt[rd][2] = hit ? f_sr : 0.f; vt[rd][3] = hit ? t3 : 0.f; vt[rd][4] = hit ? 1.f : 0.f;
            }
            if (NO > 0) {
#pragma unroll
                for (int rd = 0; rd < RND_O; ++rd) {   // obstacles: Obstacle.state (entities.py:147-148) + flag
                    const bool hit = (m[m_idx[RND_T + rd]] & o_bit) != 0u;
                    vo[rd][0] = hit ? ob.x : 0.f; vo[rd][1] = hit ? ob.y : 0.f; vo[rd][2] = hit ? ob.z : 0.f; vo[rd][3] = hit ? 1.f : 0.f;
                }
            }
            if (NC > 0) {
#pragma unroll
                for (int rd = 0; rd < RND_C; ++rd) {   // cameras + flag
                    const bool hit = (m[m_idx[NRND - RND_C + rd]] & c_bit) != 0u;
                    vc[rd][0] = hit ? c0 : 0.f; vc[rd][1] = hit ? c1 : 0.f; vc[rd][2] = hit ? f_crad : 0.f; vc[rd][3] = hit ? c3 : 0.f;
                    vc[rd][4] = hit ? c4 : 0.f; vc[rd][5] = hit ? c5 : 0.f; vc[rd][6] = hit ? 1.f : 0.f;
                }
            }
        if (has_ops && i > 0) stage_constants();
#pragma unroll
            for (int rd = 0; rd < RND_T; ++rd) {
                if ((on_bits >> rd) & 1u) {
                    float* q = q_ptr[rd];
                    q[0] = vt[rd][0]; q[1] = vt[rd][1]; q[2] = vt[rd][2]; q[3] = vt[rd][3]; q[4] = vt[rd][4];
                }
            }
            if (NO > 0) {
#pragma unroll
                for (int rd = 0; rd < RND_O; ++rd) {
                    if ((on_bits >> (RND_T + rd)) & 1u) {
                        float* q = q_ptr[RND_T + rd];
                        if (ORND.cls[rd] >= 0) {
                            // every lane's 16-byte slot of this round has the same alignment, known at compile time
                            const int al = ORND.cls[rd];
                            if (al == 0) {
                                *reinterpret_cast<float4*>(q) = make_float4(vo[rd][0], vo[rd][1], vo[rd][2], vo[rd][3]);
                            } else if (al == 2) {
                                *reinterpret_cast<float2*>(q) = make_float2(vo[rd][0], vo[rd][1]);
                                *reinterpret_cast<float2*>(q + 2) = make_float2(vo[rd][2], vo[rd][3]);
                            } else {
                                q[0] = vo[rd][0];
                                *reinterpret_cast<float2*>(q + 1) = make_float2(vo[rd][1], vo[rd][2]);
                                q[3] = vo[rd][3];
                            }
                        } else {
                            q[0] = vo[rd][0]; q[1] = vo[rd][1]; q[2] = vo[rd][2]; q[3] = vo[rd][3];
                        }
                    }
                }
            }
            if (NC > 0) {
#pragma unroll
                for (int rd = 0; rd < RND_C; ++rd) {
                    if ((on_bits >> (NRND - RND_C + rd)) & 1u) {
                        float* q = q_ptr[NRND - RND_C + rd];
                        q[0] = vc[rd][0]; q[1] = vc[rd][1]; q[2] = vc[rd][2]; q[3] = vc[rd][3]; q[4] = vc[rd][4]; q[5] = vc[rd][5]; q[6] = vc[rd][6];
                    }
                }
            }
        }
        {
            // own rows, the entries that change: lane t < NT writes target row t, lane NT + k (k < NC) the row of camera
            // c_idx (NC consecutive lanes hold NC different cameras) -- one instruction stream for both kinds of rows.
            // With wrappers folded in: RescaledObservation is one FMA per entry, RelativeCoordinates moves the eight
            // warehouse coordinates of the row (the agent's own location stays absolute, mate/constants.py:372-427)
            const bool is_t = lane < NT && (WANT_T || has_ops), is_c = NC > 0 && lane >= NT && lane < NT + NC && (WANT_C || has_ops);
            float* const q = is_t ? self_t : self_c;
            const int aff0 = is_t ? ObsLayout::AFF_TSELF : ObsLayout::AFF_CSELF;
            auto put = [&](const int j, const float x) { q[j] = (FOLD && f_resc) ? fmaf(x, aff_own[aff0 + j].x, aff_own[aff0 + j].y) : x; };
            if (is_t || is_c) {
                put(0, is_t ? t0 : c0); put(1, is_t ? t1 : c1); put(3, is_t ? t3 : c3); put(4, is_t ? s_step : c4); put(5, is_t ? s_cap : c5);
                if (FOLD && f_rel) {
                    const int ko = is_t ? lane : NT + NO + c_idx;
                    float* const pr = q - ObsLayout::SELF;   // the row's preserved block
                    const double ox = fpos[2 * ko], oy = fpos[2 * ko + 1];
#pragma unroll
                    for (int j = 0; j < 2 * NW; ++j) {
                        const float wh = (j == 0 || j == 1 || j == 3 || j == 6) ? 925.f : -925.f;   // (+,+) (-,+) (-,-) (+,-)
                        const float x = (float)((double)wh - ((j & 1) ? oy : ox));
                        constexpr int WH = ObsLayout::WAREHOUSE, AW = ObsLayout::AFF_PRES + WH;
                        pr[WH + j] = f_resc ? fmaf(x, aff_own[AW + j].x, aff_own[AW + j].y) : x;
                    }
                }
            }
            if (is_t) {
#pragma unroll
                for (int w = 0; w < NW; ++w) { put(6 + w, sg[w]); put(10 + w, se[w]); }
            }
        }
        // ---- registered observation wrappers (EnhancedObservation, SharedFieldOfView, RelativeCoordinates,
        //      RescaledObservation): applied to the staged rows, no extra pass over the observation tensors
        if (FOLD && has_ops) {
            __syncwarp();
            fold_obs_ops<NC, NT, NO>(p, env0 + i, stage, ops_scratch);
            __syncwarp();
        }
        // ---- staged rows -> HBM
        static_assert(!(S::DENSE16 && S::CAM_SKEW != 0), "the 16-byte copy of the whole block expects dense camera rows");
        __syncwarp();
        if constexpr (ROWS == ROWS_BOTH && !F16 && S::DENSE16) {
            // plain 16-byte copies of the whole block: every warp store covers 512 contiguous bytes; unlike a bulk copy
            // there is nothing to wait for before the block is reused (see DESIGN.md)
            const float4* src4 = reinterpret_cast<const float4*>(stage);
            float4* cam4 = reinterpret_cast<float4*>(cam_obs0 + (size_t)i * S::CAM_ROW);
            float4* tgt4 = reinterpret_cast<float4*>(tgt_obs0 + (size_t)i * S::TGT_ROW) - S::CAM_ROW / 4;
            constexpr int NZ = S::STAGE_FLOATS / 4;
#pragma unroll
            for (int it = 0; it < (NZ + 31) / 32; ++it) {
                const int k = it * 32 + lane;
                if (it * 32 + 32 <= NZ || k < NZ) {
                    const float4 x = src4[k];
                    float4* dst = (k < S::CAM_ROW / 4 ? cam4 : tgt4) + k;
                    __stcs(dst, x);
                }
            }
        } else {
            if constexpr (WANT_C) store_team_rows<OutT, S::CAM_ROW, DC, DCS - DC>(cam_obs0 + (size_t)i * S::CAM_ROW, stage);
            if constexpr (WANT_T) store_team_rows<OutT, S::TGT_ROW, DT, 0>(tgt_obs0 + (size_t)i * S::TGT_ROW, stage + S::STAGE_CAM);
        }
        __syncwarp();
    }
}

// joint_observation for the rows the launch's pointers ask for (without cameras, "targets only" is "both"); no pointer:
// nothing.  Each row set is an instantiation of its own, so the step kernel keeps one call per (FOLD, OutT) and the
// both-teams packer its code (ptxas allocates registers across the calls of a kernel).
template <int NC, int NT, int NO, bool FOLD, class OutT>
__device__ __noinline__ void pack_observations(const Params& p, const int env0, const int nvalid, float* stage,
                                               const uint32_t* mk, const float* val, float* ops_scratch) {
    const bool want_c = NC > 0 && p.cam_obs != nullptr, want_t = p.tgt_obs != nullptr;
    if (want_t && (want_c || NC == 0)) pack_rows<NC, NT, NO, FOLD, OutT, ROWS_BOTH>(p, env0, nvalid, stage, mk, val, ops_scratch);
    else if constexpr (NC > 0) {
        if (want_c) pack_rows<NC, NT, NO, FOLD, OutT, ROWS_CAM>(p, env0, nvalid, stage, mk, val, ops_scratch);
        else if (want_t) pack_rows<NC, NT, NO, FOLD, OutT, ROWS_TGT>(p, env0, nvalid, stage, mk, val, ops_scratch);
    }
}

// Camera.sight_range_at (entities.py:507-511) for a list of (environment, camera, bearing) queries: the same
// on-the-fly polyline evaluation the occlusion tests use, exposed for direct comparison with the reference's tables.
template <int NC, int NO>
__global__ void fov_range_kernel(const Params p, const int32_t* __restrict__ env, const int32_t* __restrict__ camera,
                                 const double* __restrict__ angle_deg, double* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int e = min(max(env[i], 0), p.num_envs - 1), c = min(max(camera[i], 0), (NC > 0 ? NC : 1) - 1);
    double a = fmod(angle_deg[i] + 180.0, 360.0);   // mate/utils.py:155-158
    if (a < 0.0) a += 360.0;
    a -= 180.0;
    if (NC == 0) { out[i] = 0.0; return; }
    if (NO == 0) { out[i] = p.cam_rmax; return; }
    const size_t bp = p.bpad;
    double sn, cs;
    sincospi(a * (1.0 / 180.0), &sn, &cs);
    out[i] = sight_range_at<NO>(ObsRef{p.obs_x + e, p.obs_y + e, p.obs_r + e, bp}, p.cam_x[(size_t)c * bp + e],
                                p.cam_y[(size_t)c * bp + e], p.cam_rmax, a, cs, sn);
}

// =============================================================================================
// The fused kernel
// =============================================================================================
template <int NC, int NT, int NO>
__global__ void __launch_bounds__(Shape2<NC, NT, NO>::WARPS * 32, kStepMinCtas)
mate_step_kernel2(const __grid_constant__ Params p) {
    using S = Shape2<NC, NT, NO>;
    static_assert(NC <= 8 && NT <= 8 && NO <= 32, "mask layout: 8 cameras, 8 targets, 32 obstacles");
    constexpr int MW = S::MW, CV = S::CV;
    constexpr int NCX = NC > 0 ? NC : 1;
    constexpr uint32_t FULL = 0xffffffffu;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned char* wbase = smem_raw + (size_t)warp * p.warp_stride;
    float* stage = reinterpret_cast<float*>(wbase + S::OFF_STAGE);
    uint32_t* mk = reinterpret_cast<uint32_t*>(wbase + S::OFF_MASK);      // [32][MSTRIDE]
    float* val = reinterpret_cast<float*>(wbase + S::OFF_VAL);            // [32][VSTRIDE]
    uint16_t* queue = reinterpret_cast<uint16_t*>(wbase + S::OFF_Q);
    uint16_t* queue2 = reinterpret_cast<uint16_t*>(wbase + S::OFF_Q2);
    uint32_t* mymk = mk + lane * S::MSTRIDE;
    float* myval = val + lane * S::VSTRIDE;
    float* mycam = myval + S::V_C;

    // A warp tile is p.tile_envs (32, 16 or 8) consecutive environments: small batches are cut into more, smaller tiles so
    // that the machine still holds ~14 warps per SM (the launch is latency bound); the lanes beyond the tile idle along.
    const int tile_envs = p.tile_envs;
    const int env0 = (blockIdx.x * S::WARPS + warp) * tile_envs;   // first env of this warp
    if (env0 >= p.num_envs) return;                            // warps never synchronise with each other
    const int e = env0 + lane;
    const bool env_ok = lane < tile_envs && e < p.num_envs;
    // lanes without an environment mirror a live one (reads only; same lines, same branches as their twin); they feed no queue
    const int twin = env0 + (lane & (tile_envs - 1));
    const int er = env_ok ? e : (twin < p.num_envs ? twin : p.num_envs - 1);
    const size_t bp = p.bpad;
    const int mode = p.mode;

    TL_MARK(0);
    // ------------------------------------------------------------------ per-env scalars
    const uint4 ea = p.env_a[er];
    const int4 eb = p.env_b[er];
    unsigned long long ccw = NC >= 2 ? p.cc_clear[er] : 0ull;   // static camera <-> camera lines of sight (per episode)
    Cargo cargo;
    cargo.aw[0] = ea.x; cargo.aw[1] = ea.y;
    int episode_step = (int)ea.z, delivered = (int)ea.w;
    int ep_reward = eb.x, delayed_ep_reward = eb.y, episode_id = eb.w;
    float coverage_sum = __int_as_float(eb.z);
    bool cargo_loaded = false, cargo_dirty = false;
    // MODE_PREPARE (this launch's Params address the second state block): the envs whose prepared state is
    // not the one for their next episode are re-initialised here, everything else is left alone
    bool need = false;
    if (mode == MODE_PREPARE) {
        episode_id = p.live_env_b[er].w;
        need = env_ok && p.ready[e] != (uint32_t)(episode_id + 1);
        if (!__any_sync(FULL, need)) return;
    }

    if (mode == MODE_STEP) {   // cargo tables -> L2: _assign_goals reads them ~50 us from now, when every other warp is storing rows
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p.cargo + er));
        asm volatile("prefetch.global.L2 [%0];" :: "l"(p.cargo + bp + er));
    }

    // ------------------------------------------------------------------ _simulate (environment.py:1326-1354)
    {   // Camera.simulate (entities.py:347-360); the next camera's state is fetched while this one is derived
        double nx_ = 0, ny_ = 0, nphi_ = 0, nth_ = 0;
        float2 na_ = make_float2(0.f, 0.f);
        if (NC > 0) {
            nx_ = p.cam_x[er]; ny_ = p.cam_y[er]; nphi_ = p.cam_phi[er]; nth_ = p.cam_theta[er];
            if (mode == MODE_STEP) na_ = reinterpret_cast<const float2*>(p.cam_act)[(size_t)er * NC];
        }
#pragma unroll 1
        for (int c = 0; c < NC; ++c) {
            const double x = nx_, y = ny_;
            double phi = nphi_, theta = nth_;
            const float2 a = na_;
            if (c + 1 < NC) {
                const size_t i = (size_t)(c + 1) * bp + er;
                nx_ = p.cam_x[i]; ny_ = p.cam_y[i]; nphi_ = p.cam_phi[i]; nth_ = p.cam_theta[i];
                if (mode == MODE_STEP) na_ = reinterpret_cast<const float2*>(p.cam_act)[(size_t)er * NC + c + 1];
            }
            if (mode == MODE_STEP) {
                const double da = fmin(fmax((double)a.x, -p.cam_rot_step), p.cam_rot_step);
                const double dv = fmin(fmax((double)a.y, -p.cam_zoom_step), p.cam_zoom_step);
                phi = normalize_angle(phi + da);
                theta = fmin(fmax(theta + dv, p.cam_min_view), 180.0);
                if (env_ok) { p.cam_phi[(size_t)c * bp + e] = phi; p.cam_theta[(size_t)c * bp + e] = theta; }
            }
            store_camera(mycam + CV * c, x, y, phi, theta, p.cam_area_product);
        }
    }
    {   // Target.simulate (entities.py:645-668): fast path = no disc within reach of the step
        uint32_t slow = 0;     // targets that may touch a disc: re-simulated exactly below
        // per target, the discs (obstacles, then cameras) within reach of its step: the exact re-simulation only looks at those
        // (worth its registers where there are many discs: Navigation's 32; with 9 the full scan is as fast, measured)
        constexpr bool REACH_MASKS = NO > 16 && NO + NC <= 32;
        uint32_t near[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) near[t] = 0u;
        if (mode == MODE_STEP) {
            // fp32 broad phase on the old locations: a disc farther than step_size + R (+ slack for fp32
            // rounding) cannot touch the step
            float otx[NT], oty[NT];
#pragma unroll
            for (int t = 0; t < NT; ++t) { otx[t] = (float)p.tgt_x[(size_t)t * bp + er]; oty[t] = (float)p.tgt_y[(size_t)t * bp + er]; }
            const float fb = (float)p.tgt_step_size * 1.00001f + 0.01f;
            // (unrolled for small NO: the loads of all discs are in flight together)
#pragma unroll (NO <= 12 ? 12 : 4)
            for (int o = 0; o < NO; ++o) {
                const float4 ob = p.obs_f4[(size_t)o * bp + er];
                const float reach = fb + ob.z, reach2 = reach * reach;
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const float dx = ob.x - otx[t], dy = ob.y - oty[t];
                    const uint32_t hit = (uint32_t)(!(dx * dx + dy * dy > reach2));
                    slow |= hit << t;
                    if (REACH_MASKS) near[t] |= hit << o;
                }
            }
            const float reach_c = fb + (float)p.cam_radius, reach_c2 = reach_c * reach_c;
#pragma unroll 1
            for (int c = 0; c < NC; ++c) {
                const float cx = mycam[CV * c], cy = mycam[CV * c + 1];
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const float dx = cx - otx[t], dy = cy - oty[t];
                    const uint32_t hit = (uint32_t)(!(dx * dx + dy * dy > reach_c2));
                    slow |= hit << t;
                    if (REACH_MASKS) near[t] |= hit << ((NO + c) & 31);
                }
            }
        }
        if (!env_ok) slow = 0u;
        if (NO > 0 && slow != 0) prefetch_discs64<NO>(p, er);
        double ntx_ = p.tgt_x[er], nty_ = p.tgt_y[er];
        uint32_t npk_ = p.tgt_pack[er];
        float2 nta_ = make_float2(0.f, 0.f);
        if (mode == MODE_STEP) nta_ = reinterpret_cast<const float2*>(p.tgt_act)[(size_t)er * NT];
#pragma unroll 1
        for (int t = 0; t < NT; ++t) {   // the next target's state is fetched while this one is stepped
            double tx = ntx_, ty = nty_;
            uint32_t tpack = npk_;
            const float2 a = nta_;
            if (t + 1 < NT) {
                const size_t i = (size_t)(t + 1) * bp + er;
                ntx_ = p.tgt_x[i]; nty_ = p.tgt_y[i]; npk_ = p.tgt_pack[i];
                if (mode == MODE_STEP) nta_ = reinterpret_cast<const float2*>(p.tgt_act)[(size_t)er * NT + t + 1];
            }
            if (mode == MODE_STEP && !((slow >> t) & 1)) {
                const int cap = tp_capacity(tpack);   // 1 or 2
                const double step_size = cap == 1 ? p.tgt_step_size : p.tgt_step_size * 0.5;
                double vx = (double)a.x, vy = (double)a.y;
                const double n2 = vx * vx + vy * vy;
                if (n2 > step_size * step_size * (1.0 - 1e-12)) {
                    const double n = sqrt(n2);
                    if (n > step_size) {   // Vector2D.norm setter (utils.py:223-229), see DESIGN.md
                        const double k = step_size / n;
                        vx *= k; vy *= k;
                    }
                }
                const double desx = tx + vx, desy = ty + vy;
                const double nx = fmin(fmax(desx, -kTerrain), kTerrain);
                const double ny = fmin(fmax(desy, -kTerrain), kTerrain);
                const int colliding = !(fabs(nx - desx) <= 1e-6 && fabs(ny - desy) <= 1e-6);
                tx = nx; ty = ny;
                tpack = (tpack & ~(1u << 27)) | ((uint32_t)colliding << 27);
                if (env_ok) { p.tgt_x[(size_t)t * bp + e] = tx; p.tgt_y[(size_t)t * bp + e] = ty; }
            }
            myval[S::V_T + 3 * t + 0] = (float)tx; myval[S::V_T + 3 * t + 1] = (float)ty;
            myval[S::V_T + 3 * t + 2] = __uint_as_float(tpack);
        }
        // exact re-simulation of the targets near a disc: queued and processed 32 at a time, one per lane
        __syncwarp();
        TL_MARK(1);
        {
            int count = 0;   // warp-uniform
            for (;;) {
                const bool more = __any_sync(FULL, slow != 0);
                if (more) {
                    const bool has = slow != 0;
                    const int t = has ? (__ffs(slow) - 1) : 0;
                    slow &= slow - 1;
                    const uint32_t ballot = __ballot_sync(FULL, has);
                    if (has) queue[count + __popc(ballot & ((1u << lane) - 1u))] = (uint16_t)((lane << 8) | t);
                    count += __popc(ballot);
                    __syncwarp();
                }
                if (count >= 32 || (!more && count > 0)) {
                    const int n = min(count, 32);
                    count -= n;
                    process_slow_targets<NC, NT, NO, S>(p, env0, val, queue, count, n, near);
                    __syncwarp();
                }
                if (!more && count == 0) break;
            }
        }
    }

    TL_MARK(2);
    uint32_t tdone_bits = 0;            // target_dones
    int reward_i = 0, delayed_i = 0;    // this step's rewards (integers)
    int done = 0;
    float cov_now = 0.f, cov_real = 0.f;
    bool auto_reset_needed = false;
    int draw_step = (mode == MODE_STEP) ? episode_step + 1 : episode_step;
    RngKey key{p.seed, (uint32_t)(p.env_index_base + e), (uint32_t)episode_id};

    const float fsr = (float)p.tgt_sight_range;
    const float fsr2 = fsr * fsr, fsrc = fsr + (float)p.cam_radius, fsrc2 = fsrc * fsrc;
    const double sr = p.tgt_sight_range, src = sr + p.cam_radius;

#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        const bool do_reset = (pass == 0)
            ? (mode == MODE_PREPARE ? need : ((mode == MODE_RESET) && env_ok && (p.env_mask == nullptr || p.env_mask[e] != 0)))
            : auto_reset_needed;
        // auto-reset: adopt the prepared state (and first view) of the next episode if it is ready
        bool adopted = false;
        if (do_reset && mode == MODE_STEP && p.next != nullptr && p.replay_transmit == nullptr && p.replay_choice == nullptr)
            adopted = ld_acquire_u32(p.ready + e) == (uint32_t)(episode_id + 1);
        const bool view_active = mode == MODE_PREPARE ? need : (((pass == 0) || do_reset) && !adopted);
        // ============================================================== reset (environment.py:679-775)
        if (__any_sync(FULL, do_reset)) {
            {
                uint4 c0 = make_uint4(0, 0, 0, 0), c1 = c0, ea2 = c0;
                unsigned long long cc = 0ull;
                if (adopted) {   // lane-private part: in flight while the warp copies the rest
                    const Params& nx = *p.next;
                    const int en = e + p.next_offset;
                    c0 = nx.cargo[en]; c1 = nx.cargo[bp + en]; ea2 = nx.env_a[en];
                    if (NC >= 2) cc = nx.cc_clear[en];
                }
                const uint32_t adopting = __ballot_sync(FULL, adopted);
                if (adopting != 0u) adopt_prepared_warp<NC, NT, NO, S>(p, *p.next, env0, adopting, val, mk);
                __syncwarp();
                if (adopted) {
                    cargo.rem[0] = c0.x; cargo.rem[1] = c0.y; cargo.rem[2] = c0.z; cargo.rem[3] = c0.w;
                    cargo.rem[4] = c1.x; cargo.rem[5] = c1.y; cargo.rem[6] = c1.z; cargo.rem[7] = c1.w;
                    cargo.aw[0] = ea2.x; cargo.aw[1] = ea2.y;
                    ccw = cc;
                    if (NC >= 2) p.cc_clear[e] = cc;
                }
            }
            if (adopted) {
                atomicAdd(&p.stats[6], 1.0f);   // auto-resets served from the prepared state
                cargo_loaded = true; cargo_dirty = true;
                episode_id += 1; key.episode = (uint32_t)episode_id;
                episode_step = 0; delivered = 0; ep_reward = 0; delayed_ep_reward = 0; coverage_sum = 0.f;
                tdone_bits = 0; draw_step = 0;
            } else if (do_reset) {
                if (mode == MODE_STEP) atomicAdd(&p.stats[7], 1.0f);   // auto-resets computed in place
                RngKey k2 = key;
                k2.episode = (uint32_t)(episode_id + 1);
                const uint32_t cap2 = reset_env_global<NC, NT, NO>(p, e, k2, &cargo);
                cargo_loaded = true; cargo_dirty = true;
                episode_id += 1; key.episode = (uint32_t)episode_id;
                episode_step = 0; delivered = 0; ep_reward = 0; delayed_ep_reward = 0; coverage_sum = 0.f;
                ccw = 0ull; tdone_bits = 0; draw_step = 0;
#pragma unroll 1
                for (int c = 0; c < NC; ++c) {
                    const size_t i = (size_t)c * bp + e;
                    store_camera(mycam + CV * c, p.cam_x[i], p.cam_y[i], p.cam_phi[i], p.cam_theta[i], p.cam_area_product);
                }
#pragma unroll 1
                for (int t = 0; t < NT; ++t) {
                    myval[S::V_T + 3 * t + 0] = (float)p.tgt_x[(size_t)t * bp + e];
                    myval[S::V_T + 3 * t + 1] = (float)p.tgt_y[(size_t)t * bp + e];
                    myval[S::V_T + 3 * t + 2] = __uint_as_float(pack_target(0, -1, 0, ((cap2 >> t) & 1) ? 2 : 1, 0, 0));
                }
            }
        }

        // ============================================================== _update_view (environment.py:1356-1388)
        unsigned long long pend = 0ull;     // bit c * NT + t: camera c reaches target t (range + sector)
        if (__any_sync(FULL, view_active)) {
            float ftx[NT], fty[NT];
#pragma unroll
            for (int t = 0; t < NT; ++t) { ftx[t] = myval[S::V_T + 3 * t]; fty[t] = myval[S::V_T + 3 * t + 1]; }
            float fcx[NCX], fcy[NCX];
#pragma unroll
            for (int c = 0; c < NC; ++c) { fcx[c] = mycam[CV * c]; fcy[c] = mycam[CV * c + 1]; }
            uint32_t crow[NCX], crow2[NCX], trow[NT], trow2[NT];
#pragma unroll
            for (int c = 0; c < NC; ++c) { crow[c] = bit_cam(c); crow2[c] = 0; }   // environment.py:1383-1384
#pragma unroll
            for (int t = 0; t < NT; ++t) { trow[t] = bit_tgt(t); trow2[t] = 0; }   // environment.py:1376-1377
            // ---- omnidirectional sensing by targets, Sensor.perceive (entities.py:229-232) ----
            // fp32 on squares; inside a 4e-6 relative band the fp64 test decides (resolve_band, rare)
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                uint32_t band_t = 0, band_c = 0;
#pragma unroll
                for (int u = t + 1; u < NT; ++u) {   // symmetric
                    const float dx = ftx[u] - ftx[t], dy = fty[u] - fty[t], d2 = dx * dx + dy * dy;
                    if (d2 < fsr2 * (1.0f - 4e-6f)) { trow[t] |= bit_tgt(u); trow[u] |= bit_tgt(t); }
                    else if (d2 <= fsr2 * (1.0f + 4e-6f)) band_t |= 1u << u;
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) {       // target t senses camera c
                    const float dx = fcx[c] - ftx[t], dy = fcy[c] - fty[t], d2 = dx * dx + dy * dy;
                    if (d2 < fsrc2 * (1.0f - 4e-6f)) trow[t] |= bit_cam(c);
                    else if (d2 <= fsrc2 * (1.0f + 4e-6f)) band_c |= 1u << c;
                }
                if (band_t | band_c) {
                    const double* ax = p.tgt_x + (size_t)t * bp + er;
                    const double* ay = p.tgt_y + (size_t)t * bp + er;
                    if (band_t) {
                        const uint32_t fix = resolve_band(p, er, ax, ay, band_t, 0, sr, false);
#pragma unroll
                        for (int u = t + 1; u < NT; ++u) if ((fix >> u) & 1) { trow[t] |= bit_tgt(u); trow[u] |= bit_tgt(t); }
                    }
                    if (band_c) trow[t] |= resolve_band(p, er, ax, ay, band_c, 1, src, false);   // bit_cam(c) == 1 << c
                }
            }
#pragma unroll (NO <= 12 ? 3 : 4)
            for (int o = 0; o < NO; ++o) {
                const float4 ob = p.obs_f4[(size_t)o * bp + er];
                const uint32_t obit = MW == 1 ? (1u << (16 + o)) : (1u << (o & 31));
                const float rtf = fsr + ob.z, rt2 = rtf * rtf;
                const float rcf = (float)p.cam_rmax + ob.z, rc2 = rcf * rcf;
                uint32_t band_t = 0, band_c = 0;
#pragma unroll
                for (int t = 0; t < NT; ++t) {       // target t senses obstacle o
                    const float dx = ob.x - ftx[t], dy = ob.y - fty[t], d2 = dx * dx + dy * dy;
                    if (d2 < rt2 * (1.0f - 4e-6f)) { if (MW == 1) trow[t] |= obit; else trow2[t] |= obit; }
                    else if (d2 <= rt2 * (1.0f + 4e-6f)) band_t |= 1u << t;
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) {       // camera c has obstacle o in its set (entities.py:363-368, strict <)
                    const float dx = ob.x - fcx[c], dy = ob.y - fcy[c], d2 = dx * dx + dy * dy;
                    if (d2 < rc2 * (1.0f - 4e-6f)) { if (MW == 1) crow[c] |= obit; else crow2[c] |= obit; }
                    else if (d2 <= rc2 * (1.0f + 4e-6f)) band_c |= 1u << c;
                }
                if (band_t | band_c) {
                    const size_t io = (size_t)o * bp + er;
                    const double orad = p.obs_r[io];
                    const uint32_t fix_t = band_t ? resolve_band(p, er, p.obs_x + io, p.obs_y + io, band_t, 0, sr + orad, false) : 0u;
                    const uint32_t fix_c = band_c ? resolve_band(p, er, p.obs_x + io, p.obs_y + io, band_c, 1, p.cam_rmax + orad, true) : 0u;
#pragma unroll
                    for (int t = 0; t < NT; ++t) if ((fix_t >> t) & 1) { if (MW == 1) trow[t] |= obit; else trow2[t] |= obit; }
#pragma unroll
                    for (int c = 0; c < NC; ++c) if ((fix_c >> c) & 1) { if (MW == 1) crow[c] |= obit; else crow2[c] |= obit; }
                }
            }
            // ---- cameras: range + sector (Camera.perceive, entities.py:494-501) ----
            // camera -> camera: the occlusion part is static within an episode and cached in `ccw`
            if (NC >= 2 && view_active && (ccw >> 63) == 0ull) {
                ccw = build_cc_cache<NC, NO>(p, er);
                if (env_ok) p.cc_clear[e] = ccw;
            }
            // With 8 cameras the fully unrolled loop nest (8 x 16 inlined range + sector tests, 50 KB of code) does not fit the
            // 32 KB instruction cache and a fifth of the warps' stalls are instruction fetches: the loop over the observing
            // camera stays rolled there (its own entries come from shared memory, its camera -> camera bits go through `cc_bits`)
            constexpr bool ROLL_C = NC >= kRollCamerasFrom;
            unsigned long long cc_bits = 0ull;
#pragma unroll (ROLL_C ? 1 : (NC > 0 ? NC : 1))
            for (int c = 0; c < NC; ++c) {
                const float* cv = mycam + CV * c;
                const float cs = cv[3], sn = cv[4], rs2 = cs * cs + sn * sn;   // heading scaled by Rs
                const float ch = cospif(cv[2] * (1.0f / 360.0f)), ch2 = ch * ch;
                const float mx = ROLL_C ? cv[0] : fcx[ROLL_C ? 0 : c], my = ROLL_C ? cv[1] : fcy[ROLL_C ? 0 : c];
                uint32_t reach_t = 0, band_t = 0, reach_c = 0, band_c = 0;
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const int reach = fov_reach32(mx, my, rs2, cs, sn, ch2, ftx[t], fty[t]);
                    reach_t |= (uint32_t)(reach == 1) << t;
                    band_t |= (uint32_t)(reach == 2) << t;
                }
#pragma unroll
                for (int j = 0; j < NC; ++j) {
                    if (!ROLL_C && j == c) continue;
                    const int reach = fov_reach32(mx, my, rs2, cs, sn, ch2, fcx[j], fcy[j]);
                    reach_c |= (uint32_t)(reach == 1) << j;
                    band_c |= (uint32_t)(reach == 2) << j;
                }
                if (ROLL_C) { reach_c &= ~(1u << c); band_c &= ~(1u << c); }   // the camera itself (the diagonal is set elsewhere)
                if (band_t) reach_t |= resolve_fov_band(p, er, c, band_t, 0);
                if (band_c) reach_c |= resolve_fov_band(p, er, c, band_c, 1);
                pend |= (unsigned long long)reach_t << (c * NT);
                // bits 8 j + c of ccw, j = 0..NC-1: camera c has a clear line of sight to camera j
                uint32_t clear_c = 0;
#pragma unroll
                for (int j = 0; j < NC; ++j) clear_c |= (uint32_t)((ccw >> (8 * j + c)) & 1ull) << j;
                if (ROLL_C) cc_bits |= (unsigned long long)(reach_c & clear_c) << (8 * c);
                else crow[ROLL_C ? 0 : c] |= reach_c & clear_c;   // bit_cam(j) == 1 << j
            }
            if (ROLL_C) {
#pragma unroll
                for (int c = 0; c < NC; ++c) crow[c] |= (uint32_t)(cc_bits >> (8 * c)) & 0xFFu;
            }
            if (view_active) {
#pragma unroll
                for (int c = 0; c < NC; ++c) { mymk[c * MW] = crow[c]; if (MW == 2) mymk[c * MW + 1] = crow2[c]; }
#pragma unroll
                for (int t = 0; t < NT; ++t) { mymk[(NC + t) * MW] = trow[t]; if (MW == 2) mymk[(NC + t) * MW + 1] = trow2[t]; }
            } else {
                pend = 0ull;
            }
        }
        __syncwarp();
        if (pass == 0) TL_MARK(3);
        // ---- then the stochastic transmittance draw and the occlusion test (entities.py:503-505) ----
        // All pending (camera, target) pairs of the warp's 32 environments go through a queue in shared
        // memory and are evaluated 32 at a time, one pair per lane; pairs the conservative occlusion
        // classification cannot decide go through a second queue to the exact polyline.
        if (NC > 0) {
            if (!env_ok) pend = 0ull;
            int count = 0, count2 = 0;   // warp-uniform
            for (;;) {
                const bool more = __any_sync(FULL, pend != 0ull);
                if (more) {
                    const bool has = pend != 0ull;
                    const int b = has ? (__ffsll((long long)pend) - 1) : 0;
                    pend &= pend - 1ull;
                    const uint32_t ballot = __ballot_sync(FULL, has);
                    const int pos = count + __popc(ballot & ((1u << lane) - 1u));
                    if (has) queue[pos] = (uint16_t)((lane << 8) | b);
                    count += __popc(ballot);
                    __syncwarp();
                }
                if (count >= 32 || (!more && count > 0)) {
                    const int n = min(count, 32);
                    count -= n;
                    const bool has = lane < n;
                    const uint32_t item = has ? queue[count + lane] : 0u;
                    const int src = item >> 8, b = item & 0xFF;
                    const int c = b / NT, t = b - c * NT;
                    const uint32_t src_episode = __shfl_sync(FULL, (uint32_t)episode_id, src);
                    const int src_draw = __shfl_sync(FULL, draw_step, src);
                    bool need_exact = false;
                    if (has) {
                        const int env = env0 + src;
                        const int envr = min(env, p.num_envs - 1);
                        bool sees;
                        if (p.replay_transmit) {
                            sees = p.replay_transmit[((size_t)envr * NC + c) * NT + t] != 0;
                        } else {
                            const RngKey k{p.seed, (uint32_t)(p.env_index_base + env), src_episode};
                            sees = rng_u01(k, STREAM_TRANSMIT, (uint32_t)src_draw * (uint32_t)(NC * NT) + (uint32_t)(c * NT + t)) < p.transmittance;
                        }
                        if (!sees) {
                            if (NO == 0 || p.transmittance_is_one) {
                                sees = true;   // polyline is the flat max_sight_range circle; dist <= rs <= Rmax
                            } else {
                                const float* v = val + src * S::VSTRIDE;
                                const float cx = v[S::V_C + CV * c], cy = v[S::V_C + CV * c + 1];
                                const int fast = occlusion_fast<NO>(p.obs_f4 + envr, bp, cx, cy, v[S::V_T + 3 * t] - cx, v[S::V_T + 3 * t + 1] - cy, (float)p.cam_rmax);
                                sees = fast == 1;
                                need_exact = fast == 2;
                                if (need_exact) prefetch_discs64<NO>(p, envr);
                            }
                        }
                        if (sees) atomicOr(&mk[src * S::MSTRIDE + c * MW], bit_tgt(t));
                    }
                    const uint32_t ballot2 = __ballot_sync(FULL, need_exact);
                    if (need_exact) queue2[count2 + __popc(ballot2 & ((1u << lane) - 1u))] = (uint16_t)item;
                    count2 += __popc(ballot2);
                    __syncwarp();
                }
                if (count2 >= 32 || (!more && count == 0 && count2 > 0)) {
                    const int n = min(count2, 32);
                    count2 -= n;
                    process_exact<NC, NT, NO, S>(p, env0, mk, queue2, count2, n);
                    __syncwarp();
                }
                if (!more && count == 0 && count2 == 0) break;
            }
            __syncwarp();
        }

        if (pass == 0) TL_MARK(4);
        // ============================================================== _assign_goals (environment.py:1271-1324)
        const bool step_goals = (pass == 0) && (mode == MODE_STEP);
        const bool goals_active = step_goals || (do_reset && !adopted);
        uint32_t tracked_bits = 0;
        {
            uint32_t any_c = 0;
#pragma unroll
            for (int c = 0; c < NC; ++c) any_c |= mymk[c * MW];
            tracked_bits = (any_c >> 8) & 0xFFu;
        }
        if (__any_sync(FULL, goals_active)) {
            int r = 0, delayed = 0;
            uint32_t in_bits = 0, whs = 0, old_goals = 0;
            if (goals_active) {
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    uint32_t tpack = __float_as_uint(myval[S::V_T + 3 * t + 2]);
                    int bounty = tp_bounty(tpack);
                    const int tracked = (tracked_bits >> t) & 1;
                    if (tracked && bounty > 0) r -= 1;
                    bounty = max(bounty - tracked, 0);
                    tpack = (tpack & ~0xFFFFu) | (uint32_t)bounty;
                    myval[S::V_T + 3 * t + 2] = __uint_as_float(tpack);
                    old_goals |= (uint32_t)(tp_goal(tpack) + 1) << (3 * t);
                    // the four warehouses sit at (+-925, +-925): the one this target could be in is given by
                    // the signs of its coordinates (constants.py:70-72 order: ++, -+, --, +-)
                    const float fx = myval[S::V_T + 3 * t], fy = myval[S::V_T + 3 * t + 1];
                    const float m = fmaxf(fabsf(fabsf(fx) - (float)kWarehouseCoord), fabsf(fabsf(fy) - (float)kWarehouseCoord));
                    bool inside = m < (float)kWarehouseRadius - 1e-3f;
                    if (!inside && m <= (float)kWarehouseRadius + 1e-3f) {
                        const double tx = p.tgt_x[(size_t)t * bp + er], ty = p.tgt_y[(size_t)t * bp + er];
                        inside = fmax(fabs(fabs(tx) - kWarehouseCoord), fabs(fabs(ty) - kWarehouseCoord)) <= kWarehouseRadius;
                    }
                    if (inside) {
                        const int wq = (fy >= 0.0f) ? ((fx >= 0.0f) ? 0 : 1) : ((fx >= 0.0f) ? 3 : 2);
                        in_bits |= 1u << t;
                        whs |= (uint32_t)wq << (2 * t);
                    }
                }
            }
            // Sequential over the targets standing in a warehouse, ascending index, one per lane and iteration
            while (__any_sync(FULL, in_bits != 0)) {
                if (in_bits != 0) {
                    if (!cargo_loaded) {
                        const uint4 c0 = p.cargo[er], c1 = p.cargo[bp + er];
                        cargo.rem[0] = c0.x; cargo.rem[1] = c0.y; cargo.rem[2] = c0.z; cargo.rem[3] = c0.w;
                        cargo.rem[4] = c1.x; cargo.rem[5] = c1.y; cargo.rem[6] = c1.z; cargo.rem[7] = c1.w;
                        cargo_loaded = true;
                    }
                    const int t = __ffs(in_bits) - 1;
                    in_bits &= in_bits - 1;
                    const int w = (whs >> (2 * t)) & 3;
                    const uint32_t tp_t = __float_as_uint(myval[S::V_T + 3 * t + 2]);
                    int goal = tp_goal(tp_t), weight = tp_weight(tp_t), bnty = tp_bounty(tp_t);
                    const int capacity = tp_capacity(tp_t);
                    int empty = tp_empty(tp_t);
                    bool proceed = true;
                    if (goal >= 0) {
                        if (goal == w) {
                            const int reward = weight * p.freight_scale + bnty;
                            r += reward;
                            delayed += reward - (weight * p.bounty_scale - bnty);
                            delivered += weight;
                            cargo.awaiting_add(goal, -weight);
                        } else {
                            proceed = false;
                        }
                    }
                    if (proceed) {
                        bnty = 0; weight = 0; goal = -1;
                        if (cargo.row_any(w)) {
                            int new_goal;
                            if (p.replay_choice) {
                                new_goal = p.replay_choice[(size_t)er * NT + t];
                            } else {   // np_random.choice(flatnonzero(remaining[w] > 0))
                                const uint32_t ncand = (uint32_t)((cargo.get(w, 0) > 0) + (cargo.get(w, 1) > 0) + (cargo.get(w, 2) > 0) + (cargo.get(w, 3) > 0));
                                const int pick = (int)rng_below(key, STREAM_CHOICE, (uint32_t)draw_step * (uint32_t)NT + (uint32_t)t, ncand);
                                new_goal = 0;
                                int seen = 0;
#pragma unroll
                                for (int gg = 0; gg < NW; ++gg) {
                                    if (cargo.get(w, gg) > 0) { if (seen == pick) new_goal = gg; ++seen; }
                                }
                            }
                            new_goal = min(max(new_goal, 0), NW - 1);
                            const int rem = cargo.get(w, new_goal);
                            weight = min(capacity, rem);
                            cargo.add(w, new_goal, -weight);
                            bnty = weight * p.bounty_scale;
                            goal = new_goal;
                        }
                        cargo_dirty = true;
                    }
                    // empty_bits for the warehouse the target stands in (environment.py:1317-1318)
                    empty = cargo.row_any(w) ? (empty & ~(1 << w)) : (empty | (1 << w));
                    myval[S::V_T + 3 * t + 2] = __uint_as_float(pack_target(bnty, goal, weight, capacity, empty, tp_colliding(tp_t)));
                }
            }
            if (goals_active) {
                tdone_bits = 0;
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const int old_goal = (int)((old_goals >> (3 * t)) & 7u) - 1;
                    const int goal = tp_goal(__float_as_uint(myval[S::V_T + 3 * t + 2]));
                    tdone_bits |= (uint32_t)((goal != old_goal) && (old_goal >= 0)) << t;
                }
            }
            if (step_goals) { reward_i = r; delayed_i = delayed; }
            if (do_reset && !adopted) {
                tdone_bits = 0; delivered = 0;   // environment.py:785-788
                // targets_start_with_cargoes (environment.py:789-812): sequential over targets without a goal
                if (p.start_with_cargoes) {
#pragma unroll 1
                    for (int t = 0; t < NT; ++t) {
                        const uint32_t tp_t = __float_as_uint(myval[S::V_T + 3 * t + 2]);
                        if (tp_goal(tp_t) >= 0) continue;
                        int perm[NW] = {0, 1, 2, 3};   // np_random.permutation(4)
#pragma unroll
                        for (int i = NW - 1; i >= 1; --i) {
                            const int k = (int)rng_below(key, STREAM_INIT_GOAL, (uint32_t)(t * 8 + i), (uint32_t)(i + 1));
                            int vi = perm[0], vk = perm[0];
#pragma unroll
                            for (int q = 1; q < NW; ++q) { vi = (q == i) ? perm[q] : vi; vk = (q == k) ? perm[q] : vk; }
#pragma unroll
                            for (int q = 0; q < NW; ++q) { if (q == i) perm[q] = vk; else if (q == k) perm[q] = vi; }
                        }
                        bool assigned = false;
#pragma unroll
                        for (int k = 0; k < NW; ++k) {
                            const int w = perm[k];
                            if (!assigned && cargo.row_any(w)) {
                                const uint32_t ncand = (uint32_t)((cargo.get(w, 0) > 0) + (cargo.get(w, 1) > 0) + (cargo.get(w, 2) > 0) + (cargo.get(w, 3) > 0));
                                const int pick = (int)rng_below(key, STREAM_INIT_GOAL, (uint32_t)(t * 8 + 4), ncand);
                                int goal = 0, seen = 0;
#pragma unroll
                                for (int gg = 0; gg < NW; ++gg) {
                                    if (cargo.get(w, gg) > 0) { if (seen == pick) goal = gg; ++seen; }
                                }
                                const int capacity = tp_capacity(tp_t);
                                const int weight = min(capacity, cargo.get(w, goal));
                                cargo.add(w, goal, -weight);
                                myval[S::V_T + 3 * t + 2] = __uint_as_float(pack_target(weight * p.bounty_scale, goal, weight, capacity, tp_empty(tp_t), 0));
                                assigned = true;
                            }
                        }
                    }
                }
            }
        }
        // coverage statistics of the current view (environment.py:966-972)
        if (view_active || goals_active || adopted) {
            uint32_t wb_bits = 0;
#pragma unroll
            for (int t = 0; t < NT; ++t) wb_bits |= (uint32_t)(tp_bounty(__float_as_uint(myval[S::V_T + 3 * t + 2])) > 0) << t;
            const int nwb = __popc(wb_bits);
            cov_now = (float)__popc(tracked_bits) / (float)NT;
            cov_real = nwb > 0 ? (float)__popc(wb_bits & tracked_bits) / (float)nwb : 0.f;
        }

        const bool last_pass = !step_goals;
        if (step_goals) {
            // ============================================================== finish step (environment.py:614-632)
            ep_reward += reward_i;
            delayed_ep_reward += delayed_i;
            episode_step += 1;
            coverage_sum += cov_now;
            done = !(episode_step <= p.max_episode_steps && cargo.any_awaiting());
            if (env_ok) {
                const int r_out = p.reward_sparse ? delayed_i : reward_i;
                reinterpret_cast<float2*>(p.rewards)[e] = make_float2(-(float)r_out, (float)r_out);
                p.done[e] = (uint8_t)done;
                if (done) {
                    atomicAdd(&p.stats[0], 1.0f);
                    atomicAdd(&p.stats[1], (float)ep_reward);
                    atomicAdd(&p.stats[2], (float)episode_step);
                    atomicAdd(&p.stats[3], (float)delivered);
                    atomicAdd(&p.stats[4], coverage_sum / (float)episode_step);
                }
            }
            auto_reset_needed = env_ok && done && (p.flags & MATE_STEP_AUTO_RESET);
            if (env_ok && !done && p.next != nullptr && (p.flags & MATE_STEP_AUTO_RESET) && episode_step == p.max_episode_steps)
                prefetch_prepared<NC, NT, NO, S>(*p.next, e + p.next_offset);   // the next step ends this episode (time limit)
        }
        // aux reflects the step just taken (before any auto-reset) / the observed or reset state
        if (p.has_aux && env_ok && (step_goals || mode != MODE_STEP)) {
            const float transport = delivered > 0 ? (float)((double)delayed_ep_reward / ((double)p.reward_scale * (double)delivered)) : 0.f;
            if (!p.has_aux_detail) {   // the common case: only the info-dict scalars (environment.py:634-639)
                if (p.aux.coverage) {
                    p.aux.coverage[(size_t)e * 3 + 0] = cov_now;
                    p.aux.coverage[(size_t)e * 3 + 1] = cov_real;
                    p.aux.coverage[(size_t)e * 3 + 2] = transport;
                }
                if (p.aux.num_delivered) p.aux.num_delivered[e] = delivered;
                if (p.aux.episode_step) p.aux.episode_step[e] = episode_step;
            } else {
                write_aux_env<NC, NT, NO, S>(p, e, mymk, myval, tdone_bits, cov_now, cov_real, transport, delivered, episode_step);
            }
        }
        if (last_pass || !__any_sync(FULL, auto_reset_needed)) break;
    }
    const int nvalid = min(tile_envs, p.num_envs - env0);
    if (mode == MODE_STEP && lane == 0) atomicAdd(&p.stats[5], (float)nvalid);

    // ------------------------------------------------------------------ write state back
    if (env_ok && mode != MODE_OBSERVE && (mode != MODE_PREPARE || need)) {
#pragma unroll
        for (int t = 0; t < NT; ++t) p.tgt_pack[(size_t)t * bp + e] = __float_as_uint(myval[S::V_T + 3 * t + 2]);
        if (cargo_dirty) {
            p.cargo[e] = make_uint4(cargo.rem[0], cargo.rem[1], cargo.rem[2], cargo.rem[3]);
            p.cargo[bp + e] = make_uint4(cargo.rem[4], cargo.rem[5], cargo.rem[6], cargo.rem[7]);
        }
        p.env_a[e] = make_uint4(cargo.aw[0], cargo.aw[1], (uint32_t)episode_step, (uint32_t)delivered);
        p.env_b[e] = make_int4(ep_reward, delayed_ep_reward, __float_as_int(coverage_sum), episode_id);
    }
    if (mode == MODE_PREPARE) {   // first-view masks of the prepared episode, then publish the tag
        if (need) {
#pragma unroll 1
            for (int w = 0; w < S::R * MW; ++w) p.masks[(size_t)w * bp + e] = mymk[w];
#pragma unroll 1
            for (int k = 0; k < S::VN; ++k) p.vals[(size_t)k * bp + e] = myval[k];
            __threadfence();
            st_release_u32(p.ready + e, (uint32_t)episode_id);
        }
        return;
    }
    __syncwarp();

    // ------------------------------------------------------------------ joint_observation (environment.py:908-983)
    TL_MARK(5);
    if (p.obs_format == MATE_OBS_FORMAT_F16) {
        if (p.obs_ops.n > 0) pack_observations<NC, NT, NO, true, __half>(p, env0, nvalid, stage, mk, val, reinterpret_cast<float*>(wbase + S::WARP_BYTES));
        else pack_observations<NC, NT, NO, false, __half>(p, env0, nvalid, stage, mk, val, nullptr);
    } else {
        if (p.obs_ops.n > 0) pack_observations<NC, NT, NO, true, float>(p, env0, nvalid, stage, mk, val, reinterpret_cast<float*>(wbase + S::WARP_BYTES));
        else pack_observations<NC, NT, NO, false, float>(p, env0, nvalid, stage, mk, val, nullptr);
    }
    TL_MARK(6);
}

}  // namespace mate
