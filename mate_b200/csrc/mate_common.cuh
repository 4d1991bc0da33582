// mate_common.cuh -- device helpers shared by the step kernels: constants, launch parameters, Philox,
// the cargo table, Obstacle.obstruct, the on-the-fly field-of-view polyline and the reset routine.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mate_b200.h"

namespace mate {

constexpr int NW = MATE_NUM_WAREHOUSES;
constexpr double kTerrain = 1000.0;          // mate/constants.py:52
constexpr double kWarehouseRadius = 75.0;    // mate/constants.py:67
constexpr double kWarehouseCoord = 925.0;    // mate/constants.py:70-72
constexpr double kRad2Deg = 57.295779513082320876798154814105;
constexpr double kDeg2Rad = 0.017453292519943295769236907684886;
constexpr int kResetRetries = 500;           // mate/environment.py:53

enum Mode : int { MODE_STEP = 0, MODE_OBSERVE = 1, MODE_RESET = 2, MODE_PREPARE = 3 };

enum Stream : uint32_t {
    STREAM_SHUFFLE_CAM = 0, STREAM_SHUFFLE_TGT = 1, STREAM_SHUFFLE_OBS = 2, STREAM_CAPACITY = 3,
    STREAM_PLACE = 4, STREAM_CARGO = 5, STREAM_INIT_GOAL = 6, STREAM_TRANSMIT = 7, STREAM_CHOICE = 8
};

// ---- packed per-target integer state (one u32 per target) -------------------------------
// bits 0-15 bounty | 16-18 goal+1 | 19-20 cargo weight | 21-22 capacity | 23-26 empty_bits | 27 colliding
__host__ __device__ inline uint32_t pack_target(int bounty, int goal, int weight, int capacity, int empty, int colliding) {
    return (uint32_t)(bounty & 0xFFFF) | ((uint32_t)(goal + 1) << 16) | ((uint32_t)(weight & 3) << 19) |
           ((uint32_t)(capacity & 3) << 21) | ((uint32_t)(empty & 15) << 23) | ((uint32_t)(colliding & 1) << 27);
}
__host__ __device__ inline int tp_bounty(uint32_t p) { return (int)(p & 0xFFFF); }
__host__ __device__ inline int tp_goal(uint32_t p) { return (int)((p >> 16) & 7) - 1; }
__host__ __device__ inline int tp_weight(uint32_t p) { return (int)((p >> 19) & 3); }
__host__ __device__ inline int tp_capacity(uint32_t p) { return (int)((p >> 21) & 3); }
__host__ __device__ inline int tp_empty(uint32_t p) { return (int)((p >> 23) & 15); }
__host__ __device__ inline int tp_colliding(uint32_t p) { return (int)((p >> 27) & 1); }

// ---- observation row layout (mate/constants.py:267-300), the reference's format ----------------
// A row is the preserved block, the observer's own (private) state, then one entry per entity: its public state and a
// visibility flag.  Camera rows list targets, obstacles, cameras; target rows list cameras, obstacles, targets.
// Kernels use it as `constexpr ObsLayout L{NC, NT, NO}` (every value a compile-time constant), the host with run-time counts.
enum EntityKind : int { KIND_TARGET = 0, KIND_OBSTACLE = 1, KIND_CAMERA = 2 };

struct ObsLayout {
    int nc, nt, no;
    // preserved block, the same in both teams' rows: counts (3), own index, warehouse locations (2 NW), warehouse radius
    static constexpr int PRESERVED = 3 + 1 + 2 * NW + 1;
    static constexpr int WAREHOUSE = 3 + 1;                   // first of the 2 NW warehouse coordinates (x, y per warehouse)
    // own state: location in columns SELF, SELF + 1; a target's ends with its NW empty bits
    static constexpr int SELF = PRESERVED;
    static constexpr int CAM_PRIVATE = 9, TGT_PRIVATE = 6 + 2 * NW;
    static constexpr int TGT_EMPTY = SELF + TGT_PRIVATE - NW;
    // one entry of an entity list: public state + flag
    static constexpr int TGT_ENTRY = 4 + 1, OBS_ENTRY = 3 + 1, CAM_ENTRY = 6 + 1;
    __host__ __device__ static constexpr int width(int kind) {
        return kind == KIND_TARGET ? TGT_ENTRY : (kind == KIND_OBSTACLE ? OBS_ENTRY : CAM_ENTRY);
    }
    __host__ __device__ constexpr int count(int kind) const { return kind == KIND_TARGET ? nt : (kind == KIND_OBSTACLE ? no : nc); }
    // first column of the entity list of `kind` in a camera / target row
    __host__ __device__ constexpr int block(bool cam_row, int kind) const {
        const int c_tgt = SELF + CAM_PRIVATE, c_obs = c_tgt + TGT_ENTRY * nt, c_cam = c_obs + OBS_ENTRY * no;
        const int t_cam = SELF + TGT_PRIVATE, t_obs = t_cam + CAM_ENTRY * nc, t_tgt = t_obs + OBS_ENTRY * no;
        return cam_row ? (kind == KIND_TARGET ? c_tgt : (kind == KIND_OBSTACLE ? c_obs : c_cam))
                       : (kind == KIND_CAMERA ? t_cam : (kind == KIND_OBSTACLE ? t_obs : t_tgt));
    }
    __host__ __device__ constexpr int entry_offset(bool cam_row, int kind, int index) const {
        return block(cam_row, kind) + width(kind) * index;
    }
    __host__ __device__ constexpr int dc() const { return block(true, KIND_CAMERA) + CAM_ENTRY * nc; }
    __host__ __device__ constexpr int dt() const { return block(false, KIND_TARGET) + TGT_ENTRY * nt; }
    // (scale, shift) columns of the packer's RescaledObservation (FoldOps): preserved | target own state | camera own
    // state | one target, obstacle and camera entry
    static constexpr int AFF_PRES = 0, AFF_TSELF = AFF_PRES + PRESERVED, AFF_CSELF = AFF_TSELF + TGT_PRIVATE;
    static constexpr int AFF_TGT = AFF_CSELF + CAM_PRIVATE, AFF_OBS = AFF_TGT + TGT_ENTRY, AFF_CAM = AFF_OBS + OBS_ENTRY;
    static constexpr int AFF_COLS = AFF_CAM + CAM_ENTRY;
};

// observation wrappers (mate_wrappers.cuh), innermost first
constexpr int kMaxObsOps = MATE_MAX_OBS_OPS;
struct ObsOps { int n; int op[kMaxObsOps]; };

// The reference's wrapper ordering rules (enhanced_observation.py:33-47, shared_field_of_view.py:35-49,
// relative_coordinates / rescaled_observation asserts) only admit stacks of the form
//   (EnhancedObservation | SharedFieldOfView)*  RelativeCoordinates?  RescaledObservation?
// For those the packer of the step kernel applies the wrappers while it composes the rows (mate_step.cuh, FOLD):
// mask ops act on the observer rows' mask words, RelativeCoordinates subtracts the observer's fp64 location from the
// visible entities' locations, RescaledObservation is one FMA per entry with (scale, shift) read from this block
// (kernel parameters live in the constant bank).
struct FoldOps {
    int fast;                           // the registered stack has the canonical form; 0 = generic shared-memory path
    int n_mask; int mask_op[kMaxObsOps];
    int relative, rescaled;
    float2 pres[ObsLayout::PRESERVED];  // (scale, shift) of the preserved block's columns (the same for both teams)
    float2 cself[ObsLayout::CAM_PRIVATE], tself[ObsLayout::TGT_PRIVATE];                        // private state of a camera / a target row
    float2 tgt[ObsLayout::TGT_ENTRY], obs[ObsLayout::OBS_ENTRY], cam[ObsLayout::CAM_ENTRY];     // a target / obstacle / camera entry with its flag
};

struct Params {
    // --- state (device, struct-of-arrays, row stride = bpad) ---
    double* cam_x; double* cam_y; double* cam_phi; double* cam_theta;   // [NC][bpad]
    double* tgt_x; double* tgt_y;                                       // [NT][bpad]
    double* obs_x; double* obs_y; double* obs_r;                        // [NO][bpad]
    float4* obs_f4;                                                     // [NO][bpad] fp32 shadow {x, y, r, 0} of the obstacles
    uint32_t* tgt_pack;                                                 // [NT][bpad]
    uint4* cargo;      // [2][bpad]  remaining_cargoes as 16 x u16
    uint4* env_a;      // [bpad] x: awaiting0|awaiting1<<16, y: awaiting2|awaiting3<<16, z: episode_step, w: delivered
    int4* env_b;       // [bpad] x: episode reward, y: delayed episode reward, z: coverage_sum (float bits), w: episode_id
    unsigned long long* cc_clear;   // [bpad] per-episode cache: bit 63 valid, bit (8 j + c) = camera c has a clear line of sight to camera j
    float* stats;      // [16] episode statistics accumulators
    // --- prepared next episodes (mate_step.cuh, "prepared resets"): a second state block holds, per env, the
    //     complete initial state of its NEXT episode; auto-reset adopts it instead of running the reset ---
    uint32_t* masks;          // [R * MW][bpad] observer mask words of the initial view (filled by MODE_PREPARE in the second block)
    float* vals;              // [3 NT + 5 NC][bpad] fp32 entity entries of the initial state (same, second block only)
    uint32_t* ready;          // [bpad] episode id the prepared state of an env is valid for (0 = none)
    const int4* live_env_b;   // MODE_PREPARE: env_b of the live state (current episode ids)
    const Params* next;       // MODE_STEP: device copy of the parameter block that addresses the second state block (nullptr = none)
    // --- per-call I/O (device) ---
    const float* cam_act; const float* tgt_act;
    float* cam_obs; float* tgt_obs; float* rewards; uint8_t* done;
    const uint8_t* env_mask;
    MateStepAux aux; int has_aux; int has_aux_detail;   // detail = anything beyond coverage / num_delivered / episode_step
    const uint8_t* replay_transmit; const int8_t* replay_choice;
    // observation wrappers applied to the rows before they leave the SM (mate_b200_set_observation_ops)
    ObsOps obs_ops; const float* cam_affine; const float* tgt_affine; FoldOps fold;
    int tile_envs;     // environments per warp tile of the step kernel: 32, 16 or 8 (MateSim::tile_envs)
    int warp_stride;   // bytes between the shared-memory blocks of two warps of a CTA (Shape2::WARP_BYTES, + scratch with obs_ops)
    unsigned long long l2_window_bytes;   // host side only: bytes of obs_f4 the launch asks the L2 to keep (0 = no window), mate_b200.cu
    // --- scalars ---
    int num_envs; int bpad; int mode; uint32_t flags;
    int next_offset;   // a launch over [begin, begin + num_envs) of the batch: env e of the launch is env e + next_offset of the arrays `next` addresses
    long long env_index_base; unsigned long long seed;
    int max_episode_steps; int num_cargoes_per_target; int num_high_capacity; int start_with_cargoes;
    int shuffle; int reward_sparse; int transmittance_is_one;
    int freight_scale; int bounty_scale; int reward_scale;
    double cam_radius, cam_min_view, cam_rmax, cam_rot_step, cam_zoom_step, cam_area_product;
    double tgt_step_size, tgt_sight_range, transmittance;
    double obs_r_low, obs_r_high;
    const double* cam_ranges; const double* tgt_ranges; const double* obs_ranges;  // device [N][4]
    int obs_format;    // element type of cam_obs / tgt_obs: MATE_OBS_FORMAT_F32 or _F16 (mate_b200_set_observation_format)
};

// ---- small math helpers --------------------------------------------------------------------
// mate/utils.py:155-158: (a + 180) % 360 - 180 with Python's float modulo.  Every angle the
// kernel normalises lies in (-540, 540), where fmod reduces to one exact add/subtract, so this
// produces the same bits as the reference expression.
__device__ __forceinline__ double normalize_angle(double a) {
    double x = a + 180.0;
    if (x < 0.0) x += 360.0;
    else if (x >= 360.0) x -= 360.0;
    return x - 180.0;
}
// sqrt(d2) <= t, decided on squares; the exact square root is only taken inside a 1e-12 band
__device__ __noinline__ bool dist_cmp_exact(double d2, double t, bool strict) {
    const double d = sqrt(d2);
    return strict ? d < t : d <= t;
}
// t2lo = t^2 (1 - 1e-12), t2hi = t^2 (1 + 1e-12)
__device__ __forceinline__ bool dist_le(double d2, double t, double t2lo, double t2hi) {
    if (d2 < t2lo) return true;
    if (d2 > t2hi) return false;
    return dist_cmp_exact(d2, t, false);
}
__device__ __forceinline__ bool dist_lt(double d2, double t, double t2lo, double t2hi) {
    if (d2 < t2lo) return true;
    if (d2 > t2hi) return false;
    return dist_cmp_exact(d2, t, true);
}
__device__ __forceinline__ double norm2(double x, double y) { return sqrt(x * x + y * y); }
__device__ __forceinline__ double atan2_deg(double y, double x) { return atan2(y, x) * kRad2Deg; }
__device__ __forceinline__ void sincos_deg(double deg, double* s, double* c) { sincos(deg * kDeg2Rad, s, c); }

// ---- Philox4x32-10, same draw scheme as oracle/mate_oracle.c ------------------------------
struct RngKey { unsigned long long seed; uint32_t env; uint32_t episode; };

// the rounds, for a second out-of-line copy (philox_comm, mate_agents.cuh): ptxas allocates registers across every caller
// of an out-of-line function, so new callers of `philox` would change the step kernel's code
__device__ __forceinline__ uint4 philox_rounds(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __noinline__ uint4 philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    return philox_rounds(c0, c1, c2, c3, k0, k1);
}
__device__ inline uint4 rng_words(const RngKey& k, uint32_t stream, uint32_t index) {
    return philox(index, stream, k.env, k.episode, (uint32_t)k.seed, (uint32_t)(k.seed >> 32));
}
__device__ inline double rng_u01(const RngKey& k, uint32_t stream, uint32_t index) {
    uint4 w = rng_words(k, stream, index);
    unsigned long long bits = ((unsigned long long)w.y << 32) | w.x;
    return (double)(bits >> 11) * (1.0 / 9007199254740992.0);
}
__device__ inline uint32_t rng_below(const RngKey& k, uint32_t stream, uint32_t index, uint32_t n) {
    return __umulhi(rng_words(k, stream, index).x, n);
}

// ---- per-env cargo table, replicated in every lane of the group ---------------------------
struct Cargo {
    uint32_t rem[8];   // remaining[w][g] as u16: word (w*4+g)/2, half (w*4+g)&1
    uint32_t aw[2];    // awaiting[4] as u16
    __device__ __forceinline__ int get(int w, int g) const {
        int i = w * 4 + g;
        uint32_t word = rem[0];
#pragma unroll
        for (int k = 1; k < 8; ++k) word = (i >> 1) == k ? rem[k] : word;
        return (int)((word >> ((i & 1) * 16)) & 0xFFFF);
    }
    __device__ __forceinline__ void add(int w, int g, int delta) {
        int i = w * 4 + g;
        uint32_t inc = (uint32_t)delta << ((i & 1) * 16);
#pragma unroll
        for (int k = 0; k < 8; ++k) if ((i >> 1) == k) rem[k] += inc;
    }
    __device__ __forceinline__ bool row_any(int w) const {
        uint32_t a = rem[0] | rem[1];
#pragma unroll
        for (int k = 1; k < 4; ++k) a = (w == k) ? (rem[2 * k] | rem[2 * k + 1]) : a;
        return a != 0;
    }
    __device__ __forceinline__ int awaiting(int g) const { return (int)((aw[g >> 1] >> ((g & 1) * 16)) & 0xFFFF); }
    __device__ __forceinline__ void awaiting_add(int g, int delta) {
        uint32_t inc = (uint32_t)delta << ((g & 1) * 16);
        if (g >> 1) aw[1] += inc; else aw[0] += inc;
    }
    __device__ __forceinline__ bool any_awaiting() const { return (aw[0] | aw[1]) != 0; }
};

// =============================================================================================
// Obstacle.obstruct(ray, keep_tangential=True) for target motion (mate/entities.py:158-184).
// (vx, vy) is the step vector with cached norm n (valid if has_n), origin (ox, oy); disc centre
// (px, py), radius R.
// =============================================================================================
struct StepVec { double vx, vy, n, ang, bound; bool has_n, has_ang; };   // bound >= |v| for the cheap reject

__device__ __noinline__ StepVec obstruct_exact(StepVec s, double ox, double oy, double px, double py, double R) {
    const double relx = px - ox, rely = py - oy;
    const double reln = norm2(relx, rely);
    if (!s.has_n) { s.n = norm2(s.vx, s.vy); s.has_n = true; }
    const double norm = s.n;
    if (norm == 0.0 || reln < R) {   // return -ray
        s.vx = -s.vx; s.vy = -s.vy; s.has_n = false; s.has_ang = false;
        return s;
    }
    if (reln >= norm + R) return s;
    const double inner = relx * s.vx + rely * s.vy;
    if (inner >= 0.0) {
        const double c = fmin(1.0, inner / (reln * norm));
        const double perp = reln * sqrt(1.0 - c * c);
        if (R > perp) {
            const double hc = sqrt(R * R - perp * perp);
            const double nn = fmax(0.0, reln * c - hc);
            if (nn < norm) {
                // unit vector of the step: the reference goes through (cos, sin) of atan2(v); v / |v| is the
                // same direction to 1 ulp (same class of deviation as the step-size clamp, DESIGN.md)
                const double inv = 1.0 / norm;
                const double cs = s.vx * inv, sn = s.vy * inv;
                const double radx = (ox + nn * cs) - px, rady = (oy + nn * sn) - py;
                const double k = (norm - nn) * hc / (R * R);
                s.vx = s.vx + radx * k; s.vy = s.vy + rady * k;
                s.has_n = false; s.has_ang = false;
                s.bound = fabs(s.vx) + fabs(s.vy);
            }
        }
    }
    return s;
}

// cheap conservative reject: with |v| <= bound, `relative.norm >= norm + radius` certainly holds
__device__ __forceinline__ void obstruct_step(StepVec& s, double ox, double oy, double px, double py, double R) {
    const double relx = px - ox, rely = py - oy;
    const double reach = s.bound + R;
    if (relx * relx + rely * rely > reach * reach * (1.0 + 1e-9)) return;
    s = obstruct_exact(s, ox, oy, px, py, R);
}

// =============================================================================================
// On-the-fly field-of-view range: value of the reference's sampled (phi, rho) polyline
// (Camera.add_obstacles + interp1d, mate/entities.py:362-479, 507-511) at bearing `a`
// (degrees, already normalised to [-180, 180)), WITHOUT materialising the polyline.
// The polyline's sample angles are: the 360 integer degrees; per visible obstacle the four
// edge rays L-+0.01, R-+0.01 and the lattice linspace(L, R, n+1).  We find the two samples
// that bracket `a`, cast those two rays against all obstacle discs (sequential shortening ==
// min over discs) and interpolate linearly like np.interp.
// =============================================================================================
struct RaySample { double angle; double n0; int tangent_of; };
// fp64 obstacle discs of one environment: element o of field f is f[o * stride]
struct ObsRef { const double* x; const double* y; const double* r; size_t stride; };

// `discs`: the discs that can meet the ray (a superset is fine: a disc the ray misses changes nothing)
template <int NO>
__device__ __forceinline__ double cast_ray(const ObsRef ob, double cx, double cy,
                                           double angle, double n0, int tangent_of, unsigned long long discs) {
    double sn, cs;
    sincospi(angle * (1.0 / 180.0), &sn, &cs);
    double n = n0;
    while (discs != 0ull) {
        const int o = __ffsll((long long)discs) - 1;
        discs &= discs - 1ull;
        if (o == tangent_of) continue;   // exact tangent ray: never shortened by its own disc (DESIGN.md)
        const double relx = ob.x[o * ob.stride] - cx, rely = ob.y[o * ob.stride] - cy, R = ob.r[o * ob.stride];
        const double proj = relx * cs + rely * sn;
        if (proj < 0.0) continue;
        const double d2 = relx * relx + rely * rely;
        const double perp2 = d2 - proj * proj;
        if (!(R * R > perp2)) continue;
        const double hc = sqrt(R * R - fmax(perp2, 0.0));
        const double nn = fmax(0.0, proj - hc);
        if (nn < n) n = nn;
    }
    return n;
}

__device__ __forceinline__ void consider(RaySample& P, RaySample& S, double a, double s, double n0, int tangent_of) {
    if (s <= a) {
        if (s > P.angle || (s == P.angle && n0 < P.n0)) { P.angle = s; P.n0 = n0; P.tangent_of = tangent_of; }
    } else {
        if (s < S.angle || (s == S.angle && n0 < S.n0)) { S.angle = s; S.n0 = n0; S.tangent_of = tangent_of; }
    }
}

template <int NO>
__device__ __noinline__ double sight_range_at(const ObsRef ob, double cx, double cy,
                                              double rmax, double a, double ux, double uy) {
    // (ux, uy): unit vector of bearing a (rel / dist), used only for the conservative prefilter
    const double fl = floor(a);
    RaySample P{fl, rmax, -1}, S{fl + 1.0, rmax, -1};
    const double c1 = 0.99984154; // cos(1.02 deg)
    const double s1 = 0.01780139; // sin(1.02 deg)
    // phase 1: which obstacles of the camera's set can have a sample angle inside (floor(a), floor(a) + 1)?
    unsigned long long passing = 0ull;
    bool inside = false;
#pragma unroll 1
    for (int o = 0; o < NO; ++o) {
        const double relx = ob.x[o * ob.stride] - cx, rely = ob.y[o * ob.stride] - cy, R = ob.r[o * ob.stride];
        const double d2 = relx * relx + rely * rely;
        {   // entities.py:365 (strict <) and :378 (camera inside the disc), on squares
            const double reach = rmax + R, reach2 = reach * reach;
            if (d2 > reach2 * (1.0 + 1e-12)) continue;
            if (d2 > reach2 * (1.0 - 1e-12) && !dist_cmp_exact(d2, reach, true)) continue;
            if (d2 < R * R * (1.0 + 1e-12) && dist_cmp_exact(d2, R, true)) { inside = true; continue; }
        }
        // angular distance bearing<->centre must be <= half + 1.02 deg
        const double p = relx * ux + rely * uy + R * s1 * 1.0000001;
        if (p < 0.0) continue;
        if (p * p < (d2 - R * R) * (c1 * c1) * 0.9999999) continue;
        passing |= 1ull << o;
    }
    if (inside) return 0.0;
    // Both bracketing samples lie within 1 degree of the bearing, so a disc that cuts one of those two rays
    // is at an angular distance <= half + 1 degree from the bearing: it is in `passing` (discs outside the
    // camera's obstacle set are farther than rmax + R and cannot shorten a ray of length <= rmax).
    const unsigned long long near_discs = passing;
    // phase 2: the sample angles of those obstacles, one obstacle per iteration (lanes of a warp that
    // evaluate different obstacles stay converged)
    while (passing != 0ull) {
        const int o = __ffsll((long long)passing) - 1;
        passing &= passing - 1ull;
        const double relx = ob.x[o * ob.stride] - cx, rely = ob.y[o * ob.stride] - cy, R = ob.r[o * ob.stride];
        const double d2 = relx * relx + rely * rely;
        const double d = sqrt(d2);
        const double ang_o = atan2_deg(rely, relx);
        const double half = asin(R / d) * kRad2Deg;
        const double left = ang_o - half, right = ang_o + half;
        consider(P, S, a, normalize_angle(left - 0.01), rmax, -1);
        consider(P, S, a, normalize_angle(left + 0.01), rmax, -1);
        consider(P, S, a, normalize_angle(right - 0.01), rmax, -1);
        consider(P, S, a, normalize_angle(right + 0.01), rmax, -1);
        const int two_half = (int)(2.0 * half);
        const int nlat = two_half > 16 ? two_half : 16;
        const double step = (right - left) / (double)nlat;   // np.linspace: arange(num) * step + start
        const double max_rho = fmin(rmax, d + R);
        if (step > 0.0) {
#pragma unroll 1
            for (int k = -1; k <= 1; ++k) {
                const double ap = a + 360.0 * (double)k;
                if (ap < left - step || ap > right + step) continue;
                const int i0 = (int)floor((ap - left) / step);
#pragma unroll 1
                for (int i = i0 - 1; i <= i0 + 2; ++i) {
                    if (i < 0 || i > nlat) continue;
                    const double raw = (i == nlat) ? right : ((double)i * step + left);
                    consider(P, S, a, normalize_angle(raw), max_rho, (i == 0 || i == nlat) ? o : -1);
                }
            }
        }
    }
    const double rho_p = cast_ray<NO>(ob, cx, cy, P.angle, P.n0, P.tangent_of, near_discs);
    if (a == P.angle) return rho_p;                // np.interp: exact hit on a sample
    // the closing sample (phi0 + 360, rho0) of the polyline is the -180 grid ray (entities.py:470-471)
    const double s_angle = (S.angle >= 180.0) ? -180.0 : S.angle;
    const double rho_s = cast_ray<NO>(ob, cx, cy, s_angle, S.n0, S.tangent_of, near_discs);
    const double slope = (rho_s - rho_p) / (S.angle - P.angle);
    return slope * (a - P.angle) + rho_p;
}

// The same evaluation by a QUAD of lanes (lanes 4k .. 4k+3 of a warp work on one query; all 32 lanes must call
// this together).  Lane q of the quad owns the discs o = q, q + 4, q + 8, ... in registers: the disc loops are a
// quarter as long, the candidate samples P / S and the two ray casts are reduced over the quad with shuffles
// (lexicographic max / min, exactly the order `consider` imposes; minimum over the cut lengths).  Arithmetic per
// disc is the scalar routine's, so the result is the same.
template <int NO>
__device__ __forceinline__ double sight_range_quad(const ObsRef ob, double cx, double cy, double rmax, double a,
                                                   double ux, double uy, const int q) {
    constexpr uint32_t FULL = 0xffffffffu;
    constexpr int SL = (NO + 3) / 4 > 0 ? (NO + 3) / 4 : 1;
    double X[SL], Y[SL], R[SL];
#pragma unroll
    for (int s = 0; s < SL; ++s) {
        const int o = q + 4 * s;
        const bool has = o < NO;
        X[s] = has ? ob.x[o * ob.stride] - cx : 0.0; Y[s] = has ? ob.y[o * ob.stride] - cy : 0.0; R[s] = has ? ob.r[o * ob.stride] : -1.0;
    }
    const double fl = floor(a);
    RaySample P{fl, rmax, -1}, S{fl + 1.0, rmax, -1};
    const double c1 = 0.99984154; // cos(1.02 deg)
    const double s1 = 0.01780139; // sin(1.02 deg)
    uint32_t mine = 0;            // bit s: my disc of slot s can have a sample angle inside (floor(a), floor(a) + 1)
    bool inside = false;
#pragma unroll
    for (int s = 0; s < SL; ++s) {
        const double relx = X[s], rely = Y[s], Rr = R[s];
        if (Rr < 0.0) continue;
        const double d2 = relx * relx + rely * rely;
        {
            const double reach = rmax + Rr, reach2 = reach * reach;
            if (d2 > reach2 * (1.0 + 1e-12)) continue;
            if (d2 > reach2 * (1.0 - 1e-12) && !dist_cmp_exact(d2, reach, true)) continue;
            if (d2 < Rr * Rr * (1.0 + 1e-12) && dist_cmp_exact(d2, Rr, true)) { inside = true; continue; }
        }
        const double pp = relx * ux + rely * uy + Rr * s1 * 1.0000001;
        if (pp < 0.0) continue;
        if (pp * pp < (d2 - Rr * Rr) * (c1 * c1) * 0.9999999) continue;
        mine |= 1u << s;
    }
    {
        uint32_t any_inside = inside ? 1u : 0u;
        any_inside |= __shfl_xor_sync(FULL, any_inside, 1);
        any_inside |= __shfl_xor_sync(FULL, any_inside, 2);
        inside = any_inside != 0u;
    }
    // sample angles of my passing discs (compacted: the warp iterates max-popcount times, not once per slot)
    uint32_t todo = mine;
#pragma unroll 1
    while (todo != 0u) {
        const int s = __ffs(todo) - 1;
        todo &= todo - 1u;
        double relx = X[0], rely = Y[0], Rr = R[0];
#pragma unroll
        for (int k = 1; k < SL; ++k) { relx = s == k ? X[k] : relx; rely = s == k ? Y[k] : rely; Rr = s == k ? R[k] : Rr; }
        const int o = q + 4 * s;
        const double d2 = relx * relx + rely * rely;
        const double d = sqrt(d2);
        const double ang_o = atan2_deg(rely, relx);
        const double half = asin(Rr / d) * kRad2Deg;
        const double left = ang_o - half, right = ang_o + half;
        consider(P, S, a, normalize_angle(left - 0.01), rmax, -1);
        consider(P, S, a, normalize_angle(left + 0.01), rmax, -1);
        consider(P, S, a, normalize_angle(right - 0.01), rmax, -1);
        consider(P, S, a, normalize_angle(right + 0.01), rmax, -1);
        const int two_half = (int)(2.0 * half);
        const int nlat = two_half > 16 ? two_half : 16;
        const double step = (right - left) / (double)nlat;
        const double max_rho = fmin(rmax, d + Rr);
        if (step > 0.0) {
#pragma unroll 1
            for (int k = -1; k <= 1; ++k) {
                const double ap = a + 360.0 * (double)k;
                if (ap < left - step || ap > right + step) continue;
                const int i0 = (int)floor((ap - left) / step);
#pragma unroll 1
                for (int i = i0 - 1; i <= i0 + 2; ++i) {
                    if (i < 0 || i > nlat) continue;
                    const double raw = (i == nlat) ? right : ((double)i * step + left);
                    consider(P, S, a, normalize_angle(raw), max_rho, (i == 0 || i == nlat) ? o : -1);
                }
            }
        }
    }
    // the quad's best samples: P = latest angle <= a (ties: smaller range), S = earliest angle > a (ties: smaller range)
#pragma unroll
    for (int sh = 1; sh <= 2; sh <<= 1) {
        const double pa = __shfl_xor_sync(FULL, P.angle, sh), pn = __shfl_xor_sync(FULL, P.n0, sh);
        const int pt = __shfl_xor_sync(FULL, P.tangent_of, sh);
        if (pa > P.angle || (pa == P.angle && pn < P.n0)) { P.angle = pa; P.n0 = pn; P.tangent_of = pt; }
        const double sa = __shfl_xor_sync(FULL, S.angle, sh), sn = __shfl_xor_sync(FULL, S.n0, sh);
        const int st = __shfl_xor_sync(FULL, S.tangent_of, sh);
        if (sa < S.angle || (sa == S.angle && sn < S.n0)) { S.angle = sa; S.n0 = sn; S.tangent_of = st; }
    }
    // both bracketing rays against my discs near the bearing, minimum over the quad
    const double s_angle = (S.angle >= 180.0) ? -180.0 : S.angle;
    double sn_p, cs_p, sn_s, cs_s;
    sincospi(P.angle * (1.0 / 180.0), &sn_p, &cs_p);
    sincospi(s_angle * (1.0 / 180.0), &sn_s, &cs_s);
    double rho_p = P.n0, rho_s = S.n0;
#pragma unroll
    for (int s = 0; s < SL; ++s) {
        if (!((mine >> s) & 1u)) continue;
        const int o = q + 4 * s;
        const double relx = X[s], rely = Y[s], Rr = R[s];
        const double d2 = relx * relx + rely * rely;
        if (o != P.tangent_of) {
            const double proj = relx * cs_p + rely * sn_p;
            const double perp2 = d2 - proj * proj;
            if (proj >= 0.0 && Rr * Rr > perp2) rho_p = fmin(rho_p, fmax(0.0, proj - sqrt(Rr * Rr - fmax(perp2, 0.0))));
        }
        if (o != S.tangent_of) {
            const double proj = relx * cs_s + rely * sn_s;
            const double perp2 = d2 - proj * proj;
            if (proj >= 0.0 && Rr * Rr > perp2) rho_s = fmin(rho_s, fmax(0.0, proj - sqrt(Rr * Rr - fmax(perp2, 0.0))));
        }
    }
#pragma unroll
    for (int sh = 1; sh <= 2; sh <<= 1) {
        rho_p = fmin(rho_p, __shfl_xor_sync(FULL, rho_p, sh));
        rho_s = fmin(rho_s, __shfl_xor_sync(FULL, rho_s, sh));
    }
    if (inside) return 0.0;
    if (a == P.angle) return rho_p;
    const double slope = (rho_s - rho_p) / (S.angle - P.angle);
    return slope * (a - P.angle) + rho_p;
}

// Camera.perceive (mate/entities.py:491-505) up to the stochastic draw, exact arithmetic of
// the reference: returns 0 = not in range/sector, 1 = reached the draw.  The test itself is inline for callers
// outside the step (the renderer): ptxas allocates registers across every caller of an out-of-line function, so
// a new caller of `fov_reach_exact` would change the step kernel's code.  The distance is rounded like the C oracle
// (oracle/mate_oracle.c, built with -ffp-contract=off) rounds it, without contracting the sum of squares into an FMA: a
// target exactly on the arc of the sight range is one unit in the last place outside or inside depending on that
// rounding.  (The Python reference's np.linalg.norm goes through a BLAS dot product, whose rounding is its own.)
__device__ __forceinline__ int fov_reach_test(double cx, double cy, double phi, double theta, double rs,
                                              double qx, double qy) {
    const double relx = qx - cx, rely = qy - cy;
    const double dist = sqrt(__dadd_rn(__dmul_rn(relx, relx), __dmul_rn(rely, rely)));
    if (dist > rs) return 0;
    const double ang = atan2_deg(rely, relx);
    double ra = fabs(phi - ang);
    ra = fmin(ra, 360.0 - ra);
    if (ra * 2.0 > theta) return 0;
    return 1;
}
__device__ __noinline__ int fov_reach_exact(double cx, double cy, double phi, double theta, double rs,
                                            double qx, double qy) {
    return fov_reach_test(cx, cy, phi, theta, rs, qx, qy);
}

// Conservative occlusion classification of the query point q = cam + rel against all obstacle
// discs, WITHOUT evaluating the sampled polyline.  Both polyline samples that bracket the query
// bearing lie inside a fan of +-1.05 degrees around it (integer-degree grid).  Per disc, with
// `perp` the distance of its centre from the line of sight and `w` the half-width of the fan at
// the farthest range where it can meet the disc, every ray of the fan passes the centre at a
// lateral offset in [pmin, pmax] = [perp - w, perp + w], and a ray with offset p < R is cut at
// range rho(p) = sqrt(d_o^2 - p^2) - sqrt(R^2 - p^2), which grows with p.  Hence
//   * perp - w > R, disc behind the camera or entirely beyond the target: the disc is irrelevant;
//   * pmax < R and |rel| > rho(pmax): every fan ray is cut short of the target  -> occluded (0);
//   * |rel| < rho(pmin): no fan ray is cut before the target                    -> irrelevant;
//   * otherwise (silhouette edge inside the fan, or target at the disc's front surface): exact.
// Returns 1 = certainly visible, 0 = certainly occluded, 2 = evaluate the polyline exactly.
// All margins (>= 0.05 units, 0.04 degrees) are far above fp32 rounding (<= 1e-3 units here), so
// the classification runs in fp32 on the shadow entries Fobs[o * fstride] = {x, y, r, -}.
template <int NO>
__device__ __forceinline__ int occlusion_fast(const float4* __restrict__ Fobs, size_t fstride, float cx, float cy,
                                              float relx, float rely, float rmax) {
    const float d2 = relx * relx + rely * rely;
    const float inv_dist = rsqrtf(d2);
    const float dist = d2 * inv_dist;
    const float ux = relx * inv_dist, uy = rely * inv_dist;    // unit bearing
    const float tan_fan = 0.018332f;                           // tan(1.05 deg)
    const float d_hi = dist * (1.0f + 1e-4f) + 0.05f, d_lo = dist * (1.0f - 1e-4f) - 0.05f;
    bool all_clear = true;
    float4 nxt = Fobs[0];
#pragma unroll 1
    for (int o = 0; o < NO; ++o) {
        const float4 ob = nxt;
        if (o + 1 < NO) nxt = Fobs[(o + 1) * fstride];        // fetched while this disc is classified
        const float ox = ob.x - cx, oy = ob.y - cy, R = ob.z;
        const float do2 = ox * ox + oy * oy;
        const float reach = rmax + R + 0.05f;
        if (do2 > reach * reach) continue;                     // certainly not in the camera's obstacle set (entities.py:365)
        const float proj = ox * ux + oy * uy;                  // along the line of sight
        if (proj + R < 0.0f || proj - R > d_hi) continue;      // behind the camera / beyond the target
        const float perp = fabsf(ox * uy - oy * ux);           // distance of the centre from the line of sight
        const float w = tan_fan * fminf(d_hi, proj + R) + 0.05f;
        const float pmin = fmaxf(perp - w, 0.0f), pmax = perp + w;
        if (pmin >= R) continue;                               // the fan passes beside the disc
        const float inner = rmax + R - 0.05f;
        const bool in_set = do2 < inner * inner;               // certainly in the camera's obstacle set
        const float R2 = R * R;
        if (pmax < R * 0.9999f && in_set && do2 > R2 + 1.0f) {
            const float rho_max = sqrtf(do2 - pmax * pmax) - sqrtf(R2 - pmax * pmax);
            if (d_lo > rho_max * 1.0001f) return 0;            // every ray of the fan is cut before the target
        }
        const float rho_min = sqrtf(fmaxf(do2 - pmin * pmin, 0.0f)) - sqrtf(R2 - pmin * pmin);
        if (d_hi < rho_min * 0.9999f) continue;                // the target is in front of the disc
        all_clear = false;
    }
    return all_clear ? 1 : 2;
}

// Camera.perceive after the draw (entities.py:505): dist <= sight_range_at(angle) * (1 + 1e-6)
template <int NO>
__device__ __noinline__ bool occlusion_exact(const ObsRef ob, double cx, double cy,
                                             double relx, double rely, double dist, double rmax) {
    const double ang = atan2_deg(rely, relx);
    const double range = sight_range_at<NO>(ob, cx, cy, rmax, normalize_angle(ang), relx / dist, rely / dist);
    return dist <= range * (1.0 + 1e-6);
}

// =============================================================================================
// Rare paths, kept out of line so that the hot path stays inside the instruction cache
// =============================================================================================

struct ResetCfg {
    double cam_radius, cam_min_view, cam_rot_step, cam_area_product, tgt_step_size, obs_r_low, obs_r_high;
    const double* cam_ranges; const double* tgt_ranges; const double* obs_ranges;
    int shuffle, num_high_capacity, num_cargoes_per_target;
};

// MultiAgentTracking.reset (mate/environment.py:679-775) for one environment, executed by ONE
// lane: entity shuffle, capacities, rejection placement (cameras, obstacles, targets) and the
// cargo table, on the counter-based Philox streams.  Results go to the shared-memory entity
// block and to the 16-word scratch: [0..7] remaining cargoes (u16 pairs), [8..9] awaiting
// (u16 pairs), [10] capacity-2 bit set.
template <int NC, int NT, int NO, int CF>
__device__ __noinline__ void env_reset(ResetCfg cfg, RngKey key, double* Ecam, double* Etgt, double* Eobs,
                                       uint32_t* scr) {
    int perm_c[NC > 0 ? NC : 1], perm_t[NT], perm_o[NO > 0 ? NO : 1];
    for (int i = 0; i < NC; ++i) perm_c[i] = i;
    for (int i = 0; i < NT; ++i) perm_t[i] = i;
    for (int i = 0; i < NO; ++i) perm_o[i] = i;
    if (cfg.shuffle) {   // environment.py:707-710 (Fisher-Yates from the top, like RandomState.shuffle)
        for (int i = NC - 1; i >= 1; --i) { int k = (int)rng_below(key, STREAM_SHUFFLE_CAM, i, i + 1); int t = perm_c[i]; perm_c[i] = perm_c[k]; perm_c[k] = t; }
        for (int i = NT - 1; i >= 1; --i) { int k = (int)rng_below(key, STREAM_SHUFFLE_TGT, i, i + 1); int t = perm_t[i]; perm_t[i] = perm_t[k]; perm_t[k] = t; }
        for (int i = NO - 1; i >= 1; --i) { int k = (int)rng_below(key, STREAM_SHUFFLE_OBS, i, i + 1); int t = perm_o[i]; perm_o[i] = perm_o[k]; perm_o[k] = t; }
    }
    uint32_t cap2 = 0;   // bit t set => capacity 2 (environment.py:712-722)
    if (cfg.num_high_capacity > 0) {
        if (cfg.shuffle) {
            int idx[NT];
            for (int i = 0; i < NT; ++i) idx[i] = i;
            for (int i = 0; i < cfg.num_high_capacity; ++i) {
                int k = i + (int)rng_below(key, STREAM_CAPACITY, i, NT - i);
                int t = idx[i]; idx[i] = idx[k]; idx[k] = t;
                cap2 |= 1u << idx[i];
            }
        } else {
            for (int i = 0; i < cfg.num_high_capacity; ++i) cap2 |= 1u << i;
        }
    }
    // rejection placement (environment.py:724-737): cameras, obstacles, targets
    int serial = 0;
    for (int kind = 0; kind < 3; ++kind) {
        const int count = kind == 0 ? NC : (kind == 1 ? NO : NT);
        for (int i = 0; i < count; ++i, ++serial) {
            const double* range = kind == 0 ? cfg.cam_ranges + 4 * perm_c[i]
                                : (kind == 1 ? cfg.obs_ranges + 4 * perm_o[i] : cfg.tgt_ranges + 4 * perm_t[i]);
            const double r0 = range[0], r1 = range[1], r2 = range[2], r3 = range[3];
            const double min_distance = kind == 2 ? 0.0 : cfg.tgt_step_size;
            double x = 0, y = 0, radius = kind == 0 ? cfg.cam_radius : 0.0, phi = 0, theta = 0, rs = 0;
            bool ok = false;
            for (int attempt = 0; attempt < kResetRetries && !ok; ++attempt) {
                const uint32_t base = ((uint32_t)serial * kResetRetries + (uint32_t)attempt) * 8u;
                if (kind == 1)   // Obstacle.reset: radius first (entities.py:150-152)
                    radius = __dadd_rn(cfg.obs_r_low, __dmul_rn(cfg.obs_r_high - cfg.obs_r_low, rng_u01(key, STREAM_PLACE, base + 2)));
                x = __dadd_rn(r0, __dmul_rn(r1 - r0, rng_u01(key, STREAM_PLACE, base + 0)));   // Entity.reset (entities.py:60-65)
                y = __dadd_rn(r2, __dmul_rn(r3 - r2, rng_u01(key, STREAM_PLACE, base + 1)));
                const double lim = __dsub_rn(kTerrain, __dmul_rn(1.2, radius));
                x = fmin(fmax(x, -lim), lim);
                y = fmin(fmax(y, -lim), lim);
                if (kind == 0) {   // Camera.reset (entities.py:326-334)
                    const uint32_t nrot = (uint32_t)(360.0 / cfg.cam_rot_step);
                    phi = normalize_angle(__dmul_rn(cfg.cam_rot_step, (double)rng_below(key, STREAM_PLACE, base + 3, nrot)));
                    theta = __dadd_rn(cfg.cam_min_view, __dmul_rn(180.0 - cfg.cam_min_view, rng_u01(key, STREAM_PLACE, base + 4)));
                    rs = sqrt(cfg.cam_area_product / theta);
                }
                ok = true;
                for (int w = 0; w < NW && ok; ++w) {   // warehouse discs, radius 0.75 * 75 (environment.py:724-727)
                    const double wx = (w == 0 || w == 3) ? kWarehouseCoord : -kWarehouseCoord;
                    const double wy = (w < 2) ? kWarehouseCoord : -kWarehouseCoord;
                    const double dx = x - wx, dy = y - wy;
                    const double dist = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
                    if (__dmul_rn(dist, 1.0 + 1e-6) < __dadd_rn(__dadd_rn(radius, 0.75 * kWarehouseRadius), min_distance)) ok = false;
                }
                const int ncam_placed = kind == 0 ? i : NC;
                for (int q = 0; q < ncam_placed && ok; ++q) {
                    const double dx = x - Ecam[q * CF], dy = y - Ecam[q * CF + 1];
                    const double dist = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
                    if (__dmul_rn(dist, 1.0 + 1e-6) < __dadd_rn(__dadd_rn(radius, cfg.cam_radius), min_distance)) ok = false;
                    else if (kind == 0 && dist < __dmul_rn(0.1, fmin(rs, Ecam[q * CF + 4]))) ok = false;   // Camera.overlap (entities.py:484-489)
                }
                const int nobs_placed = kind == 0 ? 0 : (kind == 1 ? i : NO);
                for (int q = 0; q < nobs_placed && ok; ++q) {
                    const double dx = x - Eobs[3 * q], dy = y - Eobs[3 * q + 1];
                    const double dist = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
                    if (__dmul_rn(dist, 1.0 + 1e-6) < __dadd_rn(__dadd_rn(radius, Eobs[3 * q + 2]), min_distance)) ok = false;
                }
                // already placed targets have radius 0 and targets use min_distance 0:
                // dist * (1 + 1e-6) < 0 never holds (entities.py:96-100)
            }
            if (!ok && kind == 1) radius = 0.0;   // environment.py:734-736
            if (kind == 0) { Ecam[i * CF] = x; Ecam[i * CF + 1] = y; Ecam[i * CF + 2] = phi; Ecam[i * CF + 3] = theta; Ecam[i * CF + 4] = rs; }
            else if (kind == 1) { Eobs[3 * i] = x; Eobs[3 * i + 1] = y; Eobs[3 * i + 2] = radius; }
            else { Etgt[2 * i] = x; Etgt[2 * i + 1] = y; }
        }
    }
    // cargo table (environment.py:768-775)
    Cargo cargo;
    for (int k = 0; k < 8; ++k) cargo.rem[k] = 0;
    uint32_t draw = 0;
    for (;;) {
        bool all_rows = true;
        for (int w = 0; w < NW; ++w) all_rows = all_rows && cargo.row_any(w);
        if (all_rows) break;
        for (int i = 0; i < cfg.num_cargoes_per_target * NT; ++i, ++draw) {
            const uint4 w4 = rng_words(key, STREAM_CARGO, draw);
            const int sender = (int)__umulhi(w4.x, NW);
            int recipient = (int)__umulhi(w4.y, NW - 1);
            if (recipient >= sender) recipient += 1;   // choice(4, size=2, replace=False)
            cargo.add(sender, recipient, 1);
        }
    }
    cargo.aw[0] = cargo.aw[1] = 0;
    for (int gg = 0; gg < NW; ++gg) { int sum = 0; for (int w = 0; w < NW; ++w) sum += cargo.get(w, gg); cargo.awaiting_add(gg, sum); }
    for (int k = 0; k < 8; ++k) scr[k] = cargo.rem[k];
    scr[8] = cargo.aw[0]; scr[9] = cargo.aw[1]; scr[10] = cap2;
}

}  // namespace mate
