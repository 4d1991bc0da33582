// mate_render.cuh -- rgb_array frames of chosen environments (mate_b200_render, DESIGN.md section 7k), drawn from the
// live state on the device.  The picture is defined in include/mate_b200.h (MATE_RENDER_*); this file only shades it.
//
// One CTA per (frame, tile of kRenderRows x kRenderCols pixels); each thread shades 4 consecutive pixels of one row and
// stores them as three 32-bit words, so a warp writes 384 contiguous bytes of a row.  The CTA stages its environment's
// entities in shared memory and keeps, per tile, only the cameras whose sight circle can reach the tile and the
// obstacles, cameras and targets whose discs can touch it.  The field of view is decided by the step's own routines:
// fov_reach32 with its guard band, the fp64 test of fov_reach_exact inside the band, then occlusion_fast and occlusion_exact (the
// polyline of sight_range_at).  Every other test is fp64 without contraction (__dmul_rn / __dadd_rn), so a NumPy
// float64 restatement reproduces the frame bit for bit.
#pragma once

#include "mate_step.cuh"

namespace mate {

constexpr int kRenderRows = 8, kRenderCols = 128;           // pixels of a tile
constexpr int kRenderThreads = kRenderRows * kRenderCols / 4;

// pixel centres: one exact product and one correctly rounded division
__device__ __forceinline__ double render_x(int j, int size) { return __ddiv_rn(__dmul_rn((double)(2 * j + 1 - size), MATE_RENDER_HALF_EXTENT), (double)size); }
__device__ __forceinline__ double render_y(int i, int size) { return __ddiv_rn(__dmul_rn((double)(size - 2 * i - 1), MATE_RENDER_HALF_EXTENT), (double)size); }
__device__ __forceinline__ double render_d2(double dx, double dy) { return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)); }
// squared distance of (x, y) from the box [xlo, xhi] x [ylo, yhi] (culling only)
__device__ __forceinline__ double box_d2(double x, double y, double xlo, double xhi, double ylo, double yhi) {
    const double dx = fmax(fmax(xlo - x, x - xhi), 0.0), dy = fmax(fmax(ylo - y, y - yhi), 0.0);
    return dx * dx + dy * dy;
}
__device__ __forceinline__ uint32_t render_blend(uint32_t dst, uint32_t src) {
    constexpr uint32_t A = MATE_RENDER_FOV_ALPHA;
    uint32_t out = 0;
#pragma unroll
    for (int s = 0; s < 24; s += 8) out |= ((((dst >> s) & 0xFFu) * (255u - A) + ((src >> s) & 0xFFu) * A + 127u) / 255u) << s;
    return out;
}

template <int NC, int NT, int NO>
struct RenderEnv {
    static constexpr int C = NC > 0 ? NC : 1, T = NT > 0 ? NT : 1, O = NO > 0 ? NO : 1;
    double cx[C], cy[C], phi[C], theta[C], rs[C];
    double tx[T], ty[T];
    double ox[O], oy[O], orad[O];
    float4 of4[O];
    float fcx[C], fcy[C], rs2[C], hx[C], hy[C], ch2[C];
    uint32_t tpack[T];
    uint32_t fov_cams, draw_obs, draw_cams, draw_tgts, tracked;
};

// Camera.perceive of a target at (qx, qy) with a transmission draw of 0: the step's range + sector test, then its occlusion
// test unless the obstacles cannot occlude (none, or transmittance 1)
template <int NC, int NT, int NO>
__device__ __forceinline__ bool render_sees(const Params& p, const RenderEnv<NC, NT, NO>& s, int c, double qx, double qy) {
    const float fqx = (float)qx, fqy = (float)qy;
    const int reach = fov_reach32(s.fcx[c], s.fcy[c], s.rs2[c], s.hx[c], s.hy[c], s.ch2[c], fqx, fqy);
    if (reach == 0) return false;
    if (reach == 2 && !fov_reach_test(s.cx[c], s.cy[c], s.phi[c], s.theta[c], s.rs[c], qx, qy)) return false;
    if (NO == 0 || p.transmittance_is_one) return true;
    const int fast = occlusion_fast<NO>(s.of4, 1, s.fcx[c], s.fcy[c], fqx - s.fcx[c], fqy - s.fcy[c], (float)p.cam_rmax);
    if (fast != 2) return fast == 1;
    const double relx = qx - s.cx[c], rely = qy - s.cy[c];
    return occlusion_exact<NO>(ObsRef{s.ox, s.oy, s.orad, 1}, s.cx[c], s.cy[c], relx, rely, sqrt(relx * relx + rely * rely), p.cam_rmax);
}

// env[f] is the environment of frame f (nullptr: frame f is environment f); an entry outside [0, num_envs) is skipped
template <int NC, int NT, int NO>
__global__ void __launch_bounds__(kRenderThreads)
render_kernel(const Params p, const int32_t* __restrict__ env, int count, int size, int words, uint8_t* __restrict__ out) {
    __shared__ RenderEnv<NC, NT, NO> s;
    const int tiles_x = (size + kRenderCols - 1) / kRenderCols;
    const int ty0 = (int)blockIdx.x / tiles_x, tx0 = (int)blockIdx.x - ty0 * tiles_x;
    const int i0 = ty0 * kRenderRows, j0 = tx0 * kRenderCols;
    const int i1 = min(i0 + kRenderRows, size) - 1, j1 = min(j0 + kRenderCols, size) - 1;
    const double xlo = render_x(j0, size), xhi = render_x(j1, size), ylo = render_y(i1, size), yhi = render_y(i0, size);
    const double pitch = __ddiv_rn(2.0 * MATE_RENDER_HALF_EXTENT, (double)size);
    const double r_in = fmax(MATE_RENDER_TARGET_INNER, __dmul_rn(MATE_RENDER_TARGET_INNER_PITCH, pitch));
    const double r_out = fmax(MATE_RENDER_TARGET_OUTER, __dmul_rn(MATE_RENDER_TARGET_OUTER_PITCH, pitch));
    const double r_in2 = __dmul_rn(r_in, r_in), r_out2 = __dmul_rn(r_out, r_out);
    const double cam_r2 = __dmul_rn(p.cam_radius, p.cam_radius);
    const int tid = threadIdx.x;
    const int row = i0 + tid / (kRenderCols / 4), col = j0 + 4 * (tid % (kRenderCols / 4));
    const size_t bp = p.bpad;

    for (int f = blockIdx.y; f < count; f += gridDim.y) {
        const int e = env ? env[f] : f;
        if (e < 0 || e >= p.num_envs) continue;   // uniform over the CTA
        __syncthreads();                          // the previous frame's reads of `s` are done
        if (tid < NC) {
            const size_t k = (size_t)tid * bp + e;
            const double x = p.cam_x[k], y = p.cam_y[k], phi = p.cam_phi[k], theta = p.cam_theta[k];
            const double rs = sqrt(p.cam_area_product / theta);
            double sn, cs;
            sincospi(phi * (1.0 / 180.0), &sn, &cs);
            s.cx[tid] = x; s.cy[tid] = y; s.phi[tid] = phi; s.theta[tid] = theta; s.rs[tid] = rs;
            s.fcx[tid] = (float)x; s.fcy[tid] = (float)y;
            const float hx = (float)(rs * cs), hy = (float)(rs * sn), ch = cospif((float)theta * (1.0f / 360.0f));
            s.hx[tid] = hx; s.hy[tid] = hy; s.rs2[tid] = hx * hx + hy * hy; s.ch2[tid] = ch * ch;
        }
        if (tid >= 32 && tid < 32 + NT) {
            const size_t k = (size_t)(tid - 32) * bp + e;
            s.tx[tid - 32] = p.tgt_x[k]; s.ty[tid - 32] = p.tgt_y[k]; s.tpack[tid - 32] = p.tgt_pack[k];
        }
        if (tid >= 64 && tid < 64 + NO) {
            const size_t k = (size_t)(tid - 64) * bp + e;
            s.ox[tid - 64] = p.obs_x[k]; s.oy[tid - 64] = p.obs_y[k]; s.orad[tid - 64] = p.obs_r[k]; s.of4[tid - 64] = p.obs_f4[k];
        }
        if (tid == 0) s.tracked = 0u;
        __syncthreads();
        if (tid < 32) {   // the tile's lists (a margin of one unit keeps every culled entity clear of the tile)
            const int lane = tid;
            uint32_t fov = 0u, cams = 0u, tgts = 0u;
            if (lane < NC) {
                const double d2 = box_d2(s.cx[lane], s.cy[lane], xlo, xhi, ylo, yhi);
                const double reach = s.rs[lane] + 1.0, body = p.cam_radius + 1.0;
                fov = d2 <= reach * reach ? 1u << lane : 0u;
                cams = d2 <= body * body ? 1u << lane : 0u;
            }
            if (lane < NT) {
                const double reach = r_out + 1.0;
                tgts = box_d2(s.tx[lane], s.ty[lane], xlo, xhi, ylo, yhi) <= reach * reach ? 1u << lane : 0u;
            }
            uint32_t obs = 0u;
            if (lane < NO) {
                const double reach = s.orad[lane] + 1.0;
                obs = box_d2(s.ox[lane], s.oy[lane], xlo, xhi, ylo, yhi) <= reach * reach ? 1u << lane : 0u;
            }
            fov = __reduce_or_sync(0xffffffffu, fov); cams = __reduce_or_sync(0xffffffffu, cams);
            tgts = __reduce_or_sync(0xffffffffu, tgts); obs = __reduce_or_sync(0xffffffffu, obs);
            if (lane == 0) { s.fov_cams = fov; s.draw_cams = cams; s.draw_tgts = tgts; s.draw_obs = obs; }
        }
        __syncthreads();
        if (NC > 0 && tid < NC * NT) {   // "tracked": some camera sees the target's own location
            const int c = tid / (NT > 0 ? NT : 1), t = tid - c * (NT > 0 ? NT : 1);
            if (((s.draw_tgts >> t) & 1u) && render_sees(p, s, c, s.tx[t], s.ty[t])) atomicOr(&s.tracked, 1u << t);
        }
        __syncthreads();
        if (row >= size || col >= size) continue;

        const double y = render_y(row, size);
        uint32_t rgb[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (col + k >= size) { rgb[k] = 0u; continue; }
            const double x = render_x(col + k, size);
            uint32_t c = (fabs(x) <= kTerrain && fabs(y) <= kTerrain) ? MATE_RENDER_TERRAIN : MATE_RENDER_OUTSIDE;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                const double wx = (w == 0 || w == 3) ? MATE_RENDER_WAREHOUSE_CENTER : -MATE_RENDER_WAREHOUSE_CENTER;
                const double wy = (w < 2) ? MATE_RENDER_WAREHOUSE_CENTER : -MATE_RENDER_WAREHOUSE_CENTER;
                if (fmax(fabs(__dadd_rn(x, -wx)), fabs(__dadd_rn(y, -wy))) <= MATE_RENDER_WAREHOUSE_HALF_SIZE)
                    c = w == 0 ? MATE_RENDER_WAREHOUSE_0 : w == 1 ? MATE_RENDER_WAREHOUSE_1 : w == 2 ? MATE_RENDER_WAREHOUSE_2 : MATE_RENDER_WAREHOUSE_3;
            }
            for (uint32_t m = s.fov_cams; m != 0u; m &= m - 1u)
                if (render_sees(p, s, __ffs(m) - 1, x, y)) c = render_blend(c, MATE_RENDER_FOV);
            for (uint32_t m = s.draw_obs; m != 0u; m &= m - 1u) {
                const int o = __ffs(m) - 1;
                if (render_d2(__dadd_rn(x, -s.ox[o]), __dadd_rn(y, -s.oy[o])) <= __dmul_rn(s.orad[o], s.orad[o])) c = MATE_RENDER_OBSTACLE;
            }
            for (uint32_t m = s.draw_cams; m != 0u; m &= m - 1u) {
                const int cc = __ffs(m) - 1;
                if (render_d2(__dadd_rn(x, -s.cx[cc]), __dadd_rn(y, -s.cy[cc])) <= cam_r2) c = MATE_RENDER_CAMERA;
            }
            for (uint32_t m = s.draw_tgts; m != 0u; m &= m - 1u) {
                const int t = __ffs(m) - 1;
                const double d2 = render_d2(__dadd_rn(x, -s.tx[t]), __dadd_rn(y, -s.ty[t]));
                if (d2 <= r_in2) {
                    const uint32_t q = s.tpack[t];
                    const int g = tp_goal(q);
                    c = (g >= 0 && tp_weight(q) > 0)
                            ? (g == 0 ? MATE_RENDER_WAREHOUSE_0 : g == 1 ? MATE_RENDER_WAREHOUSE_1 : g == 2 ? MATE_RENDER_WAREHOUSE_2 : MATE_RENDER_WAREHOUSE_3)
                            : MATE_RENDER_TARGET_EMPTY;
                } else if (d2 <= r_out2 && ((s.tracked >> t) & 1u)) {
                    c = MATE_RENDER_TRACKED;
                }
            }
            rgb[k] = c;
        }
        // bytes R, G, B per pixel: 0xRRGGBB -> memory order
        uint8_t* dst = out + ((size_t)f * size * size + (size_t)row * size + col) * 3;
        if (words && col + 3 < size) {
            uint32_t b[12];
#pragma unroll
            for (int k = 0; k < 4; ++k) { b[3 * k] = (rgb[k] >> 16) & 0xFFu; b[3 * k + 1] = (rgb[k] >> 8) & 0xFFu; b[3 * k + 2] = rgb[k] & 0xFFu; }
            uint32_t* d32 = reinterpret_cast<uint32_t*>(dst);
#pragma unroll
            for (int w = 0; w < 3; ++w) d32[w] = b[4 * w] | (b[4 * w + 1] << 8) | (b[4 * w + 2] << 16) | (b[4 * w + 3] << 24);
        } else {
            for (int k = 0; k < 4 && col + k < size; ++k) {
                dst[3 * k] = (uint8_t)(rgb[k] >> 16); dst[3 * k + 1] = (uint8_t)(rgb[k] >> 8); dst[3 * k + 2] = (uint8_t)rgb[k];
            }
        }
    }
}

}  // namespace mate
