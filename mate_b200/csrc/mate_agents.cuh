// mate_agents.cuh -- batched rule-based opponents for the single-team wrappers (SURVEY.md section 8f, N4).
//
// GreedyTargetAgent (mate/agents/greedy.py:235-365), driven like MultiCamera drives its opponents
// (mate/wrappers/single_team.py:79-92, 261-279: observe -> communicate -> act), for all targets of all
// environments in one launch.  One thread = one environment: the team's message exchange (broadcast of the
// remembered non-empty warehouses, greedy.py:338-365, routed to every teammate, environment.py:1249-1269) is an
// AND over at most 8 four-bit sets and stays in registers; with communication wrappers registered (DESIGN.md section 7h)
// it is one AND per recipient over the copies that reached it.  The agents read their private state from the
// simulator's state arrays (not from the observation tensors, which observation wrappers may have transformed).
#pragma once

#include "mate_common.cuh"

namespace mate {

constexpr uint32_t STREAM_AGENT_BINOMIAL = 16, STREAM_AGENT_SAMPLE = 17, STREAM_AGENT_CHOICE = 18, STREAM_AGENT_RESET = 19, STREAM_AGENT_DELAY = 20;
constexpr uint32_t STREAM_AGENT_COMM = 21;
constexpr int kAgentMemory = 6;   // per target: goal, non-empty warehouse set, previous x, y, previous noise x, y; stored FIELD-MAJOR [6][Nt][B]

// The communication wrappers of one team as its agent kernel applies them (mate_b200_set_message_filter, DESIGN.md
// section 7h).  A message is delivered iff it passes the range rule and the dropout draw.
struct CommFilter {
    double range_limit;            // RestrictedCommunicationRange; +inf = unrestricted
    unsigned long long keep;       // kept iff its 32-bit draw < keep: 1 << 32 = no dropout, 0 = NoCommunication
    unsigned long long seed;       // the handle's Philox key (mate_b200_seed), not the agents' seed
    uint64_t* delivered;           // [B] nullable: bit 8 s + r = the message of s reached r in this call
    int32_t* totals;               // [B, N, N] nullable: delivered since the environment's agents were reset
    int pairwise;                  // greedy targets: decide per (sender, recipient) (N <= 8); 0 = every copy arrives
};

// RestrictedCommunicationRange: the distance in fp64 without fused multiply-add, so that NumPy decides it identically
__device__ inline bool comm_in_range(double sx, double sy, double rx, double ry, double limit) {
    if (isinf(limit)) return true;
    const double dx = __dsub_rn(sx, rx), dy = __dsub_rn(sy, ry);
    return __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))) <= limit;
}

// the Philox draw of rng_words, out of line on its own (mate_common.cuh, philox_rounds)
__device__ __noinline__ uint4 philox_comm(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    return philox_rounds(c0, c1, c2, c3, k0, k1);
}

// RandomMessageDropout: word r % 4 of the Philox call keyed on (handle seed, global environment, 'COMM') with counter
// (call serial, team, sender, r / 4); the draw does not depend on the batch split or on the lane that takes it
__device__ inline bool comm_kept(const CommFilter& f, uint32_t env, uint32_t serial, uint32_t team, int s, int r) {
    if (f.keep > 0xFFFFFFFFull) return true;
    if (f.keep == 0ull) return false;
    const uint4 w = philox_comm(serial, (STREAM_AGENT_COMM << 16) | (team << 8) | ((uint32_t)s << 2) | ((uint32_t)r >> 2),
                                env, 0x434F4D4Du /* 'COMM' */, (uint32_t)f.seed, (uint32_t)(f.seed >> 32));
    const uint32_t x = (r & 3) == 0 ? w.x : (r & 3) == 1 ? w.y : (r & 3) == 2 ? w.z : w.w;
    return x < f.keep;
}

// one sender's row of the per-episode totals [N] (sender-major): restarted at the agents' reset, then this call's row added
__device__ inline void add_edge_row(int32_t* total, int n, uint32_t row, bool reset) {
    if (!reset && row == 0u) return;
    for (int r = 0; r < n; ++r) {
        const int bit = (int)((row >> r) & 1u);
        if (reset) total[r] = bit;
        else if (bit) total[r] += 1;
    }
}

// one agent's view of a field-major table: entry k of the agent is `stride` doubles after entry k - 1
struct Field {
    double* base;
    size_t stride;
    __device__ __forceinline__ double& operator[](int k) const { return base[(size_t)k * stride]; }
    __device__ __forceinline__ Field from(int k) const { return Field{base + (size_t)k * stride, stride}; }
};

__global__ void greedy_target_kernel(const Params p, const int nt, double* __restrict__ memory, const uint8_t* __restrict__ reset_mask,
                                     const double noise_scale, const unsigned long long seed, const unsigned long long serial,
                                     const MateAgentReplay replay, const CommFilter comm, float* __restrict__ tgt_act) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.num_envs) return;
    const size_t bp = p.bpad;
    const bool reset = reset_mask != nullptr && reset_mask[e] != 0;
    const RngKey key{seed, (uint32_t)(p.env_index_base + e), 0x41474E54u /* 'AGNT' */};
    // per-step stride 16 = 2 * (at most 8 targets): the SAMPLE / RESET streams read draw + 2 t + {0, 1}, so with a
    // stride of 8 target t >= 4 at step s would have re-read the draw of target t - 4 at step s + 1
    const uint32_t draw = (uint32_t)serial * 16u;
    // observe -> process_messages (greedy.py:330-336), and the sets that are broadcast
    uint32_t sent_and = 15u;
    uint32_t senders = 0u, sent_sets = 0u;   // pairwise: bit s / bits 4 s .. 4 s + 3 = target s broadcasts this set
    for (int t = 0; t < nt; ++t) {
        const Field m{memory + (size_t)t * p.num_envs + e, (size_t)nt * p.num_envs};
        const uint32_t tp = p.tgt_pack[(size_t)t * bp + e];
        if (reset) {   // reset(observation), greedy.py:265-277
            const double x = p.tgt_x[(size_t)t * bp + e], y = p.tgt_y[(size_t)t * bp + e];
            const double step_size = p.tgt_step_size / (double)tp_capacity(tp);
            double sx, sy;
            if (replay.reset_sample) { sx = replay.reset_sample[((size_t)e * nt + t) * 2]; sy = replay.reset_sample[((size_t)e * nt + t) * 2 + 1]; }
            else {
                sx = (2.0 * rng_u01(key, STREAM_AGENT_RESET, draw + (uint32_t)t * 2u) - 1.0) * step_size;
                sy = (2.0 * rng_u01(key, STREAM_AGENT_RESET, draw + (uint32_t)t * 2u + 1u) - 1.0) * step_size;
            }
            m[0] = (tp_goal(tp) >= 0 && tp_weight(tp) > 0) ? (double)tp_goal(tp) : -1.0;
            m[1] = 15.0; m[2] = x; m[3] = y; m[4] = 0.5 * sx; m[5] = 0.5 * sy;
        }
        uint32_t non_empty = (uint32_t)m[1];
        const uint32_t seen = (uint32_t)tp_empty(tp);
        if (seen & non_empty) {
            non_empty &= ~seen;
            m[1] = (double)non_empty;
            sent_and &= non_empty;
            if (comm.pairwise) { senders |= 1u << t; sent_sets |= non_empty << (4 * t); }
        }
    }
    uint64_t delivered = 0ull;
    // receive_responses (greedy.py:355-365) + act (greedy.py:289-328)
    for (int t = 0; t < nt; ++t) {
        const Field m{memory + (size_t)t * p.num_envs + e, (size_t)nt * p.num_envs};
        const uint32_t tp = p.tgt_pack[(size_t)t * bp + e];
        const double x = p.tgt_x[(size_t)t * bp + e], y = p.tgt_y[(size_t)t * bp + e];
        const double step_size = p.tgt_step_size / (double)tp_capacity(tp);
        const bool state_has_goal = tp_goal(tp) >= 0 && tp_weight(tp) > 0;
        uint32_t received = sent_and;
        if (comm.pairwise) {   // recipient t ANDs the sets of the senders whose copy reached it (its own copy changes nothing)
            received = 15u;
            for (uint32_t rest = senders; rest != 0u; rest &= rest - 1u) {
                const int s = __ffs(rest) - 1;
                if (!comm_in_range(p.tgt_x[(size_t)s * bp + e], p.tgt_y[(size_t)s * bp + e], x, y, comm.range_limit) ||
                    !comm_kept(comm, key.env, (uint32_t)serial, 1u, s, t)) continue;
                received &= sent_sets >> (4 * s);
                delivered |= 1ull << (8 * s + t);
            }
        }
        const uint32_t non_empty = (uint32_t)m[1] & received;
        int goal = (int)m[0];
        if (state_has_goal) goal = tp_goal(tp);
        if (goal < 0 || (!state_has_goal && !((non_empty >> goal) & 1u))) {
            goal = -1;
            if (non_empty != 0u) {   // np_random.choice(list(non_empty_warehouses)): uniform over the set, ascending order
                if (replay.choice) goal = replay.choice[(size_t)e * nt + t];
                else {
                    int pick = (int)rng_below(key, STREAM_AGENT_CHOICE, draw + (uint32_t)t, (uint32_t)__popc(non_empty));
                    for (int w = 0; w < NW; ++w) if ((non_empty >> w) & 1u) { if (pick == 0) { goal = w; break; } --pick; }
                }
                goal = min(max(goal, 0), NW - 1);
            }
        }
        const double pdx = x - m[2], pdy = y - m[3];
        double ax = 0.0, ay = 0.0;
        if (goal >= 0) {
            ax = ((goal == 0 || goal == 3) ? kWarehouseCoord : -kWarehouseCoord) - x;
            ay = ((goal < 2) ? kWarehouseCoord : -kWarehouseCoord) - y;
        }
        const double norm = sqrt(ax * ax + ay * ay);
        if (norm > step_size) { const double k = step_size / norm; ax *= k; ay *= k; }
        const double prob = sqrt(pdx * pdx + pdy * pdy) > 0.2 * step_size ? 0.05 : 0.75;
        bool redraw;
        if (replay.binomial) redraw = replay.binomial[(size_t)e * nt + t] != 0;
        else redraw = rng_u01(key, STREAM_AGENT_BINOMIAL, draw + (uint32_t)t) < prob;
        double nx = m[4], ny = m[5];
        if (redraw) {   // noise_scale * action_space.sample(): uniform over the agent's own action box
            double sx, sy;
            if (replay.sample) { sx = replay.sample[((size_t)e * nt + t) * 2]; sy = replay.sample[((size_t)e * nt + t) * 2 + 1]; }
            else {
                sx = (2.0 * rng_u01(key, STREAM_AGENT_SAMPLE, draw + (uint32_t)t * 2u) - 1.0) * step_size;
                sy = (2.0 * rng_u01(key, STREAM_AGENT_SAMPLE, draw + (uint32_t)t * 2u + 1u) - 1.0) * step_size;
            }
            nx = noise_scale * sx; ny = noise_scale * sy;
        }
        ax = fmin(fmax(ax + nx, -step_size), step_size);
        ay = fmin(fmax(ay + ny, -step_size), step_size);
        reinterpret_cast<float2*>(tgt_act)[(size_t)e * nt + t] = make_float2((float)ax, (float)ay);
        m[0] = (double)goal; m[1] = (double)non_empty; m[2] = x; m[3] = y; m[4] = nx; m[5] = ny;
    }
    if (comm.delivered) comm.delivered[e] = delivered;
    if (comm.totals)
        for (int s = 0; s < nt; ++s) add_edge_row(comm.totals + ((size_t)e * nt + s) * nt, nt, (uint32_t)(delivered >> (8 * s)) & 0xFFu, reset);
}

// =============================================================================================
// GreedyCameraAgent (mate/agents/greedy.py:14-232) for the camera team of every environment, driven like
// MultiTarget drives its opponents (observe -> communicate -> act).  One THREAD = one camera agent; the agents of an
// environment are neighbouring lanes of a warp (Nc divides 32 for every preset).  Per camera the memory holds what the
// reference agent keeps between steps: the remembered public state of every target, the time-to-forget counters,
// never_loaded, the previous action, the communication delays per teammate, the set of known teammates and whether the
// agent's own state is still to be sent (first step after reset).  (Round 1: one thread per environment walked its
// 4 cameras one after the other.  Staging a warp's 32 agent memories in shared memory was measured too: 58 KB per
// block leave 12 warps per SM for a kernel whose time is the latency of fp64 chains, 0.26 ms.)  The peer-to-peer messages of a step (teammate
// state, tracked target states filtered by the recipient's range; environment.py:1249-1269 routes them through the
// message queues) are two registers of the sender, read by the recipients with warp shuffles between the send and
// the receive phase.
// Fields per camera (doubles): [4 Nt] memory (x, y, sight range, is_loaded) | [Nt] time2forget | [Nt] never_loaded |
// [2] previous action | [Nc] communication delay | neighbours (bit set) | has_state_message; stored FIELD-MAJOR,
// [M][B * Nc] (round 1 and the first half of round 2: one record per agent, every access of a warp 32 sectors wide).
// =============================================================================================
__host__ __device__ inline int camera_agent_memory(int nc, int nt) { return 6 * nt + nc + 4; }


constexpr int kCameraAgentThreads = 128;

__global__ void __launch_bounds__(kCameraAgentThreads)
greedy_camera_kernel(const Params p, const int nc, const int nt, double* __restrict__ memory,
                     const uint8_t* __restrict__ tracked, const uint8_t* __restrict__ reset_mask,
                     const unsigned long long seed, const unsigned long long serial,
                     const MateCameraAgentReplay replay, const CommFilter comm, float* __restrict__ cam_act) {
    constexpr int MAXN = 8;
    constexpr uint32_t FULL = 0xffffffffu;
    constexpr double kMemoryPeriod = 25.0, kRangeFactor = 1.1;   // greedy.py:22, 32
    const int M = camera_agent_memory(nc, nt);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long total = (long long)p.num_envs * nc;
    const long long first = ((long long)blockIdx.x * kCameraAgentThreads + warp * 32);   // first agent of this warp
    const long long agent = first + lane;
    const bool live = agent < total;
    const uint32_t active = __ballot_sync(FULL, live);          // whole environments: B * Nc agents, Nc divides 32
    if (!live) return;
    const long long ag = agent;
    const int e = (int)(ag / nc), c = (int)(ag - (long long)e * nc);
    const int lane0 = lane - c;                                  // lane of camera 0 of this environment
    const size_t bp = p.bpad;
    const bool reset = reset_mask != nullptr && reset_mask[e] != 0;
    const RngKey key{seed, (uint32_t)(p.env_index_base + e), 0x4341474Eu /* 'CAGN' */};
    const uint32_t draw = (uint32_t)serial * 64u;
    const double threshold = kRangeFactor * p.cam_rmax, thr2 = threshold * threshold;
    double tx[MAXN], ty[MAXN];
    uint32_t loaded = 0;
    for (int t = 0; t < nt; ++t) {
        tx[t] = p.tgt_x[(size_t)t * bp + e]; ty[t] = p.tgt_y[(size_t)t * bp + e];
        const uint32_t tp = p.tgt_pack[(size_t)t * bp + e];
        loaded |= (uint32_t)(tp_goal(tp) >= 0 && tp_weight(tp) > 0) << t;
    }
    const double my_x = p.cam_x[(size_t)c * bp + e], my_y = p.cam_y[(size_t)c * bp + e];
    // the memory is stored field-major, [M][B * Nc]: the agents of a warp read and write neighbouring doubles
    (void)M;
    const Field m{memory + ag, (size_t)total};
    const Field mem = m, t2f = m.from(4 * nt), never = m.from(5 * nt), prev = m.from(6 * nt), delay = m.from(6 * nt + 2);
    // ---- observe -> process_messages (greedy.py:104-115); send_responses (greedy.py:156-194)
    uint32_t msg_state = 0;                 // bit k: my state goes to camera k
    unsigned long long msg_targets = 0ull;  // byte k: the tracked targets I report to camera k
    uint32_t delivered_row = 0;             // bit k: my message reached camera k
    {
        uint32_t seen = 0;
        for (int t = 0; t < nt; ++t) seen |= (uint32_t)(tracked[((size_t)e * nc + c) * nt + t] != 0) << t;
        if (reset) {   // reset(observation), greedy.py:44-66: untracked targets read as zeros in the observation
            for (int t = 0; t < nt; ++t) {
                const bool s = (seen >> t) & 1u;
                mem[4 * t] = s ? tx[t] : 0.0; mem[4 * t + 1] = s ? ty[t] : 0.0; mem[4 * t + 2] = s ? p.tgt_sight_range : 0.0;
                mem[4 * t + 3] = s ? (double)((loaded >> t) & 1u) : 0.0;
                t2f[t] = s ? kMemoryPeriod : 0.0;
                never[t] = 1.0;
            }
            prev[0] = prev[1] = 0.0;
            for (int k = 0; k < nc; ++k) delay[k] = 0.0;
            m[6 * nt + 2 + nc] = 0.0;      // neighbours
            m[6 * nt + 3 + nc] = 1.0;      // message2send['state']
        }
        for (int t = 0; t < nt; ++t) {
            t2f[t] = fmax(t2f[t] - 1.0, 0.0);
            if ((seen >> t) & 1u) {
                t2f[t] = kMemoryPeriod;
                mem[4 * t] = tx[t]; mem[4 * t + 1] = ty[t]; mem[4 * t + 2] = p.tgt_sight_range; mem[4 * t + 3] = (double)((loaded >> t) & 1u);
                if ((loaded >> t) & 1u) never[t] = 0.0;
            }
        }
        const uint32_t neighbours = (uint32_t)m[6 * nt + 2 + nc];
        const bool has_state = m[6 * nt + 3 + nc] != 0.0;
        for (int k = 0; k < nc; ++k) delay[k] = fmax(delay[k] - 1.0, 0.0);
        // bit k: a message to camera k would pass the communication wrappers; decided in a pass of its own (uniform
        // branch) so that the send loop below keeps the registers it had without wrappers
        uint32_t pass = 0xFFu;
        if (!isinf(comm.range_limit) || comm.keep <= 0xFFFFFFFFull) {
            pass = 0u;
            for (int k = 0; k < nc; ++k) {
                const double kx = __shfl_sync(active, my_x, lane0 + k), ky = __shfl_sync(active, my_y, lane0 + k);
                if (comm_in_range(my_x, my_y, kx, ky, comm.range_limit) && comm_kept(comm, key.env, (uint32_t)serial, 0u, c, k))
                    pass |= 1u << k;
            }
        }
        for (int k = 0; k < nc; ++k) {      // every lane takes part in the shuffles; the recipient's location comes from its lane
            const double kx = __shfl_sync(active, my_x, lane0 + k), ky = __shfl_sync(active, my_y, lane0 + k);
            if (!(has_state || seen != 0u) || k == c || delay[k] > 0.0) continue;
            uint32_t targets = 0;
            if (seen != 0u && ((neighbours >> k) & 1u)) {   // the recipient's range (all cameras share max_sight_range)
                for (int t = 0; t < nt; ++t) {   // norm < threshold, decided on squares; the square root only inside a 1e-12 band
                    const double dx = tx[t] - kx, dy = ty[t] - ky, d2 = dx * dx + dy * dy;
                    if (!((seen >> t) & 1u) || d2 > thr2 * (1.0 + 1e-12)) continue;
                    if (d2 < thr2 * (1.0 - 1e-12) || sqrt(d2) < threshold) targets |= 1u << t;
                }
            }
            if (has_state || targets != 0u) {
                int d;   // np_random.randint(memory_period // 4, 2 * memory_period)
                if (replay.delay) d = replay.delay[((size_t)e * nc + c) * nc + k];
                else d = 6 + (int)rng_below(key, STREAM_AGENT_DELAY, draw + (uint32_t)(c * MAXN + k), 44u);
                delay[k] = (double)d;
                // the sender does not know about the communication wrappers: only the recipient misses a dropped message
                if (!((pass >> k) & 1u)) continue;
                msg_state |= has_state ? (1u << k) : 0u;
                msg_targets |= (unsigned long long)targets << (8 * k);
                delivered_row |= 1u << k;
            }
        }
        if (has_state || seen != 0u) m[6 * nt + 3 + nc] = 0.0;
    }
    // each lane adds its own row of the totals; the environment's bit matrix is the OR of its lanes' rows
    if (comm.totals) add_edge_row(comm.totals + ((size_t)e * nc + c) * nc, nc, delivered_row, reset);
    if (comm.delivered) {
        uint64_t bits = (uint64_t)delivered_row << (8 * c);
        for (int o = 1; o < nc; o <<= 1) bits |= __shfl_xor_sync(active, bits, o);   // the lanes of an environment: an aligned group of nc
        if (c == 0) comm.delivered[e] = bits;
    }
    // ---- receive_responses (greedy.py:196-232) + act (greedy.py:68-102)
    {
        uint32_t neighbours = (uint32_t)m[6 * nt + 2 + nc];
        for (int s = 0; s < nc; ++s) {
            const uint32_t s_state = __shfl_sync(active, msg_state, lane0 + s);
            const unsigned long long s_targets = __shfl_sync(active, msg_targets, lane0 + s);
            if (s == c) continue;
            if ((s_state >> c) & 1u) neighbours |= 1u << s;   // greedy.py:219 adds the sender unconditionally
            const uint32_t targets = (uint32_t)(s_targets >> (8 * c)) & 0xFFu;
            for (int t = 0; t < nt; ++t) {
                if (!((targets >> t) & 1u)) continue;
                mem[4 * t] = tx[t]; mem[4 * t + 1] = ty[t]; mem[4 * t + 2] = p.tgt_sight_range; mem[4 * t + 3] = (double)((loaded >> t) & 1u);
                t2f[t] = kMemoryPeriod;
                if ((loaded >> t) & 1u) never[t] = 0.0;
            }
        }
        m[6 * nt + 2 + nc] = (double)neighbours;
        // nearest remembered target within range_factor * max_sight_range (first minimum, ascending index)
        int nearest = -1;
        double best = 0.0;
        for (int t = 0; t < nt; ++t) {
            if (!(t2f[t] > 0.0)) continue;
            const double dx = mem[4 * t] - my_x, dy = mem[4 * t + 1] - my_y;
            const double dist = sqrt(dx * dx + dy * dy);
            if (!(dist < threshold)) continue;
            if (nearest < 0 || dist < best) { nearest = t; best = dist; }
        }
        double a0, a1;
        if (nearest >= 0) {   // act_from_target_states (greedy.py:117-154)
            const double phi = p.cam_phi[(size_t)c * bp + e], theta = p.cam_theta[(size_t)c * bp + e];
            const double dx = mem[4 * nearest] - my_x, dy = mem[4 * nearest + 1] - my_y;
            const double orientation = atan2(dy, dx) * kRad2Deg;
            double view;
            double sn, cs;
            sincospi(p.cam_min_view * (0.5 / 180.0), &sn, &cs);
            if (best * (1.0 + sn) >= p.cam_rmax) view = p.cam_min_view;
            else if (best <= sqrt(p.cam_area_product / 180.0) * 0.5) view = 180.0;
            else {
                double b = 180.0;
                for (int it = 0; it < 20; ++it) {   // the reference's 20 fixed-point steps; a step that reproduces its input ends them all
                    sincospi(fmin(b * 0.5, 90.0) * (1.0 / 180.0), &sn, &cs);
                    const double sight = best * (1.0 + sn);
                    const double b_next = p.cam_area_product / (sight * sight);
                    if (b_next == b) break;
                    b = b_next;
                }
                view = fmin(fmax(b, p.cam_min_view), 180.0);
            }
            a0 = fmin(fmax(normalize_angle(orientation - phi), -p.cam_rot_step), p.cam_rot_step);
            a1 = fmin(fmax(view - theta, -p.cam_zoom_step), p.cam_zoom_step);
        } else {
            bool fresh;
            if (replay.binomial) fresh = replay.binomial[(size_t)e * nc + c] == 1;
            else fresh = rng_u01(key, STREAM_AGENT_BINOMIAL, draw + (uint32_t)c) < 0.1;
            if (fresh) {
                if (replay.sample) { a0 = replay.sample[((size_t)e * nc + c) * 2]; a1 = replay.sample[((size_t)e * nc + c) * 2 + 1]; }
                else {
                    a0 = (2.0 * rng_u01(key, STREAM_AGENT_SAMPLE, draw + (uint32_t)c * 2u) - 1.0) * p.cam_rot_step;
                    a1 = (2.0 * rng_u01(key, STREAM_AGENT_SAMPLE, draw + (uint32_t)c * 2u + 1u) - 1.0) * p.cam_zoom_step;
                }
            } else { a0 = prev[0]; a1 = prev[1]; }
        }
        prev[0] = a0; prev[1] = a1;
        reinterpret_cast<float2*>(cam_act)[(size_t)e * nc + c] = make_float2((float)a0, (float)a1);
    }
}

}  // namespace mate
