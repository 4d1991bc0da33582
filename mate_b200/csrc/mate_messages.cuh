// mate_messages.cuh -- the tensor message channel of a learning team in batched mode (mate_b200_exchange_messages,
// DESIGN.md section 7i): every agent of the team sends one message of D floats to a set of teammates, the team's
// registered communication wrappers (mate_b200_set_message_filter) decide which routed copies arrive, and the kernel
// writes the recipients' inboxes (or their sum / mean over the delivered senders) and the team's edge tensors.
//
// One warp per environment.  The up to 64 (sender, recipient) pairs are decided once, one or two per lane, and OR-reduced
// into the environment's 64-bit delivered set (bit 8 s + r).  The inbox of recipient r is a masked copy of the
// environment's content block [N][D], so lanes walk that block in 16-byte (or 4-byte) words: each word of the content is
// read once and stored to the N recipients' inboxes with streaming stores.  A reduction gives each lane (recipient,
// D-chunk) items and adds the delivered senders in ascending order.
#pragma once

#include "mate_agents.cuh"

namespace mate {

constexpr uint32_t STREAM_MESSAGE_EXCHANGE = 22;   // beside STREAM_AGENT_COMM = 21 of the greedy teams
constexpr int kExchangeWarps = 8;                  // environments per block

struct ExchangeArgs {
    const float* content;          // [B, N, D]
    const uint8_t* recipients;     // [B, N, N] sender-major, non-zero = s sends to r; nullptr = broadcast
    float* inbox;                  // [B, N(r), N(s), D] (MATE_MESSAGES_NONE) or [B, N, D]
    uint8_t* delivered;            // [B, N(r), N(s)]: 1 = s's message reached r; nullable
    int32_t* episode;              // [B]: the episode the team's totals belong to
    const double* x; const double* y;   // the team's positions [N][bpad]
    const int4* env_b;             // [bpad], w: episode id
    CommFilter comm;               // the team's registered range, keep, seed and edge tensors
    int num_envs, bpad, n, dim, reduction, vec;   // vec: D % 4 == 0 and content / inbox 16-byte aligned
    uint32_t team, serial;
    long long env_index_base;
};

// RandomMessageDropout for the channel: word r % 4 of the Philox call keyed on (handle seed, global environment,
// 'COMM') with counter (call serial, STREAM_MESSAGE_EXCHANGE, team, sender, r / 4).  The rounds are inlined here: a
// call of an out-of-line Philox would change the register allocation of the kernels that already call it.
__device__ __forceinline__ bool exchange_kept(const CommFilter& f, uint32_t env, uint32_t serial, uint32_t team, int s, int r) {
    if (f.keep > 0xFFFFFFFFull) return true;
    if (f.keep == 0ull) return false;
    const uint4 w = philox_rounds(serial, (STREAM_MESSAGE_EXCHANGE << 16) | (team << 8) | ((uint32_t)s << 2) | ((uint32_t)r >> 2),
                                  env, 0x434F4D4Du /* 'COMM' */, (uint32_t)f.seed, (uint32_t)(f.seed >> 32));
    const uint32_t x = (r & 3) == 0 ? w.x : (r & 3) == 1 ? w.y : (r & 3) == 2 ? w.z : w.w;
    return x < f.keep;
}

__device__ __forceinline__ float exchange_zero(float) { return 0.0f; }
__device__ __forceinline__ float4 exchange_zero(float4) { return make_float4(0.0f, 0.0f, 0.0f, 0.0f); }
__device__ __forceinline__ float exchange_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float4 exchange_add(float4 a, float4 b) {
    return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
}
__device__ __forceinline__ float exchange_div(float a, float c) { return __fdiv_rn(a, c); }
__device__ __forceinline__ float4 exchange_div(float4 a, float c) {
    return make_float4(__fdiv_rn(a.x, c), __fdiv_rn(a.y, c), __fdiv_rn(a.z, c), __fdiv_rn(a.w, c));
}

// MATE_MESSAGES_NONE: inbox[r][s][:] = content[s][:] where s reached r, else zeros.  Word q of the content block
// [N][W] (W words per message) goes to word q of every recipient's block; a sender that reached nobody is not read.
template <typename T>
__device__ __forceinline__ void exchange_copy(const ExchangeArgs& a, int e, int lane, unsigned long long set) {
    const int n = a.n, w = a.dim / (int)(sizeof(T) / sizeof(float)), words = n * w;
    const T* __restrict__ src = reinterpret_cast<const T*>(a.content) + (size_t)e * words;
    T* __restrict__ dst = reinterpret_cast<T*>(a.inbox) + (size_t)e * n * words;
    const T zero = exchange_zero(T{});
    for (int q = lane; q < words; q += 32) {
        const int s = q / w;
        const uint32_t reached = (uint32_t)(set >> (8 * s)) & 0xFFu;   // bit r: s's message reached r
        T v = zero;
        if (reached != 0u) v = __ldg(src + q);
        for (int r = 0; r < n; ++r) __stcs(dst + (size_t)r * words + q, ((reached >> r) & 1u) ? v : zero);
    }
}

// MATE_MESSAGES_SUM / _MEAN: out[r][:] = the chain of float32 adds of the delivered senders' messages in ascending s,
// from 0; the mean divides it by their number (0 when there is none)
template <typename T>
__device__ __forceinline__ void exchange_reduce(const ExchangeArgs& a, int e, int lane, unsigned long long set) {
    const int n = a.n, w = a.dim / (int)(sizeof(T) / sizeof(float)), words = n * w;
    const T* __restrict__ src = reinterpret_cast<const T*>(a.content) + (size_t)e * words;
    T* __restrict__ dst = reinterpret_cast<T*>(a.inbox) + (size_t)e * words;
    for (int q = lane; q < words; q += 32) {
        const int r = q / w, d = q - r * w;
        T acc = exchange_zero(T{});
        int count = 0;
        for (int s = 0; s < n; ++s) {
            if (!((set >> (8 * s + r)) & 1ull)) continue;
            acc = exchange_add(acc, __ldg(src + (size_t)s * w + d));
            ++count;
        }
        if (a.reduction == MATE_MESSAGES_MEAN) acc = count > 0 ? exchange_div(acc, (float)count) : exchange_zero(T{});
        __stcs(dst + q, acc);
    }
}

__global__ void __launch_bounds__(kExchangeWarps * 32) message_exchange_kernel(const ExchangeArgs a) {
    constexpr uint32_t FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int e = blockIdx.x * kExchangeWarps + (int)(threadIdx.x >> 5);
    if (e >= a.num_envs) return;   // the whole warp
    const int n = a.n, pairs = n * n;
    const size_t bp = a.bpad;
    const uint32_t env = (uint32_t)(a.env_index_base + e);
    const int episode = a.env_b[e].w;
    const bool restart = a.comm.totals != nullptr && a.episode[e] != episode;   // the first exchange of a new episode
    // ---- decide pair p = s n + r (sender-major); s = floor(p / n) exactly for p < 64 with a 16-bit reciprocal
    const uint32_t inv_n = (65536u + (uint32_t)n - 1u) / (uint32_t)n;
    uint32_t lo = 0u, hi = 0u;   // bits 8 s + r of the delivered set
    for (int p = lane; p < pairs; p += 32) {
        const int s = (int)(((uint32_t)p * inv_n) >> 16), r = p - s * n;
        bool ok = a.recipients == nullptr || a.recipients[(size_t)e * pairs + p] != 0;
        ok = ok && comm_in_range(a.x[s * bp + e], a.y[s * bp + e], a.x[r * bp + e], a.y[r * bp + e], a.comm.range_limit);
        ok = ok && exchange_kept(a.comm, env, a.serial, a.team, s, r);
        const int bit = 8 * s + r;
        if (ok) { if (bit < 32) lo |= 1u << bit; else hi |= 1u << (bit - 32); }
        if (a.delivered) a.delivered[(size_t)e * pairs + r * n + s] = ok ? 1 : 0;
        if (a.comm.totals) {
            int32_t* total = a.comm.totals + (size_t)e * pairs + p;
            if (restart) *total = ok ? 1 : 0;
            else if (ok) *total += 1;
        }
    }
    lo = __reduce_or_sync(FULL, lo);
    hi = __reduce_or_sync(FULL, hi);
    const unsigned long long set = ((unsigned long long)hi << 32) | lo;
    if (lane == 0) {   // every lane has read episode[e] above
        if (a.comm.delivered) a.comm.delivered[e] = set;
        if (restart) a.episode[e] = episode;
    }
    // ---- the inboxes
    if (a.reduction == MATE_MESSAGES_NONE) {
        if (a.vec) exchange_copy<float4>(a, e, lane, set);
        else exchange_copy<float>(a, e, lane, set);
    } else {
        if (a.vec) exchange_reduce<float4>(a, e, lane, set);
        else exchange_reduce<float>(a, e, lane, set);
    }
}

}  // namespace mate
