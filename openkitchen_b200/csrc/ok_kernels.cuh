// ok_kernels.cuh -- the auxiliary kernels of the C ABI (ok_capi.cu): agent resets, the genetic policy, track queries, the
// host flush of observations, the PCIe probe, the CMA-ES controller, the PPO actor, discounted returns, population
// counters, sincosf and action fills.  The step kernels are in ok_step.cuh.
#pragma once

#include "ok_device.cuh"

namespace ok
{

// Environment::resetAgent (Environment.cpp:79-122) + Agent::reset (Agent.cpp:123-135) of agent `a` with the draws
// (pt, alpha, off) made explicit, and the episode bookkeeping (main_eigen.cpp:121-130: prev_track_idx_ = nearest index of the
// post-reset pose, fitness restarts) and the restart of the lap state (OkLaps, with accounting on or off); the standstill
// record is not touched (Environment.cpp never resets it).
__device__ __forceinline__ void reset_agent(const StepParams &p, const TrackView &tv, const int64_t a, const int32_t pt, const bool lane,
                                            const float alpha, const float off)
{
    const float3 q = reset_pose(tv.pts, tv.headings, tv.seg, tv.n_pts, pt, lane, alpha, off);
    p.x[a] = q.x, p.y[a] = q.y;
    p.rot[a]       = q.z;
    p.accel[a]     = 0.0f;
    p.speed[a]     = 0.0f;
    p.crashed[a]   = 0;
    p.timed_out[a] = 0;
    p.done[a]      = 0;
    p.act_thr[a]   = 0.0f;
    p.act_steer[a] = 0.0f;
    p.reset_pt[a]  = pt;
    p.start_x[a]   = q.x;
    p.start_y[a]   = q.y;
    float   d2;
    int32_t near  = nearest_index(tv, q.x, q.y, 0, 1, d2);
    p.prev[a]     = near;
    p.nearest[a]  = near;
    p.fitness[a]  = 0.0f;
    p.reward[a]   = 0.0f;
    lap_restart(p.lap, a, near);
}

// ok_reset_agents: one thread per request, reading the track blobs from global memory.
struct ResetParams
{
    const int64_t *agent_idx; // nullable
    const int32_t *pt_idx;
    const float   *lane_alpha;  // nullable
    const float   *heading_off; // nullable
    int64_t        n, n_agents;
};

__global__ void reset_kernel(const StepParams p, const ResetParams r)
{
    const int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k >= r.n)
        return;
    const int64_t a = r.agent_idx ? r.agent_idx[k] : k;
    if (a < 0 || a >= r.n_agents)
        return;
    const TrackView tv = make_view(p.arena + p.tracks[p.track_id[a]].offset);
    const int32_t   pt = min(max(r.pt_idx[k], 0), tv.n_pts - 1);
    reset_agent(p, tv, a, pt, r.lane_alpha != nullptr, r.lane_alpha ? r.lane_alpha[k] : 0.0f, r.heading_off ? r.heading_off[k] : 0.0f);
}

// ok_reset_agents_drawn: a drawn reset (reset_draw) of agent agent_idx[k], or of agent k when mask is NULL or mask[k] != 0;
// one thread per request.
struct DrawnResetParams
{
    const int64_t *agent_idx; // nullable
    const uint8_t *mask;      // nullable; not with agent_idx
    int64_t        n, n_agents;
};

__global__ void reset_drawn_kernel(const StepParams p, const DrawnResetParams r)
{
    const int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k >= r.n)
        return;
    const int64_t a = r.agent_idx ? r.agent_idx[k] : k;
    if (a < 0 || a >= r.n_agents || (r.mask && !r.mask[a]))
        return;
    const TrackView tv = make_view(p.arena + p.tracks[p.track_id[a]].offset);
    const uint32_t  k0 = p.reset_k[a];
    const ResetDraw d  = reset_draw(p.reset_seed, p.reset_flags, p.id_base + static_cast<uint64_t>(a), k0, tv.n_pts,
                                    min(kStartingIdx, tv.n_pts - 1));
    reset_agent(p, tv, a, d.pt, d.lane, d.alpha, d.off);
    p.reset_k[a] = k0 + 1u;
}

// ok_set_laps switching accounting on: the restart of every agent's lap state at its current pose, one thread per agent.
__global__ void laps_restart_kernel(const StepParams p)
{
    const int64_t a = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= p.n_agents)
        return;
    const TrackView tv = make_view(p.arena + p.tracks[p.track_id[a]].offset);
    float           d2;
    lap_restart(p.lap, a, nearest_index(tv, p.x[a], p.y[a], 0, 1, d2));
}

// GeneticAgent::updateAction + Network::infer for every agent (EvolutionaryRacer/GeneticAgent.hpp:37-50,
// Network.hpp:119-155).  One warp per agent, lane j = hidden unit j.  The weights are streamed exactly once with
// coalesced row reads (W1 row i = `hidden` consecutive floats), so the kernel is HBM bound:
// 4*(R+2)*hidden + 4*hidden*6 bytes per agent (4,800 B at R = 32, hidden = 30).
__global__ void genetic_policy_kernel(const StepParams p, const float *__restrict__ w1, const float *__restrict__ w2,
                                      int hidden, int64_t n_agents)
{
    const int     lane = threadIdx.x & 31;
    const int64_t a    = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (a >= n_agents)
        return;
    const int    R      = p.rays;
    const int    inputs = R + 2;
    const float *W1     = w1 + a * inputs * hidden;
    const float *W2     = w2 + a * hidden * 6;
    // inputs, Network.hpp:125-132
    float rot = p.rot[a];
    int   guard = 0;
    while (rot < 360.0f && guard++ < 100000) // normalizeAngleDeg, Utils.h:3-14
        rot = fadd(rot, 360.0f);
    while (rot >= 360.0f && guard++ < 200000)
        rot = fsub(rot, 360.0f);
    const float in0 = __fdiv_rn(p.speed[a], p.speed_limit);
    const float in1 = __fdiv_rn(rot, 360.0f);
    const bool  unit = lane < hidden;
    float       acc  = 0.0f;
    if (unit)
    {
        acc = fmul(in0, W1[lane]);
        acc = fadd(acc, fmul(in1, W1[hidden + lane]));
    }
    for (int r0 = 0; r0 < R; r0 += 32)
    { // 32 lidar inputs at a time: one coalesced read, then broadcast one by one
        const float mine = (r0 + lane < R) ? p.obs[a * R + r0 + lane] : 0.0f;
        const int   cnt  = min(32, R - r0);
        int         k    = 0;
        for (; k + 8 <= cnt; k += 8)
        { // 8 independent row loads in flight per lane
            float wv[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                wv[u] = unit ? W1[(2 + r0 + k + u) * hidden + lane] : 0.0f;
#pragma unroll
            for (int u = 0; u < 8; ++u)
                acc = fadd(acc, fmul(__shfl_sync(0xffffffffu, mine, k + u), wv[u]));
        }
        for (; k < cnt; ++k)
        {
            const float x = __shfl_sync(0xffffffffu, mine, k);
            if (unit)
                acc = fadd(acc, fmul(x, W1[(2 + r0 + k) * hidden + lane]));
        }
    }
    const float h = unit ? fmaxf(acc, 0.0f) : 0.0f; // relu
    float       o[6];
#pragma unroll
    for (int k = 0; k < 6; ++k)
        o[k] = unit ? fmul(h, W2[lane * 6 + k]) : 0.0f;
#pragma unroll
    for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int s = 16; s > 0; s >>= 1)
            o[k] = fadd(o[k], __shfl_xor_sync(0xffffffffu, o[k], s));
    if (lane == 0)
    {
        bool on[6];
#pragma unroll
        for (int k = 0; k < 6; ++k)
            on[k] = __fdiv_rn(1.0f, fadd(1.0f, expf(-o[k]))) > 0.5f; // sigmoid > kOutputActivationLim
        // GeneticAgent.hpp:37-50
        float thr = 0.0f, st = 0.0f;
        thr = fadd(thr, on[0] ? 0.3f : 0.0f);
        thr = fadd(thr, on[1] ? -0.3f : 0.0f);
        st  = fadd(st, on[2] ? 1.0f : 0.0f);
        st  = fadd(st, on[3] ? 4.0f : 0.0f);
        st  = fadd(st, on[4] ? -1.0f : 0.0f);
        st  = fadd(st, on[5] ? -4.0f : 0.0f);
        p.act_thr[a]   = thr;
        p.act_steer[a] = st;
    }
}

// RaceTrack::findNearestTrackIndexBruteForce / getDistanceToLaneCenter / getNearestDistanceToTrackBoundary
// (RaceTrack.cpp:16-72) for arbitrary query points: one warp per query, the 32 lanes split the points and combine with
// the order-independent lexicographic minimum (distance, index) -- the reference's strict '<' keeps the lowest index.
struct QueryParams
{
    const float   *x, *y;
    const int32_t *track; // nullable: track 0
    int64_t        n;
    int32_t        n_tracks;
    int32_t       *nearest;     // nullable outputs
    float         *lane_center; // sqrt(min d2) / (w_left + w_right) at the nearest point
    float         *boundary;    // sqrt(min d2 to the LI / RI points)
};

__global__ void track_query_kernel(const StepParams p, const QueryParams q)
{
    const int     lane = threadIdx.x & 31;
    const int64_t k    = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (k >= q.n)
        return;
    int32_t t = q.track ? q.track[k] : 0;
    t         = min(max(t, 0), q.n_tracks - 1);
    const TrackView tv = make_view(p.arena + p.tracks[t].offset);
    const float     qx = q.x[k], qy = q.y[k];
    if (q.nearest || q.lane_center)
    {
        float     d2;
        const int idx = nearest_index(tv, qx, qy, lane, 32, d2);
        if (lane == 0)
        {
            if (q.nearest)
                q.nearest[k] = idx;
            if (q.lane_center)
                q.lane_center[k] = __fdiv_rn(__fsqrt_rn(d2), tv.widths[idx]); // widths = w_left + w_right
        }
    }
    if (q.boundary)
    { // LI / RI points are the start points of the LI / RI segment chains; the last ones start the closure segments
        const int n    = tv.n_pts;
        float     best = FLT_MAX;
        for (int i = lane; i < n; i += 32)
        {
            const float4 ls = tv.seg[i < n - 1 ? i : 4 * (n - 1)];
            const float4 rs = tv.seg[i < n - 1 ? 2 * (n - 1) + i : 4 * (n - 1) + 1];
            float        ddx = fsub(qx, ls.x), ddy = fsub(qy, ls.y);
            float        d   = fadd(fmul(ddx, ddx), fmul(ddy, ddy));
            best             = d < best ? d : best;
            ddx = fsub(qx, rs.x), ddy = fsub(qy, rs.y);
            d   = fadd(fmul(ddx, ddx), fmul(ddy, ddy));
            best = d < best ? d : best;
        }
        for (int o = 16; o > 0; o >>= 1)
        {
            const float od = __shfl_xor_sync(0xffffffffu, best, o);
            best           = od < best ? od : best;
        }
        if (lane == 0)
            q.boundary[k] = __fsqrt_rn(best);
    }
}

// measurement only (ok_pcie_probe): full-warp 16-byte stores of a device buffer through a host mapping
// ok_step_host's flusher: a few CTAs on SMs of their own, launched next to the step kernel.  CTA f takes the tiles f, f + F,
// ... in list order, waits until the step kernel has published a tile (flag[tile] == epoch) and copies its observations
// from device memory (L2) to the pinned host buffer through the mapping, 16 bytes per lane.  The step kernel's CTAs never
// wait for the host link: they publish and move on.
__global__ void __launch_bounds__(1024, 1) obs_flush_kernel(const Tile *__restrict__ tiles, const int n_tiles, const uint32_t *flags, const uint32_t epoch,
                                                            const float *obs, float *host_obs, const int R)
{
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x)
    {
        if (threadIdx.x == 0)
        {
            uint32_t v;
            for (;;)
            {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + t) : "memory");
                if (v == epoch)
                    break;
                __nanosleep(200);
            }
        }
        __syncthreads();
        const Tile    tl   = tiles[t];
        const int64_t base = tl.begin * R;
        const int     n    = tl.count * R;
        const float  *src  = obs + base;
        float        *dst  = host_obs + base;
        if (((base | n) & 3) == 0)
            for (int i = threadIdx.x; i < (n >> 2); i += blockDim.x)
                reinterpret_cast<float4 *>(dst)[i] = __ldcg(reinterpret_cast<const float4 *>(src) + i);
        else
            for (int i = threadIdx.x; i < n; i += blockDim.x)
                dst[i] = __ldcg(src + i);
        __syncthreads(); // (thread 0 must not run ahead into the next wait while others still read `tl`: harmless, but keep the CTA together)
    }
}

__global__ void probe_store_kernel(const float4 *__restrict__ src, float4 *__restrict__ dst, size_t n)
{
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
        dst[i] = src[i];
}

// CmaEsAgent::updateAction + Controller::forward for every candidate of a CMA-ES population (main_torch.cpp:61-71,
// Controller.cpp:16-23): candidate a owns the flat parameter vector params[a] (torch parameters() order: fc1.weight
// [H][R], fc1.bias [H], fc2.weight [H/2][H], fc2.bias [H/2], fc3.weight [1][H/2], fc3.bias [1]) and evaluates
// tanh(fc3 tanh(fc2 tanh(fc1 obs))) on its own lidar observation; throttle = `throttle`, steering = out * steer_scale.
// One warp per agent.  The weights are read exactly once, every row as one coalesced warp load, so the kernel is HBM
// bound: 4 * (H*R + H + H*H/2 + H/2 + H/2 + 1) bytes per agent (2,692 B at R = 32, H = 16).  Sums are reduced across
// the warp with shuffles (a different summation order than the reference's sgemv: parity is to 1e-6 on tanh outputs).
template <int H> __device__ __forceinline__ float warp_reduce_rows(float (&v)[H], const int lane)
{ // in: v[j] = this lane's partial of row j; out: the full sum of row (lane & (H - 1)) -- H - 1 + (5 - log2 H) shuffles
    static_assert(H == 16, "written for the reference's 16 hidden units");
    float a8[8], a4[4], a2[2];
    {
        const bool hi = lane & 16;
#pragma unroll
        for (int j = 0; j < 8; ++j)
        {
            const float send = hi ? v[j] : v[j + 8];
            const float keep = hi ? v[j + 8] : v[j];
            a8[j]            = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool hi = lane & 8;
#pragma unroll
        for (int j = 0; j < 4; ++j)
        {
            const float send = hi ? a8[j] : a8[j + 4];
            const float keep = hi ? a8[j + 4] : a8[j];
            a4[j]            = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool hi = lane & 4;
#pragma unroll
        for (int j = 0; j < 2; ++j)
        {
            const float send = hi ? a4[j] : a4[j + 2];
            const float keep = hi ? a4[j + 2] : a4[j];
            a2[j]            = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
    }
    const bool  hi   = lane & 2;
    const float send = hi ? a2[0] : a2[1];
    const float keep = hi ? a2[1] : a2[0];
    float       r    = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    r += __shfl_xor_sync(0xffffffffu, r, 1);
    // lane bits (16, 8, 4, 2) chose row 8*b4 + 4*b3 + 2*b2 + b1: lane l holds row ((l >> 1) & 15)
    return r;
}

__global__ void __launch_bounds__(256) cmaes_controller_kernel(const StepParams p, const float *__restrict__ params,
                                                               const int n_params, const float throttle,
                                                               const float steer_scale, const int64_t n_agents)
{
    constexpr int H = 16, H2 = 8;
    const int     lane = threadIdx.x & 31;
    const int64_t a    = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (a >= n_agents)
        return;
    const int    R  = p.rays;
    const float *w  = params + a * n_params;
    const float *W1 = w, *b1 = w + H * R, *W2 = b1 + H, *b2 = W2 + H2 * H, *W3 = b2 + H2, *b3 = W3 + H2;
    // the small tail (fc1.bias .. fc3.bias: 16 + 128 + 8 + 8 + 1 = 161 floats) is requested up front
    const float bias1 = lane < H ? b1[lane] : 0.0f;
    float       w2[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        w2[k] = W2[lane + 32 * k]; // element (row (lane >> 4) + 2k, column lane & 15)
    const float bias2 = lane < H2 ? b2[lane] : 0.0f;
    const float w3    = lane < H2 ? W3[lane] : 0.0f;
    const float bias3 = b3[0];
    // layer 1: lane = input (mod 32), 16 row partials per lane
    float acc[H];
#pragma unroll
    for (int j = 0; j < H; ++j)
        acc[j] = 0.0f;
    for (int r0 = 0; r0 < R; r0 += 32)
    {
        const bool  in = r0 + lane < R;
        const float x  = in ? p.obs[a * R + r0 + lane] : 0.0f;
        float       wv[H];
#pragma unroll
        for (int j = 0; j < H; ++j)
            wv[j] = in ? W1[j * R + r0 + lane] : 0.0f; // 16 independent coalesced row loads in flight
#pragma unroll
        for (int j = 0; j < H; ++j)
            acc[j] = fmaf(wv[j], x, acc[j]);
    }
    const float row = warp_reduce_rows<H>(acc, lane); // lane l: row (l >> 1) & 15
    // hidden unit i to every lane with (lane & 15) == i
    const float h1 = tanhf(__shfl_sync(0xffffffffu, row, (lane & 15) << 1) + __shfl_sync(0xffffffffu, bias1, lane & 15));
    // layer 2: lane holds W2[(lane >> 4) + 2k][lane & 15]; sum over the 16 lanes of a half warp
    float o2[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        o2[k] = w2[k] * h1;
#pragma unroll
    for (int s = 8; s > 0; s >>= 1)
#pragma unroll
        for (int k = 0; k < 4; ++k)
            o2[k] += __shfl_xor_sync(0xffffffffu, o2[k], s);
    // row j of layer 2 sits in o2[j >> 1] of the half warp (j & 1): bring row `lane` to lanes 0..7
    float h2 = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k)
    {
        const float v = __shfl_sync(0xffffffffu, o2[k], (lane & 1) << 4);
        h2            = ((lane >> 1) == k) ? v : h2;
    }
    h2 = lane < H2 ? tanhf(h2 + bias2) : 0.0f;
    float o3 = w3 * h2;
#pragma unroll
    for (int s = 4; s > 0; s >>= 1)
        o3 += __shfl_xor_sync(0xffffffffu, o3, s);
    if (lane == 0)
    {
        p.act_thr[a]   = throttle;                                  // main_torch.cpp:68
        p.act_steer[a] = fmul(tanhf(o3 + bias3), steer_scale);      // main_torch.cpp:69
    }
}

__global__ void __launch_bounds__(256) ppo_actor_kernel(const StepParams p, const ActorParams q, const int64_t n_agents)
{
    extern __shared__ float s_w[]; // w1 | b1 | w2 | b2
    if (q.act)
        actor_stage_weights(q, p.rays, s_w, threadIdx.x, blockDim.x);
    __syncthreads();
    const int64_t a = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) / kActorLanes;
    actor_agent(p, q, s_w, a, a < n_agents, threadIdx.x & (kActorLanes - 1));
}

// ExperienceBuffer::calculateDiscountedRewards (RLRacers/PPO/ExperienceBuffer.hpp:45-62) for every agent: one thread per
// agent scans its column of rewards[T][N] backwards in binary32 with the reference's operation order
// (cum = r + gamma * cum, no contraction); done[t][a] != 0 cuts the scan where an episode ended at tick t.
__global__ void discounted_returns_kernel(const float *__restrict__ rewards, const uint8_t *__restrict__ done, float *__restrict__ out,
                                          const int32_t steps, const int64_t n_agents, const float gamma)
{
    const int64_t a = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= n_agents)
        return;
    float cum = 0.0f;
    for (int32_t t = steps - 1; t >= 0; --t)
    {
        const int64_t i = static_cast<int64_t>(t) * n_agents + a;
        if (done && done[i])
            cum = 0.0f;
        cum    = fadd(rewards[i], fmul(gamma, cum));
        out[i] = cum;
    }
}

// metrics (SURVEY 5, "per-step device counters"): how many agents are alive / crashed / timed out / done right now.
// out[4] must be zero; one atomic per warp and counter.
__global__ void population_counters_kernel(const uint8_t *__restrict__ crashed, const uint8_t *__restrict__ timed_out,
                                           const uint8_t *__restrict__ done, const int64_t n, unsigned long long *out)
{
    unsigned c[4] = {0u, 0u, 0u, 0u};
    for (int64_t a = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; a < n; a += static_cast<int64_t>(gridDim.x) * blockDim.x)
    {
        const bool cr = crashed[a] != 0;
        c[0] += !cr, c[1] += cr, c[2] += timed_out[a] != 0, c[3] += done[a] != 0;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
    {
        const unsigned w = __reduce_add_sync(0xffffffffu, c[k]);
        if ((threadIdx.x & 31) == 0 && w)
            atomicAdd(out + k, static_cast<unsigned long long>(w));
    }
}

__global__ void sincosf_kernel(const float *in, float *s_out, float *c_out, int64_t n)
{
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    float s, c;
    sincosf(in[i], s, c);
    s_out[i] = s;
    c_out[i] = c;
}

__global__ void fill_actions_kernel(const StepParams p, int64_t n)
{
    const int64_t a = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= n)
        return;
    uint32_t       o[4];
    const uint64_t id = p.id_base + static_cast<uint64_t>(a);
    philox4x32_10(static_cast<uint32_t>(id), static_cast<uint32_t>(id >> 32),
                  static_cast<uint32_t>(p.step), static_cast<uint32_t>(p.step >> 32), p.seed, 0u, o);
    float thr, steer;
    if (p.movement_mode == 1)
    {
        const uint32_t ti = o[0] % 3u, si = o[1] % 5u;
        thr   = ti == 0 ? -0.3f : (ti == 1 ? 0.0f : 0.3f);
        steer = si == 0 ? -4.0f : (si == 1 ? -1.0f : (si == 2 ? 0.0f : (si == 3 ? 1.0f : 4.0f)));
    }
    else
    {
        thr   = fmul(100.0f, fmul(static_cast<float>(o[0] >> 8), 0x1p-24f));
        steer = fsub(fmul(10.0f, fmul(static_cast<float>(o[1] >> 8), 0x1p-24f)), 5.0f);
    }
    p.act_thr[a]   = thr;
    p.act_steer[a] = steer;
}

} // namespace ok
