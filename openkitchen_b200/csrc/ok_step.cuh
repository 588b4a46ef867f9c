// ok_step.cuh -- the step kernels of the batched step loop and the tile loop they share.
//
// One fused kernel per tick replaces, per agent, the whole of
//   Environment::step stages 1-2            Environment.cpp:125-146
//     Agent::move                           Agent.cpp:82-98,108-119
//     checkAndUpdateStandstill              Environment.cpp:16-39
//     CollisionChecker pack/kernel/unpack   CollisionChecker.cu:8-71,113-172
//   + the app-side progress / reward / done RaceTrack.cpp:16-31,53-72 and SURVEY.md 8a row R
// with no host round trip.
//
// Mapping to the machine
//   * persistent CTAs, one per SM (the staged track fills most of the 227 KB of shared memory) x 1024 threads; the
//     agent range is cut into tiles (batches) of same-track agents that the CTAs pull from a global cursor;
//   * a track is staged with ONE TMA bulk copy (cp.async.bulk ... mbarrier::complete_tx) of its blob: segments as
//     float4, the uniform-grid cell table, the centre line; the copy runs under phase 1;
//   * phase 1 (kinematics, standstill; agent_pre) is one thread per agent; phase 4 (crash flag, nearest centre-line
//     index, reward; agent_post) four lanes or one thread per agent; both leave / read a 64-byte record per agent in
//     shared memory;
//   * the rays: beam_step_kernel reads precomputed candidate lists (ok_beam.hpp) -- warps pull groups of 32 rays, a ray's
//     first chunk of candidates is tested by its own lane, the rest is dealt evenly over the warp, results meet in a
//     64-bit atomicMin key per ray; grid_step_kernel (ok_step_grid.cu) walks a uniform grid ray by ray from a CTA-wide
//     pool (or tests every segment: the reference's loop);
//   * state is structure-of-arrays; per-ray outputs are written coalesced (lane = ray).
// The path is warp-issue bound, not HBM bound, and is not a contraction: no tensor cores (DESIGN.md section 4).
//
// Every step kernel is compiled in a translation unit of its own (ok_step_staged.cu, ok_step_unstaged.cu,
// ok_step_actor.cu, ok_step_grid.cu; tests/test_step_units_cpu.py checks it): with two of them in one unit ptxas shares
// the out-of-line device functions (beam_literal_key, beam_walk_fallback) between kernels with different launch bounds
// and address spaces, and the staged kernel lost a third of its speed (0.139 vs 0.095 ms per tick, DESIGN.md section 7).
#pragma once

#include "ok_device.cuh"

namespace ok
{

// The table constants the ray loop needs, in SHARED memory (beam kernel): they are uniform over a tile, and ptxas, short
// of registers, used to spill them to local memory -- where a CTA's 64 KB of stack frames thrash the ~23 KB of L1 this
// kernel leaves, so that every reload in the hot loop was a trip to the L2 (ncu: 328,000 local loads per launch, 1.7 %
// L1 hits).  Read through ld_hot() at the point of use: one LDS instead.
struct BeamHot
{
    const uint4 *entries;
    const uint2 *chunks;
    float        bin_scale, rb;
    int32_t      nb_mask, nb;
};
template <typename T> __device__ __forceinline__ T ld_hot(const T &field)
{
    return *const_cast<const volatile T *>(&field);
}

__device__ __forceinline__ BeamView make_beam_view(const TrackRef &tr)
{
    BeamView       v;
    const uint8_t *blob = reinterpret_cast<const uint8_t *>(tr.beam_offset);
    v.rows              = reinterpret_cast<const uint32_t *>(blob + tr.boff_rows);
    v.entries           = reinterpret_cast<const uint4 *>(blob + tr.boff_entries);
    v.chunks            = reinterpret_cast<const uint2 *>(blob + tr.boff_items);
    v.x0 = tr.bx0, v.y0 = tr.by0, v.inv_h = tr.binv_h, v.bin_scale = tr.bbin_scale, v.rb = tr.brb;
    v.nx = tr.bnx, v.ny = tr.bny, v.nb = tr.bnb;
    v.n_rows = tr.bn_rows, v.n_chunks = tr.bn_chunks;
    v.valid = true;
    return v;
}

__device__ __forceinline__ unsigned long long beam_key(float t, int idx)
{ // t >= 0 (-0.0 orders as +0.0: the reference compares values)
    const uint32_t tb = (t == 0.0f) ? 0u : __float_as_uint(t);
    return (static_cast<unsigned long long>(tb) << 32) | static_cast<uint32_t>(0x7fffffff - idx);
}

// One candidate, written without branches (a warp's lanes hold unrelated rays, so every branch here would be
// taken by a few lanes while the others wait) and free of dependences on the other candidates of the chunk, so
// the four evaluations of a chunk interleave.  Returns the approximate quotient tq = a * rcp(ad)
// (|tq - RN(t)| <= 2^-21 RN(t)) and two flags:
//   el  -- a real crossing comfortably inside the segment: s in [0,1] and t > 0 hold without a division, only
//          the order of its exact t matters;
//   lit -- on an edge of the segment or at the origin (rare): needs the reference's literal predicate.
// Everything else fails the reference's predicate (sufficient conditions, see test_segment).
__device__ __forceinline__ float beam_eval(const float4 *segs, const int idx, const float ox, const float oy,
                                           const float dx, const float dy, bool &el, bool &lit, float &a_out, float &ad_out)
{
    const float4   sg    = segs[idx];
    const float    ex    = fsub(sg.x, ox);
    const float    ey    = fsub(sg.y, oy);
    const float    denom = fsub(fmul(dx, sg.w), fmul(dy, sg.z));
    const float    sn    = fsub(fmul(ex, dy), fmul(ey, dx));
    const float    tn    = fsub(fmul(ex, sg.w), fmul(ey, sg.z));
    const uint32_t db    = __float_as_uint(denom);
    const uint32_t adb   = db & 0x7fffffffu;
    const uint32_t sgn   = db & 0x80000000u;
    const float    ad    = __uint_as_float(adb);
    const float    b     = __uint_as_float(__float_as_uint(sn) ^ sgn);
    const float    a     = __uint_as_float(__float_as_uint(tn) ^ sgn);
    const bool     rej   = (adb < 0x322BCC77u) | (b > ad) | (b < -0x1p-22f) | (a < -0x1p-22f);
    const bool     comfy = (b >= 0.0f) & (adb < 0x5d800000u /* 2^60 */) & (a >= 0x1p-60f);
    el                   = !rej & comfy;
    lit                  = !rej & !comfy;
    // a * rcp(ad): rcp.approx is within 1 ulp and the product adds half an ulp, inside the 2^-21 bound; where
    // `el` holds, ad < 2^60 and a >= 2^-60, so nothing is flushed or overflows
    // the exact quotient of a winner is a / ad: RN(tn / denom) bit for bit (both signs were flipped together)
    a_out = a, ad_out = ad;
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(ad));
    return fmul(a, r);
}

// literal predicate of the reference (CollisionChecker.cu:25-33) for a candidate flagged `lit`:
// returns the candidate's key (all ones = rejected)
static __device__ __noinline__ unsigned long long beam_literal_key(const float4 *segs, int idx, float ox, float oy, float dx, float dy)
{
    const float4 sg    = segs[idx];
    const float  ex    = fsub(sg.x, ox);
    const float  ey    = fsub(sg.y, oy);
    const float  denom = fsub(fmul(dx, sg.w), fmul(dy, sg.z));
    const float  sn    = fsub(fmul(ex, dy), fmul(ey, dx));
    const float  tn    = fsub(fmul(ex, sg.w), fmul(ey, sg.z));
    if (fabsf(denom) < 1e-8f)
        return ~0ull;
    const float t  = __fdiv_rn(tn, denom);
    const float s2 = __fdiv_rn(sn, denom);
    return ((s2 >= 0.0f) && (s2 <= 1.0f) && (t >= 0.0f)) ? beam_key(t, idx) : ~0ull;
}

__device__ __forceinline__ unsigned long long key_min(unsigned long long a, unsigned long long b)
{
    return a < b ? a : b;
}

// Four candidates (two packed words of uint16 segment indices) of ONE ray, entirely in registers: the best of them by
// the reference's rule folded into `key` ((exact t) << 32 | (0x7fffffff - segment), see beam_key).  `bound` = the
// ray's incumbent exact t (its key's high word, or the sensor range): a candidate whose approximate quotient is
// clearly beyond it is dropped without a division.  Every candidate is either strictly beaten by another one (the two
// quotients differ by more than both error bounds) or reaches the key with its exact IEEE quotient.
__device__ __forceinline__ unsigned long long beam_chunk_key(const float4 *segs, const uint32_t c01, const uint32_t c23,
                                                             const float ox, const float oy, const float dx, const float dy,
                                                             const float bound, unsigned long long key, const int n_seg = 0x7fffffff)
{
    int   idx[4];
    float tq[4], a[4], ad[4];
    bool  el[4], lit[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
    {
        // chunks are padded with the index of the track's null segment (zero length: denom = 0 fails the reference's
        // parallel test), so padding needs no special case
        idx[u] = static_cast<int>(((u < 2 ? c01 : c23) >> (16 * (u & 1))) & 0xffffu);
        OK_CHECK(idx[u] <= n_seg); // n_seg itself is the null segment
        tq[u]  = beam_eval(segs, idx[u], ox, oy, dx, dy, el[u], lit[u], a[u], ad[u]);
    }
    float tq_b  = bound, a_b = 0.0f, ad_b = 1.0f;
    int   idx_b = -1;
#pragma unroll
    for (int u = 0; u < 4; ++u)
    {
        const bool cand = el[u] & !(tq[u] > fmul(tq_b, 1.000003814697265625f));
        if (cand & !(tq[u] < fmul(tq_b, 0.999996185302734375f)) & (idx_b >= 0))
            key = key_min(key, beam_key(__fdiv_rn(a_b, ad_b), idx_b)); // near tie (rare): the displaced one keeps its claim
        tq_b  = cand ? tq[u] : tq_b;
        a_b   = cand ? a[u] : a_b;
        ad_b  = cand ? ad[u] : ad_b;
        idx_b = cand ? idx[u] : idx_b;
    }
    if (idx_b >= 0)
        key = key_min(key, beam_key(__fdiv_rn(a_b, ad_b), idx_b));
    if (lit[0] | lit[1] | lit[2] | lit[3])
    {
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (lit[u])
                key = key_min(key, beam_literal_key(segs, idx[u], ox, oy, dx, dy));
    }
    return key;
}

__device__ __forceinline__ float beam_meta_dist(const uint32_t q, const float rb)
{ // 12-bit distance field of an entry's meta word (ok_beam.hpp): 1/16 px, all ones = complete up to rb
    return q == kBeamDistFull ? rb : static_cast<float>(q) * (1.0f / kBeamDistScale);
}

// The rare ray a beam list cannot decide: uniform-grid walk from t_start with the best listed hit (best, min_t)
// as the incumbent.  Out of line on purpose: the walk's state would otherwise count against the registers of
// the hot loop around the call.
static __device__ __noinline__ int beam_walk_fallback(const uint8_t *blob, float ox, float oy, float dx, float dy, float range,
                                               float t_start, int best, float min_t)
{
    const TrackView tv = make_view(blob);
    RayWalk         w;
    if (!walk_begin(tv, w, ox, oy, dx, dy, range, t_start))
        return best;
    if (best >= 0)
    {
        w.best  = best;
        w.min_t = min_t; // the exact t of `best`
    }
    while (walk_unit(tv, w))
    {
    }
    return w.best;
}

// beam mode: AgentRec only (the per-thread scratch is static shared memory)
__host__ __device__ inline size_t beam_smem_bytes(int agents)
{
    return (static_cast<size_t>(agents) * sizeof(AgentRec) + 15u) / 16u * 16u;
}

// The beam kernel comes in two shapes, chosen by the host from the population size (ok_capi.cu, OK_BEAM_KERNEL):
//  * STAGED (kStaged = true): one 1,024-thread CTA per SM behind the track staged in shared memory with ONE TMA bulk
//    copy; about one large tile per CTA and wave (balanced tiling).  The throughput shape: a tile pays ~15 us of serial
//    latency (thread-per-agent phases, second ray pass) whatever its size, so tiles are made as large and as equal as the
//    shared memory and the SM count allow;
//  * UNSTAGED (kStaged = false): several 256-thread CTAs per SM, nothing staged -- the narrow phase reads four listed
//    segments per ray, not the whole track, so segments, centre line and the (rarely walked) grid come from the track's
//    blob in global memory through L1 / L2 (a fan's rays touch the same few 128-byte lines) and a CTA needs only its
//    agents' records.  The latency shape for small populations: no 75-140 KB staging copy, 8-warp barriers, and while
//    one CTA sits in a serial phase the SM's other CTAs cast rays.
#ifndef OK_BEAM_BLOCK
#define OK_BEAM_BLOCK 256
#endif
#ifndef OK_BEAM_MIN_CTAS
#define OK_BEAM_MIN_CTAS (1024 / OK_BEAM_BLOCK) // 64 registers per thread fill the register file
#endif
#ifndef OK_BEAM_TILE
#define OK_BEAM_TILE 64 // agents per tile of the unstaged beam kernel
#endif
constexpr int kBeamBlockStaged   = 1024;
constexpr int kBeamBlockUnstaged = OK_BEAM_BLOCK;
__host__ __device__ constexpr int beam_block(bool staged)
{
    return staged ? kBeamBlockStaged : kBeamBlockUnstaged;
}
// capacity of the CTA's queue of rays pass A leaves to pass B.  Tile-local ray indices are 16 bits, so a beam tile holds
// at most 65,535 rays (the host caps the batch); a full queue only costs speed (see pass A).
__host__ __device__ constexpr int beam_pend_cap(bool staged)
{
    return staged ? 8192 : 2048;
}
// static shared memory of the beam kernel besides the staged track and the agent records (host: batch sizing)
__host__ __device__ constexpr int beam_static_smem(bool staged)
{
    return beam_block(staged) * (16 + 8) + 2 * beam_pend_cap(staged) + 4 * (beam_pend_cap(staged) / 32) + 128;
}

__device__ __forceinline__ unsigned long long global_timer()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// trace record of one tile: {tile | smid << 32, t_start, t_phase1_done, t_passA_done, t_passB_done, t_phase4_done}
#ifdef OK_PRE_PROBE
#define OK_TRACE_ON(slot) ((slot) < 3)
#else
#define OK_TRACE_ON(slot) true
#endif
#define OK_TRACE(slot)                                                                                                 \
    do                                                                                                                 \
    {                                                                                                                  \
        if (OK_TRACE_ON(slot) && p.trace && tid == 0 && n_done < p.trace_tiles)                                       \
            p.trace[(static_cast<size_t>(blockIdx.x) * p.trace_tiles + n_done) * 6 + (slot)] = global_timer();         \
    } while (0)

// the second kernel argument of beam_step_kernel: the actor's parameters in the fused instantiation (kActor), nothing otherwise
struct NoActor
{
};
template <bool kActor> struct ActorArg
{
    using type = NoActor;
};
template <> struct ActorArg<true>
{
    using type = ActorParams;
};

// ---------------------------------------------------------------------------------------------
// the tile loop both step kernels run: fetch a tile, stage its track, phase 1, the rays, claim the next tile, phase 4
// ---------------------------------------------------------------------------------------------
// the first tile of a CTA is its own index: no trip to the global cursor before any work can start; and when the
// grid covers every tile (the balanced tiling's single wave, small populations) the cursor is never touched
#ifndef OK_SINGLE_WAVE
#define OK_SINGLE_WAVE 1
#endif
__device__ __forceinline__ bool single_wave_of(const StepParams &p)
{
    return OK_SINGLE_WAVE && p.n_tiles <= static_cast<int>(gridDim.x);
}

// tile `tile` and its track's record; a CTA's first tile (its block index, n_done == 0) comes with the record next to it
// (p.first)
__device__ __forceinline__ void fetch_tile(const StepParams &p, const int tile, const int n_done, Tile &tl, TrackRef &tr)
{
    if (p.first && n_done == 0)
    {
        tl = p.first[tile].tile;
        tr = p.first[tile].ref;
    }
    else
    {
        tl = p.tiles[tile];
        tr = p.tracks[tl.track];
    }
}

// (thread 0) the bulk copy of a track into shared memory: it runs under phase 1, which reads no staged data, and is
// awaited on `bar` before the rays
__device__ __forceinline__ void stage_track(uint8_t *blob, const uint8_t *gblob, const uint32_t bytes, uint64_t *bar)
{
    fence_proxy_async();
    mbar_expect_tx(bar, bytes);
    tma_bulk_g2s(blob, gblob, bytes, bar);
}

// ---- dynamic tile scheduler: tiles are batches of same-track agents, in agent order.  Thread 0 claims the CTA's next
// tile as LATE as possible (after the rays of this batch) and a barrier publishes it: claiming it at the start of the
// batch hides the atomic's latency but turns the schedule static -- measured 0.190 ms vs 0.150 ms per tick ----
__device__ __forceinline__ int claim_tile(const StepParams &p, const bool single_wave)
{
    return single_wave ? p.n_tiles : static_cast<int>(gridDim.x) + atomicAdd(p.sched, 1);
}

// =====================================================================================
// phase 4 -- four lanes (small batches) or one thread per agent: crash flag, centre-line search, reward, done
// =====================================================================================
template <int kBlock>
__device__ __forceinline__ void post_tile(const StepParams &p, const TrackView &tv, const AgentRec *recs, const Tile &tl, const int tid)
{
    const int lane = tid & 31, warp = tid >> 5;
    const int count = tl.count;
    if (count <= kBlock / 4)
    {
        const int  al    = tid >> 2;
        const bool valid = al < count;
        if ((warp << 3) < count) // warp-uniform: this warp has at least one agent
            agent_post<4>(p, tv, recs[valid ? al : 0], tl.begin + (valid ? al : 0), valid, lane);
    }
    else if (count <= kBlock / 2)
    { // the balanced tiling's large tiles (about 450 agents at the bench workload): two lanes per agent
        const int  al    = tid >> 1;
        const bool valid = al < count;
        if ((warp << 4) < count)
            agent_post<2>(p, tv, recs[valid ? al : 0], tl.begin + (valid ? al : 0), valid, lane);
    }
    else if ((warp << 5) < count)
    {
        const bool valid = tid < count;
        agent_post<1>(p, tv, recs[valid ? tid : 0], tl.begin + (valid ? tid : 0), valid, lane);
    }
}

// last CTA out re-arms the tile scheduler for the next launch on this stream
__device__ __forceinline__ void rearm_scheduler(const StepParams &p, const bool single_wave, const int tid)
{
    if (tid == 0 && !single_wave)
    {
        __threadfence();
        if (atomicAdd(p.sched + 1, 1) == static_cast<int>(gridDim.x) - 1)
        {
            p.sched[0] = 0;
            p.sched[1] = 0;
            __threadfence();
        }
    }
}

// The beam kernel.  kActor (ok_ppo_actor_step): the PPO racers' policy step runs as phase 0 of every tile -- the tile's
// agents choose their actions from last tick's observations (actor_agent) and the kinematics read them from the action
// buffers -- so that a rollout tick is ONE launch: at a few thousand agents a tick is latency, and two kernels pay it twice.
template <bool kStaged, bool kActor = false>
__global__ void __launch_bounds__(beam_block(kStaged), kStaged ? 1 : OK_BEAM_MIN_CTAS)
    beam_step_kernel(const StepParams p, const typename ActorArg<kActor>::type q)
{
    constexpr int kBlock   = beam_block(kStaged);
    constexpr int kPendCap = beam_pend_cap(kStaged);
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t         bar;
    __shared__ int                           s_tile, s_pool2, s_npend, s_adone, s_actdev;
    __shared__ int                           s_ready[kPendCap / 32]; // entries written, per 32-ray chunk of the queue
    __shared__ uint16_t                      s_pend[kPendCap]; // tile-local indices of the rays pass A left open

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int     R      = p.rays;

    uint8_t  *blob    = smem;
    AgentRec *recs    = reinterpret_cast<AgentRec *>(smem + (kStaged ? p.smem_blob_bytes : 0u));
    // per-thread ray parameters and result keys of the group a warp is working on
    __shared__ BeamHot                         s_hot;
    __shared__ unsigned long long              s_tns[3];
    __shared__ __align__(16) float4             s_wray[kBlock];
    __shared__ __align__(8) unsigned long long s_wkey[kBlock];

    if (kStaged && tid == 0)
        mbar_init(&bar, 1);
    __syncthreads();

    int      staged = -1;
    int      n_done = 0; // tiles this CTA has finished (trace slot)
    uint32_t phase  = 0;
    const float inv_R = 1.0f / static_cast<float>(R);
    const bool single_wave = single_wave_of(p);
    if (tid == 0)
        s_tile = static_cast<int>(blockIdx.x), s_actdev = 0;
    float  *s_actor_w   = nullptr; // kActor: the policy's weights, behind everything else in dynamic shared memory,
    float2 *s_actor_act = nullptr; //         and in front of them the tile's chosen actions (batch_agents of them)
    if constexpr (kActor)
    {
        s_actor_act = reinterpret_cast<float2 *>(smem + p.actor_smem_off);
        s_actor_w   = reinterpret_cast<float *>(s_actor_act + p.batch_agents);
        actor_stage_weights(q, R, s_actor_w, tid, kBlock); // (visible after the loop-top barrier)
    }

    for (;;)
    {
        __syncthreads(); // everyone is done with the previous batch and its track; s_tile is published
        const int tile = s_tile;
        if (tile >= p.n_tiles)
            break;
        if (p.trace && tid == 0 && n_done < p.trace_tiles)
        {
            unsigned smid;
            asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
            p.trace[(static_cast<size_t>(blockIdx.x) * p.trace_tiles + n_done) * 6] =
                static_cast<unsigned long long>(tile) | (static_cast<unsigned long long>(smid) << 32);
        }
        OK_TRACE(1);
        if (p.tile_ns && tid == 0) // thread 0: this tile's cost, for the host's tiling (ok_balance_schedule); kept in shared memory
            s_tns[0] = global_timer();

        Tile     tl;
        TrackRef tr;
        fetch_tile(p, tile, n_done, tl, tr);
        const uint8_t *gblob   = p.arena + tr.offset;
        const bool     restage = kStaged && tl.track != staged;
        if (restage && tid == 0)
            stage_track(blob, gblob, tr.bytes, &bar);
        BeamView bv;
        bv.valid = false;
        if (tr.has_beam)
            bv = make_beam_view(tr);
        const int       count    = tl.count;
        const int       n_rays   = count * R;

        // =====================================================================================
        // phase 1 -- one thread per agent: optional reset, kinematics, standstill (Environment.cpp:128-143)
        // =====================================================================================
        if constexpr (kActor)
        { // phase 0: kActorLanes lanes per agent, every warp whole (the logits meet by shuffles)
            for (int base = 0; base < count; base += kBlock / kActorLanes)
            {
                const int al = base + tid / kActorLanes;
                actor_agent(p, q, s_actor_w, tl.begin + (al < count ? al : 0), al < count, tid & (kActorLanes - 1), s_actor_act + (al < count ? al : 0));
            }
            __syncthreads(); // the chosen actions are in shared memory: the agents' own threads read them next
        }
        if (tid < count)
            recs[tid] = agent_pre(p, gblob, tr, bv, tl.begin + tid, n_done > 0 && s_actdev != 0, kActor ? s_actor_act + tid : nullptr);
        if (tid == 0)
        {
            s_pool2 = 0, s_npend = 0, s_adone = 0;
            s_hot.entries = bv.entries, s_hot.chunks = bv.chunks;
            s_hot.bin_scale = bv.bin_scale, s_hot.rb = bv.rb;
            s_hot.nb = bv.nb, s_hot.nb_mask = bv.nb - 1;
        }
        for (int i = tid; i < kPendCap / 32; i += kBlock)
            s_ready[i] = 0;
        OK_TRACE(3); // thread 0's own phase 1 is done; what follows is the wait for the staged track and for the other threads
        if (restage)
        {
            mbar_wait(&bar, phase);
            phase ^= 1u;
            staged = tl.track;
        }
        __syncthreads();
        OK_TRACE(2);
        if (p.tile_ns && tid == 0)
            s_tns[1] = global_timer();
        const uint8_t  *track    = kStaged ? blob : gblob; // where this tile reads its track from
        const TrackView tv       = make_view(track);
        const int64_t   ray_base = tl.begin * R; // global index of the batch's first ray
        // =================================================================================
        // beam phase.  PASS A -- warps pull groups of 32 consecutive rays (lane = ray): direction, ONE 16-byte table
        // entry (fetched a group ahead), the entry's four inline candidates tested in registers.  A ray whose hit
        // lies within the distance up to which those four are provably the only contenders (d1, ok_beam.hpp) is
        // finished on the spot with coalesced stores; the others (longer lists, hit beyond the list's completeness
        // distance, cell not covered) are queued.  PASS B -- the queued rays of the whole CTA, 32 at a time: the
        // rest of each list is dealt evenly over the warp's lanes (chunks of four, owner found by a shuffle binary
        // search), results meet in a 64-bit atomicMin key per ray; what even that cannot decide (~0.1 %) continues
        // with the uniform-grid walk from where its list stopped.
        // =================================================================================
        const int                n_groups = (n_rays + 31) >> 5;
        const unsigned long long key_none =
            (static_cast<unsigned long long>(__float_as_uint(p.sensor_range)) << 32) | 0x80000000ull;
        const float inf = __int_as_float(0x7f800000);
        float4             *w_ray = s_wray + (tid & ~31);
        unsigned long long *w_key = s_wkey + (tid & ~31);
        // tile-local ray q: agent, angle and its table entry
        // (`need_rest` = the caller reads ent.z, the rest's first chunk.  Pass A does not, and must not load it: left a
        // dead quarter of a 128-bit load, ptxas recycles that register for the packed active / cov flags RIGHT BEHIND the
        // load, and the write waits for the very load it was meant to run ahead of -- 12 % of all stall samples on that
        // one PRMT, ncu.  Two loads from the same sector, every destination live.)
        auto locate = [&](const int q, const bool valid, int &al, float &ang, bool &active, bool &cov, uint4 &ent,
                          const bool need_rest) {
            active = false, cov = false;
            al  = 0;
            ang = 0.0f;
            ent = make_uint4(0u, 0u, 0u, 0u);
            if (valid)
            {
                al                  = __float2int_rz((static_cast<float>(q) + 0.5f) * inv_R);
                OK_CHECK(q >= 0 && q < n_rays && al >= 0 && al < count && q - al * R >= 0 && q - al * R < R);
                const AgentRec &rec = recs[al];
                ang                 = fmul(OK_DEG2RAD, fadd(rec.rot, __ldg(p.ray_deg + (q - al * R))));
                active              = !(rec.flags & kFlagCrashed);
                if (active && rec.row >= 0 && fabsf(ang) < kBeamMaxAngle)
                {
                    const int bin = __float2int_rd(fmul(ang, ld_hot(s_hot.bin_scale))) & ld_hot(s_hot.nb_mask);
                    OK_CHECK(static_cast<uint32_t>(rec.row) < bv.n_rows);
                    const uint4 *ep = ld_hot(s_hot.entries) + static_cast<size_t>(rec.row) * ld_hot(s_hot.nb) + bin;
                    if (need_rest)
                        ent = __ldg(ep);
                    else
                    {
                        const uint2 c4 = __ldg(reinterpret_cast<const uint2 *>(ep));
                        ent            = make_uint4(c4.x, c4.y, 0u, __ldg(reinterpret_cast<const uint32_t *>(ep) + 3));
                    }
                    OK_CHECK(!need_rest || (ent.w >> 24) == 0 || ent.z + (ent.w >> 24) <= bv.n_chunks);
                    cov           = true;
                }
            }
        };
        // The full treatment of up to 32 queued rays (lane = ray `q`, `has` = the lane holds one): inline chunk on
        // the ray's own lane, the rest dealt across the warp, grid-walk fallback, outputs.  Warp-collective.
        auto process_full = [&](const int q, const bool has) {
            int   al;
            float ang;
            bool  active, cov;
            uint4 ent;
            locate(q, has, al, ang, active, cov, ent, true);
            float dx = 0.0f, dy = 0.0f;
            if (active)
                sincosf(ang, dy, dx); // cosf/sinf of CollisionChecker.cu:47-48
            const float rox = recs[al].ox, roy = recs[al].oy;
            w_ray[lane]     = make_float4(rox, roy, dx, dy);
            unsigned long long key0 = key_none;
            if (cov)
                key0 = beam_chunk_key(tv.seg, ent.x, ent.y, rox, roy, dx, dy, p.sensor_range, key_none, tv.n_seg);
            w_key[lane]        = key0;
            const uint32_t nch = cov ? (ent.w >> 24) : 0u; // chunks of the rest of the list
            uint32_t       inc = nch;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o)
                    inc += v;
            }
            const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
            const uint32_t first = ent.z - (inc - nch); // chunk j of the warp's rest chunks is chunk (first + j) of the table
            __syncwarp();
            // chunk j belongs to the lane `owner` whose prefix range contains j
            auto find_chunk = [&](uint32_t j, int &owner) -> uint32_t {
                owner = 0;
#pragma unroll
                for (int s2 = 16; s2 > 0; s2 >>= 1)
                {
                    const uint32_t v = __shfl_sync(0xffffffffu, inc, owner + s2 - 1);
                    if (v <= j)
                        owner += s2;
                }
                return __shfl_sync(0xffffffffu, first, owner) + j;
            };
            int   owner = 0;
            uint2 it    = make_uint2(0u, 0u);
            if (total > 0)
            {
                const uint32_t ch = find_chunk(lane, owner);
                if (static_cast<uint32_t>(lane) < total)
                {
                    OK_CHECK(ch < bv.n_chunks);
                    it = __ldg(ld_hot(s_hot.chunks) + ch);
                }
            }
            for (uint32_t base = 0; base < total; base += 32)
            {
                // the next round's candidates are requested before this round's are tested
                int   owner_n = 0;
                uint2 it_n    = make_uint2(0u, 0u);
                if (base + 32 < total)
                {
                    const uint32_t jn = base + 32 + lane;
                    const uint32_t ch = find_chunk(jn, owner_n);
                    if (jn < total)
                        it_n = __ldg(ld_hot(s_hot.chunks) + ch);
                }
                if (base + lane < total)
                {
                    const float4        ray = w_ray[owner];
                    unsigned long long *key = w_key + owner;
                    // the ray's incumbent exact t (already in the key) bounds what is worth a division
                    const float              m = __uint_as_float(reinterpret_cast<const uint32_t *>(key)[1]);
                    const unsigned long long k = beam_chunk_key(tv.seg, it.x, it.y, ray.x, ray.y, ray.z, ray.w, m, ~0ull, tv.n_seg);
                    if (k != ~0ull)
                        atomicMin(key, k);
                }
                owner = owner_n;
                it    = it_n;
            }
            __syncwarp();
            if (has)
            {
                const AgentRec          &rec   = recs[al];
                const unsigned long long key   = w_key[lane];
                int                      best  = static_cast<int>(0x7fffffffu - static_cast<uint32_t>(key));
                const float              min_t = __uint_as_float(static_cast<uint32_t>(key >> 32));
                const float              d_eff = beam_meta_dist(ent.w & 0xfffu, ld_hot(s_hot.rb));
                float t_known = min_t; // the key holds the exact t of `best`
                if (active && !(cov && min_t <= d_eff - kBeamSlack))
                { // undecided: everything nearer than d_eff - 1 is settled, the grid walk covers the rest
                    best = beam_walk_fallback(track, rec.ox, rec.oy, dx, dy, p.sensor_range,
                                              cov ? fmaxf(d_eff - 1.0f, 0.0f) : 0.0f, best, min_t);
                    t_known = 0.0f;
                    if (p.stats)
                        atomicAdd(p.stats + 2, 1ull);
                }
                const float sq = finish_ray<false>(p, tv.seg, rec, ray_base + q, dx, dy, best, t_known);
                // min_dist2 of CollisionChecker.cu:150,162-165: `if (sq < min) min = sq` skips NaN, and so does a
                // signed-int min over the bit patterns of values >= +0 (a NaN made here is 0x7fffffff)
                if (sq == sq)
                    smem_min(&recs[al].min_d2_bits, __float_as_int(sq));
            }
            __syncwarp(); // w_ray / w_key are reused by the next call
        };

        // ---------------------------------- pass A ----------------------------------
        // groups are dealt to the warps round-robin: every group costs the same here (the uneven part is queued), so
        // a shared cursor would only add an atomic and a shuffle per group
        constexpr int kWarps = kBlock / 32;
        int           g      = warp;
        int   al;
        float ang;
        bool  active, cov;
        uint4 ent;
        locate((g << 5) + lane, g < n_groups && (g << 5) + lane < n_rays, al, ang, active, cov, ent, false);
        while (g < n_groups)
        {
            const int g_next = g + kWarps;
            int   al_n;
            float ang_n;
            bool  active_n, cov_n;
            uint4 ent_n;
            locate((g_next << 5) + lane, g_next < n_groups && (g_next << 5) + lane < n_rays, al_n, ang_n, active_n, cov_n, ent_n, false);

            const int  q   = (g << 5) + lane;
            const bool has = q < n_rays;
            float dx = 0.0f, dy = 0.0f;
            if (active)
                sincosf(ang, dy, dx); // cosf/sinf of CollisionChecker.cu:47-48
            const AgentRec &rec = recs[al];
            unsigned long long key = key_none;
            if (cov)
                key = beam_chunk_key(tv.seg, ent.x, ent.y, rec.ox, rec.oy, dx, dy, p.sensor_range, key_none, tv.n_seg);
            const float min_t = __uint_as_float(static_cast<uint32_t>(key >> 32));
            // d1: up to there the inline four are the only contenders (= the list's completeness distance when it
            // has no rest).  The key holds the exact t of its segment, or the sensor range when nothing was hit.
            const float d1      = beam_meta_dist((ent.w >> 12) & 0xfffu, ld_hot(s_hot.rb));
            const bool  settled = cov && (min_t <= d1 - kBeamSlack);
            const bool  queue   = has && active && !settled;
            float       sq      = inf;
            if (has && !queue)
                sq = finish_ray<false>(p, tv.seg, rec, ray_base + q, dx, dy, static_cast<int>(0x7fffffffu - static_cast<uint32_t>(key)),
                                min_t);
            const unsigned qm = __ballot_sync(0xffffffffu, queue);
            if (qm)
            { // warp-aggregated append to the CTA's queue of undecided rays
                const int cnt  = __popc(qm);
                int       base = 0;
                if (lane == 0)
                    base = smem_add(&s_npend, cnt);
                base          = __shfl_sync(0xffffffffu, base, 0);
                const int pos = base + __popc(qm & ((1u << lane) - 1u));
                if (queue && pos < kPendCap)
                    s_pend[pos] = static_cast<uint16_t>(q);
                __syncwarp();
                if (lane == 0)
                { // publish: a 32-ray chunk of the queue may be taken by pass B as soon as all of it is written
                    const int lo = min(base, kPendCap), hi = min(base + cnt, kPendCap);
                    if (hi > lo)
                    {
                        __threadfence_block();
                        const int c0 = lo >> 5, c1 = (hi - 1) >> 5;
                        if (c0 == c1)
                            smem_add(&s_ready[c0], hi - lo);
                        else
                        {
                            smem_add(&s_ready[c0], ((c0 + 1) << 5) - lo);
                            smem_add(&s_ready[c1], hi - (c1 << 5));
                        }
                    }
                }
                if (base + cnt > kPendCap) // queue full (warp-uniform): these rays get the full treatment now
                    process_full(q, queue && pos >= kPendCap);
            }
            // min_dist2 of CollisionChecker.cu:150,162-165 over the rays finished here (see process_full)
            if ((R & 31) == 0)
            { // a warp's 32 rays belong to one agent: one warp-wide integer min (REDUX), one atomic per warp
                const int m = __reduce_min_sync(0xffffffffu, __float_as_int((sq == sq) ? sq : inf));
                if (has && lane == 0)
                    smem_min(&recs[al].min_d2_bits, m);
            }
            else if (has && !queue && sq == sq)
                smem_min(&recs[al].min_d2_bits, __float_as_int(sq));
            g = g_next, al = al_n, ang = ang_n, active = active_n, cov = cov_n, ent = ent_n;
        }
        // ---------------------------------- pass B ----------------------------------
        // No CTA barrier between the passes: a warp that runs out of groups starts on the queue right away.  It
        // claims the queue's next 32-ray chunk and waits until that chunk is completely written (s_ready) or every
        // warp has left pass A (s_adone), which makes the queue's length final.
        __syncwarp();
        if (lane == 0)
        {
            __threadfence_block();
            smem_add(&s_adone, 1);
        }
        for (;;)
        {
            int j = 0, size = 0;
            if (lane == 0)
            {
                j = smem_add(&s_pool2, 1);
                if (j < kPendCap / 32)
                    for (;;)
                    {
                        if (*reinterpret_cast<volatile int *>(&s_ready[j]) >= 32)
                        {
                            size = 32;
                            break;
                        }
                        if (*reinterpret_cast<volatile int *>(&s_adone) == kBlock / 32)
                        { // every append is complete and visible: what the chunk holds now is all it will ever hold
                            const int n = min(*reinterpret_cast<volatile int *>(&s_npend), kPendCap);
                            size        = max(0, min(32, n - (j << 5)));
                            break;
                        }
                        __nanosleep(100);
                    }
                __threadfence_block();
            }
            j    = __shfl_sync(0xffffffffu, j, 0);
            size = __shfl_sync(0xffffffffu, size, 0);
            if (size <= 0)
                break;
            const bool has = lane < size;
            process_full(has ? static_cast<int>(s_pend[(j << 5) + lane]) : 0, has);
        }
        // claim the next batch now: late enough to keep the schedule dynamic (see claim_tile), early enough
        // for the atomic's latency to hide behind the other warps' last groups and phase 4
        if (tid == 0)
        {
            s_tile = claim_tile(p, single_wave); // every thread read the old value before phase 1
            if (p.act_ready)
            { // have the staged actions arrived?  (Long since, normally; if not, the next tile reads the mapping.)
                uint32_t c;
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(c) : "l"(p.act_ready) : "memory");
                s_actdev = static_cast<int32_t>(c - p.act_ready_target) >= 0;
            }
        }
        __syncthreads();
        OK_TRACE(4);
        if (p.tile_ns && tid == 0)
            s_tns[2] = global_timer();
        if (p.tile_flag)
        { // (every thread's stores of this tile happened before the barrier above; the fence makes them visible device-wide
          // before the flag, PTX fences being cumulative)
            if (tid == 0)
            {
                __threadfence();
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.tile_flag + tile), "r"(p.flag_epoch) : "memory");
            }
        }
        else if (p.host_obs)
        { // End-to-end path (ok_step_host): this tile's observations are complete in device memory; they go to the pinned
          // HOST buffer now, as full 16-byte-per-lane stores through the mapping.  (The second ray pass finishes rays in
          // no particular order: storing them one by one reached the host as scattered 4-byte PCIe writes, 0.39 ms per
          // tick instead of 0.24.)  ok_step_host cuts the population into several tiles per CTA, so this copy drains
          // while the next tile is computed; trickling it through the next tile's ray loop instead measured the same.
            const float *src = p.obs + ray_base;
            float       *dst = p.host_obs + ray_base;
            if (((ray_base | n_rays) & 3) == 0)
                for (int i = tid; i < (n_rays >> 2); i += kBlock)
                    reinterpret_cast<float4 *>(dst)[i] = __ldcg(reinterpret_cast<const float4 *>(src) + i);
            else
                for (int i = tid; i < n_rays; i += kBlock)
                    dst[i] = __ldcg(src + i);
        }
        else if (p.host_obs_q16)
        { // the same flush at half width: eight observations per lane become one 16-byte store of 16-bit fixed point
            const float *src = p.obs + ray_base;
            uint16_t    *dst = p.host_obs_q16 + ray_base;
            if (((ray_base | n_rays) & 7) == 0)
                for (int i = tid; i < (n_rays >> 3); i += kBlock)
                {
                    const float4 a = __ldcg(reinterpret_cast<const float4 *>(src) + 2 * i);
                    const float4 b = __ldcg(reinterpret_cast<const float4 *>(src) + 2 * i + 1);
                    uint4        o;
                    o.x = obs_q16(a.x) | (obs_q16(a.y) << 16);
                    o.y = obs_q16(a.z) | (obs_q16(a.w) << 16);
                    o.z = obs_q16(b.x) | (obs_q16(b.y) << 16);
                    o.w = obs_q16(b.z) | (obs_q16(b.w) << 16);
                    reinterpret_cast<uint4 *>(dst)[i] = o;
                }
            else
                for (int i = tid; i < n_rays; i += kBlock)
                    dst[i] = static_cast<uint16_t>(obs_q16(__ldcg(src + i)));
        }
        if (p.stats && tid == 0)
        {
            atomicAdd(p.stats, static_cast<unsigned long long>(n_rays));
            atomicAdd(p.stats + 1, static_cast<unsigned long long>(s_npend));
        }
        post_tile<kBlock>(p, tv, recs, tl, tid);
        OK_TRACE(5); // thread 0's own phase 4 (the CTA-wide end is the next tile's start)
        if (p.tile_ns && tid == 0)
        {
            const unsigned long long t_end = global_timer(), rays_ns = s_tns[2] - s_tns[1];
            p.tile_ns[2 * tile]     = static_cast<uint32_t>(rays_ns);
            p.tile_ns[2 * tile + 1] = static_cast<uint32_t>((t_end - s_tns[0]) - rays_ns);
        }
        ++n_done;
    }
    rearm_scheduler(p, single_wave, tid);
}

// ---------------------------------------------------------------------------------------------
// the host's interface to the step kernels, one translation unit each (see the top of this file):
//   launch_step_<unit>      launches the unit's kernel on `grid` CTAs with `smem_bytes` of dynamic shared memory
//   arm_step_<unit>         sets the kernel's cudaFuncAttributeMaxDynamicSharedMemorySize to everything the device allows
//                           (an attribute of the function, not of the env); *max_dynamic = smem_optin less the kernel's
//                           static shared memory
//   occupancy_step_<unit>   CTAs per SM at `smem_bytes` of dynamic shared memory
//   violations_step_<unit>  the unit's self-check counter (OK_CHECKED builds; zero otherwise)
// ---------------------------------------------------------------------------------------------
cudaError_t launch_step_staged(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream);
cudaError_t arm_step_staged(int smem_optin, int *max_dynamic);
cudaError_t violations_step_staged(unsigned long long *count);

cudaError_t launch_step_unstaged(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream);
cudaError_t occupancy_step_unstaged(size_t smem_bytes, int *ctas_per_sm);
cudaError_t violations_step_unstaged(unsigned long long *count);

// the unstaged beam kernel with the policy step fused in
cudaError_t launch_step_actor(const StepParams &p, const ActorParams &q, int grid, size_t smem_bytes, cudaStream_t stream);
cudaError_t arm_step_actor(int smem_optin, int *max_dynamic);
cudaError_t violations_step_actor(unsigned long long *count);

// the grid / brute-force kernel (OK_RAYCAST_GRID, OK_RAYCAST_BRUTE), kGridBlock threads per CTA; its dynamic shared
// memory is the staged track and batch_smem_bytes
#ifndef OK_BLOCK
#define OK_BLOCK 1024
#endif
constexpr int kGridBlock = OK_BLOCK;
cudaError_t launch_step_grid(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream);
cudaError_t arm_step_grid(int smem_optin, int *max_dynamic);
cudaError_t violations_step_grid(unsigned long long *count);
__host__ __device__ inline size_t batch_smem_bytes(int agents, int rays)
{ // the grid kernel's batch scratch: AgentRec + per ray float2 direction
    return static_cast<size_t>(agents) * (sizeof(AgentRec) + 8u * static_cast<size_t>(rays));
}
// what arm_step_<unit> does for `kernel`
inline cudaError_t arm_dynamic_smem(const void *kernel, int smem_optin, int *max_dynamic)
{
    cudaFuncAttributes fa{};
    cudaError_t        rc = cudaFuncGetAttributes(&fa, kernel);
    if (rc != cudaSuccess)
        return rc;
    *max_dynamic = smem_optin - static_cast<int>(fa.sharedSizeBytes);
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, *max_dynamic);
}
} // namespace ok
