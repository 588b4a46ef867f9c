// ok_step_grid.cuh -- the grid / brute-force step kernel's body (OK_RAYCAST_GRID, OK_RAYCAST_BRUTE): per-ray directions in
// shared memory, rays pulled one by one from a CTA-wide pool and walked through the uniform grid (or tested against every
// segment, the reference's loop), then one thread per ray for the outputs.  Its kernel, grid_step_kernel<StepVariant>, is
// instantiated once per variant, each in a translation unit of its own (ok_step_grid.cu, ok_step_grid_drawn.cu,
// ok_step_grid_laps.cu).
#pragma once

#include "ok_step.cuh"

namespace ok
{
#ifndef OK_UNITS
#define OK_UNITS 4
#endif
constexpr int kUnitsPerRefill = OK_UNITS; // units of work a lane does between two looks at the pool

template <StepVariant kVariant>
__device__ __forceinline__ void grid_tick(const StepParams &p)
{
    constexpr bool kDraws = kVariant == StepVariant::drawn;
    constexpr bool kLaps  = kVariant == StepVariant::laps;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint16_t                      s_order[1024]; // pool order of the rays (p.ray_order)
    __shared__ __align__(8) uint64_t         bar;
    __shared__ int                           s_tile, s_pool;

    const int tid = threadIdx.x, lane = tid & 31;
    const int     R      = p.rays;

    uint8_t  *blob    = smem;
    AgentRec *recs    = reinterpret_cast<AgentRec *>(smem + p.smem_blob_bytes);
    float2   *dirs    = reinterpret_cast<float2 *>(recs + p.batch_agents);

    if (tid == 0)
        mbar_init(&bar, 1);
    for (int i = tid; i < R; i += kGridBlock)
        s_order[i] = p.ray_order[i];
    __syncthreads();

    int      staged = -1;
    int      n_done = 0; // tiles this CTA has finished
    uint32_t phase  = 0;
    const float inv_R = 1.0f / static_cast<float>(R);
    const bool single_wave = single_wave_of(p);
    if (tid == 0)
        s_tile = static_cast<int>(blockIdx.x);

    for (;;)
    {
        __syncthreads(); // everyone is done with the previous batch and its track; s_tile is published
        const int tile = s_tile;
        if (tile >= p.n_tiles)
            break;

        Tile     tl;
        TrackRef tr;
        fetch_tile(p, tile, n_done, tl, tr);
        const uint8_t *gblob   = p.arena + tr.offset;
        const bool     restage = tl.track != staged;
        if (restage && tid == 0)
            stage_track(blob, gblob, tr.bytes, &bar);
        BeamView bv; // no beam lists in this kernel
        bv.valid = false;
        const int       count    = tl.count;
        const int       n_rays   = count * R;
        const float     inv_cnt  = 1.0f / static_cast<float>(count);

        // =====================================================================================
        // phase 1 -- one thread per agent: optional reset, kinematics, standstill (Environment.cpp:128-143)
        // =====================================================================================
        if (tid < count)
            recs[tid] = agent_pre<kDraws, kLaps>(p, gblob, tr, bv, tl.begin + tid);
        if (tid == 0)
            s_pool = 0;
        if (restage)
        {
            mbar_wait(&bar, phase);
            phase ^= 1u;
            staged = tl.track;
        }
        __syncthreads();
        const TrackView tv       = make_view(blob);
        const int64_t   ray_base = tl.begin * R; // global index of the batch's first ray

        // =====================================================================================
        // phase 1b -- one thread per ray: direction (cosf/sinf of CollisionChecker.cu:47-48)
        // =====================================================================================
        for (int q = tid; q < n_rays; q += kGridBlock)
        {
            const int al = __float2int_rz((static_cast<float>(q) + 0.5f) * inv_R);
            const int r  = q - al * R;
            float     s, c;
            sincosf(fmul(OK_DEG2RAD, fadd(recs[al].rot, p.ray_deg[r])), s, c);
            dirs[q] = make_float2(c, s);
        }
        __syncthreads();

        // =====================================================================================
        // phase 2 -- the casts (grid / brute modes).  Rays are pulled from a CTA-wide pool, every lane on its own
        // (one shared-memory atomic per ray), so the long rays of the heavy tail do not hold 31 lanes hostage.
        // The pool is ordered ray-major with the fan's centre rays first (p.ray_order): those are the long ones.
        // =====================================================================================
        if (p.raycast_mode == OK_RAYCAST_GRID)
        {
            // No warp-level primitive in this loop on purpose: every lane fetches and retires on its own
            // (one shared-memory atomic per ray), so nothing depends on the lanes of a warp being converged
            // inside this heavily divergent code.  (A vote-based, warp-aggregated refill with the unit loop
            // unrolled hung on sm_100a / CUDA 12.9: lanes left the loop on different trips.)
            RayWalk w;
            int     mine = -1;   // batch-local ray (agent * R + ray) this lane is working on, -1 = idle
            bool    more = true; // the pool may still hold rays
            for (;;)
            {
                if (mine < 0)
                {
                    if (!more)
                        break;
                    const int q = atomicAdd(&s_pool, 1);
                    if (q >= n_rays)
                        more = false;
                    else
                    {
                        // pool order -> (agent, ray): ray-major, centre rays first
                        const int rank = __float2int_rz((static_cast<float>(q) + 0.5f) * inv_cnt);
                        const int al   = q - rank * count;
                        const int r    = s_order[rank];
                        const int slot = al * R + r;
                        const AgentRec &rec = recs[al];
                        // a crashed agent's rays are inactive: the kernel leaves their stale hits alone
                        // (CollisionChecker.cu:44)
                        if (!(rec.flags & kFlagCrashed))
                        {
                            const float2 d = dirs[slot];
                            if (walk_begin(tv, w, rec.ox, rec.oy, d.x, d.y, p.sensor_range))
                                mine = slot;
                            else
                                p.hit_seg[ray_base + slot] = -1;
                        }
                    }
                }
#pragma unroll 1
                for (int u = 0; u < kUnitsPerRefill; ++u)
                {
                    if (mine >= 0)
                    {
                        if (!walk_unit(tv, w))
                        { // only the index travels: phase 3 recomputes the winner's exact t
                            p.hit_seg[ray_base + mine] = w.best;
                            mine                       = -1;
                        }
                    }
                }
            }
        }
        else
        { // OK_RAYCAST_BRUTE: every segment in ascending order, the reference's own loop
            for (int q = tid; q < n_rays; q += kGridBlock)
            {
                const int       al  = __float2int_rz((static_cast<float>(q) + 0.5f) * inv_R);
                const AgentRec &rec = recs[al];
                if (rec.flags & kFlagCrashed)
                    continue;
                const float2 d          = dirs[q];
                p.hit_seg[ray_base + q] = cast_ray_brute(tv, rec.ox, rec.oy, d.x, d.y, p.sensor_range);
            }
        }
        __syncthreads();

        // =====================================================================================
        // phase 3 -- one thread per ray: hit point, unpack (CollisionChecker.cu:68-69,152-165), outputs
        // =====================================================================================
        for (int q0 = 0; q0 < n_rays; q0 += kGridBlock)
        {
            const int  q   = q0 + tid;
            const bool has = q < n_rays;
            float      sq  = __int_as_float(0x7f800000);
            int        al  = 0;
            if (has)
            {
                al                  = __float2int_rz((static_cast<float>(q) + 0.5f) * inv_R);
                const AgentRec &rec = recs[al];
                const int64_t   gi  = ray_base + q;
                const float2    d   = dirs[q];
                // (p.hit_seg: written in phase 2 by whichever lane cast this ray; finish_ray reads neither it nor d for
                // a crashed agent)
                sq = finish_ray<true>(p, tv.seg, rec, gi, d.x, d.y, p.hit_seg[gi]);
            }
            // min_dist2 of CollisionChecker.cu:150,162-165: `if (sq < min) min = sq` skips NaN, and so
            // does a signed-int min over the bit patterns of values >= +0 (a NaN made here is 0x7fffffff)
            if ((R & 31) == 0)
            { // a warp's 32 rays belong to one agent: reduce in registers, one atomic per warp
                float m = (sq == sq) ? sq : __int_as_float(0x7f800000);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
                    m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
                if (has && lane == 0)
                    atomicMin(&recs[al].min_d2_bits, __float_as_int(m));
            }
            else if (has && sq == sq)
                atomicMin(&recs[al].min_d2_bits, __float_as_int(sq));
        }
        __syncthreads();
        if (tid == 0)
            s_tile = claim_tile(p, single_wave); // every thread read the old value long ago; visible after the loop-top barrier
        post_tile<kGridBlock, kLaps>(p, tv, recs, tl, tid);
        ++n_done;
    }
    rearm_scheduler(p, single_wave, tid);
}

template <StepVariant kVariant> __global__ void __launch_bounds__(kGridBlock, 1) grid_step_kernel(const StepParams p)
{
    grid_tick<kVariant>(p);
}

template <StepVariant kVariant>
cudaError_t launch_grid_step(const StepParams &p, const ActorParams *, int grid, size_t smem_bytes, cudaStream_t stream)
{
    grid_step_kernel<kVariant><<<grid, kGridBlock, smem_bytes, stream>>>(p);
    return cudaGetLastError();
}
// the record of a grid unit; static, so that it takes the address of its own unit's unit_violations
template <StepVariant kVariant> static StepUnit grid_step_unit()
{
    return {launch_grid_step<kVariant>, reinterpret_cast<const void *>(grid_step_kernel<kVariant>), unit_violations};
}
} // namespace ok
