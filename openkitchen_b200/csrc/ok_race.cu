// ok_race.cu -- the race pass (OkRaces, include/openkitchen_b200.h): after a tick, the cars of a race see each other in the
// lidar and crash on contact.  A translation unit of its own, so the step kernels' units are untouched by it.
//
// Mapping: one warp per agent, 8 agents per CTA; nothing is staged.  The agent's race is at most 1,024 consecutive agents,
// read 32 at a time (lane k holds body base + k: one coalesced load per array), and the warps of a CTA share those lines in
// L1.  Each chunk of 32 bodies is culled by its lanes: __ballot_sync keeps the opponents whose centre lies within the
// lidar's reach of the origin, and the rays (lane = ray, looping for R > 32) then walk the kept bits in ascending order,
// with the body's centre broadcast by __shfl_sync from the lane that loaded it.  Ascending order and a strict `<` keep the
// lowest j among equal t.
//
// The pass reads only the agent's own crash flag and tick outputs and writes only its own outputs; the other agents'
// poses and tracks, which it reads, are not written by it.  So the results do not depend on the thread mapping.  The ray
// outputs come from the helpers the step kernels and the lidar query use for the unpack (lidar_origin, ray_hit, ray_rel,
// ray_obs).
#include "ok_race.cuh"

namespace ok
{

__global__ void __launch_bounds__(kRaceBlock) race_pass_kernel(const RaceParams p)
{
    const int     lane = threadIdx.x & 31;
    const int64_t a    = (static_cast<int64_t>(blockIdx.x) * kRaceBlock + threadIdx.x) >> 5;
    if (a >= p.n)
        return; // warp-uniform
    if (p.crashed[a])
    { // crashed before the pass: left as it is, apart from the contact flag, which every pass rewrites
        if (lane == 0)
            p.contact[a] = 0;
        return;
    }
    const int     R  = p.rays;
    const int64_t r0 = a / p.group * p.group;
    const int64_t r1 = min(r0 + p.group, p.n);
    OK_CHECK(r0 >= 0 && r1 <= p.n && r1 - r0 <= 1024);
    const float   xi = p.x[a], yi = p.y[a], rot = p.rot[a];
    const int32_t ti = p.track_id[a];
    OK_CHECK(ti >= 0 && ti < p.n_tracks);
    bool crash = false;

    // ---- contact: a disc of the same race and track that overlaps this one ----
    if (p.flags & OK_RACE_CONTACT)
    {
        const float lim = fmul(fadd(p.radius, p.radius), fadd(p.radius, p.radius));
        bool        hit = false;
        for (int64_t c = r0; c < r1; c += 32)
        {
            const int64_t j = c + lane;
            if (j < r1 && j != a && p.track_id[j] == ti)
            {
                const float ddx = fsub(xi, p.x[j]), ddy = fsub(yi, p.y[j]);
                hit |= fadd(fmul(ddx, ddx), fmul(ddy, ddy)) < lim;
            }
        }
        crash = __any_sync(0xffffffffu, hit);
    }

    // ---- sensing: the nearest body along each ray replaces a farther track hit ----
    if (p.flags & OK_RACE_SENSE)
    {
        float rs, rc;
        sincosf(fmul(OK_DEG2RAD, rot), rs, rc);
        const float2 o   = lidar_origin(xi, yi, rc, rs, p.sensor_offset);
        const float  rr  = fmul(p.radius, p.radius);
        bool         any = false;
        for (int r = lane; r - lane < R; r += 32)
        { // every lane runs every round: the ballots and shuffles below are warp-collective
            const bool has = r < R;
            float      dx = 0.0f, dy = 0.0f;
            if (has)
                sincosf(fmul(OK_DEG2RAD, fadd(rot, __ldg(p.ray_deg + r))), dy, dx); // exactly the tick's ray
            float   best_t = __int_as_float(0x7f800000);
            int32_t best_j = -1;
            for (int64_t c = r0; c < r1; c += 32)
            {
                const int64_t j  = c + lane;
                float         bx = 0.0f, by = 0.0f;
                bool          keep = false;
                if (j < r1 && j != a && p.track_id[j] == ti)
                {
                    bx                 = p.x[j], by = p.y[j];
                    const float wx = fsub(bx, o.x), wy = fsub(by, o.y);
                    keep               = fadd(fmul(wx, wx), fmul(wy, wy)) <= p.cull_d2; // false for NaN
                }
                for (unsigned m = __ballot_sync(0xffffffffu, keep); m; m &= m - 1u)
                {
                    const int   k  = __ffs(m) - 1;
                    const float xj = __shfl_sync(0xffffffffu, bx, k), yj = __shfl_sync(0xffffffffu, by, k);
                    const float wx = fsub(xj, o.x), wy = fsub(yj, o.y);
                    const float b  = fadd(fmul(wx, dx), fmul(wy, dy));
                    const float cc = fsub(fadd(fmul(wx, wx), fmul(wy, wy)), rr);
                    float       t;
                    if (cc <= 0.0f)
                        t = 0.0f;
                    else
                    {
                        const float q = fsub(fmul(b, b), cc);
                        if (!(b > 0.0f && q >= 0.0f))
                            continue;
                        t = fmaxf(fsub(b, __fsqrt_rn(q)), 0.0f);
                    }
                    if (t <= p.sensor_range && t < best_t)
                        best_t = t, best_j = static_cast<int32_t>(c + k);
                }
            }
            if (!has)
                continue;
            const int64_t gi = a * R + r;
            const bool    rep = best_j >= 0 && best_t < p.hit_t[gi];
            if (rep)
            {
                OK_CHECK(best_j >= r0 && best_j < r1 && best_j != a);
                const float2 hit = ray_hit(o.x, o.y, dx, dy, best_t);
                float        sq;
                const float2 rel = ray_rel(o.x, o.y, rc, rs, hit, sq);
                p.hit_t[gi]                                 = best_t;
                reinterpret_cast<float2 *>(p.hit_abs)[gi] = hit;
                reinterpret_cast<float2 *>(p.hit_rel)[gi] = rel;
                p.hit_seg[gi]                               = -1;
                p.obs[gi]                                   = ray_obs(sq, p.sensor_range);
            }
            p.hit_car[gi] = rep ? best_j : -1;
            any |= rep;
        }
        if (__any_sync(0xffffffffu, any))
        { // min_dist2 of the unpack (CollisionChecker.cu:150,162-165) over all R rays, replaced ones included: `sq < min` skips NaN
            float m = fmul(p.sensor_range, p.sensor_range);
            for (int r = lane; r < R; r += 32)
            {
                const float2 rel = reinterpret_cast<const float2 *>(p.hit_rel)[a * R + r]; // this lane's own store, if any
                const float  sq  = fadd(fmul(rel.x, rel.x), fmul(rel.y, rel.y));
                if (sq < m)
                    m = sq;
            }
            for (int s = 16; s > 0; s >>= 1)
                m = fminf(m, __shfl_xor_sync(0xffffffffu, m, s)); // no NaN left: the order does not matter
            if (lane == 0)
                p.min_dist2[a] = m;
            crash |= m < p.collision_dist2; // CollisionChecker.cu:167-171
        }
    }

    if (lane == 0)
    {
        p.contact[a] = crash;
        if (crash)
            p.crashed[a] = 1, p.done[a] = 1;
    }
}

cudaError_t launch_race_pass(const RaceParams &p, cudaStream_t stream)
{
    constexpr int per_cta = kRaceBlock / 32;
    const int64_t blocks  = (p.n + per_cta - 1) / per_cta;
    race_pass_kernel<<<static_cast<unsigned>(blocks), kRaceBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t violations_race(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
