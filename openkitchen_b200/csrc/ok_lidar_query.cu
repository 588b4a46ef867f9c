// ok_lidar_query.cu -- lidar scans at arbitrary poses (ok_lidar_query): the ray cast of the step kernels for poses that are
// not the state of an agent, in a translation unit of its own (see the top of ok_step.cuh for why every kernel that calls
// the out-of-line beam helpers gets one).
//
// Mapping: nothing is staged.  Segments, grid and beam tables come through L1 / L2 from the global arena, as in the
// unstaged beam kernel.  A thread holds one (pose, ray) pair and a warp 32 consecutive pairs, so the rays of a fan share
// a table row and the stores coalesce.  A pose's rays never leave their CTA: for R <= 32 a warp holds floor(32 / R) whole
// poses; for R > 32 a pose takes consecutive warps of one CTA (and a thread loops when R > kLidarBlock).  min_dist2 and
// the crash flag are reduced in registers and shared memory and stored once per pose.
//
// Every output is bit for bit what ok_cast_rays writes for an agent at the same pose with no crash flag set.  The lidar
// origin, the beam decision (beam_settles, beam_walk_rest), the table's meta word and result key, and the ray outputs
// (ray_hit, ray_rel, ray_obs) are the step kernels' own helpers.  This kernel's own parts are its dealing loop and its
// per-pose reductions: the rest chunks of a warp's undecided rays are dealt across its lanes as process_full deals them,
// but the rays stay where they are (the beam kernel first gathers them into full warps); tests/test_gpu_lidar_query.py
// checks those parts against ok_cast_rays bit for bit.
#include "ok_lidar_query.cuh"
#include "ok_step.cuh"

namespace ok
{

// per pose, filled by one thread before the rays
struct LidarPose
{
    float   ox, oy, rc, rs; // lidar origin, cos / sin of the heading
    float   rot;            // heading (degrees)
    int32_t track;          // clamped track index
    int32_t row;            // beam-table row of the origin's cell, -1 = not covered (beam mode only)
    int32_t pad;
};
static_assert(sizeof(LidarPose) == 32, "LidarPose layout");

__global__ void __launch_bounds__(kLidarBlock, kLidarMinCtas) lidar_query_kernel(const LidarQueryParams q)
{
    __shared__ LidarPose s_pose[kLidarBlock];
    __shared__ int       s_min[kLidarBlock]; // running min of the squared hit norms (as int: all values are >= +0)
    // per lane, while its warp deals out the rest chunks of its undecided rays (process_full): the ray, its result key, and
    // where its chunks and segments are (the poses of one warp may sit on different tracks)
    __shared__ __align__(16) float4             s_wray[kLidarBlock];
    __shared__ __align__(8) unsigned long long s_wkey[kLidarBlock];
    __shared__ const uint2                     *s_wchk[kLidarBlock];
    __shared__ const float4                    *s_wseg[kLidarBlock];
    __shared__ int                              s_wnseg[kLidarBlock];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int R = q.rays, ppc = lidar_poses_per_cta(R);
    // this thread's pose within the CTA, its first ray and the stride to its next one
    int  local, sub, stride;
    bool mine;
    if (R <= 32)
    {
        const int ppw = 32 / R;
        local = warp * ppw + lane / R, sub = lane % R, stride = R;
        mine  = lane < ppw * R;
        local = mine ? local : 0;
    }
    else
    {
        const int tpp = lidar_threads_per_pose(R);
        local = tid / tpp, sub = tid % tpp, stride = tpp;
        mine  = local < ppc;
        local = mine ? local : 0;
    }
    const int64_t pose0 = static_cast<int64_t>(blockIdx.x) * ppc;

    // ---- one thread per pose: track, lidar origin (agent_pre, CollisionChecker.cu:121-124), beam row ----
    if (tid < ppc && pose0 + tid < q.n)
    {
        const int64_t k = pose0 + tid;
        int32_t       t = q.track ? q.track[k] : 0;
        t               = min(max(t, 0), q.n_tracks - 1);
        const float x = q.x[k], y = q.y[k], rot = q.rot[k];
        float       rs, rc;
        sincosf(fmul(OK_DEG2RAD, rot), rs, rc);
        LidarPose    ps;
        const float2 o = lidar_origin(x, y, rc, rs, q.sensor_offset);
        ps.ox = o.x, ps.oy = o.y;
        ps.rc = rc, ps.rs = rs, ps.rot = rot, ps.track = t, ps.pad = 0;
        const TrackRef &tr = q.tracks[t];
        BeamView        bv;
        bv.valid = false;
        if (q.raycast_mode == OK_RAYCAST_BEAM && tr.has_beam)
            bv = make_beam_view(tr);
        ps.row      = beam_row(bv, ps.ox, ps.oy);
        s_pose[tid] = ps;
        s_min[tid]  = __float_as_int(fmul(q.sensor_range, q.sensor_range));
    }
    __syncthreads();

    // ---- one thread per ray; every thread runs the same number of rounds (the beam mode's dealing is warp-collective) ----
    const int64_t   k       = pose0 + local;
    const bool      pose_ok = mine && k < q.n;
    const LidarPose ps      = s_pose[local];
    OK_CHECK(!pose_ok || (ps.track >= 0 && ps.track < q.n_tracks));
    const TrackRef &tr   = q.tracks[pose_ok ? ps.track : 0];
    const uint8_t  *blob = q.arena + tr.offset;
    const TrackView tv   = make_view(blob);
    BeamView        bv;
    bv.valid = false;
    if (q.raycast_mode == OK_RAYCAST_BEAM && tr.has_beam)
        bv = make_beam_view(tr);
    const unsigned long long key_none = (static_cast<unsigned long long>(__float_as_uint(q.sensor_range)) << 32) | 0x80000000ull;
    float                    m        = __int_as_float(0x7f800000);
    const int                rounds   = (R + stride - 1) / stride;
    for (int rd = 0; rd < rounds; ++rd)
    {
        const int r   = sub + rd * stride;
        const bool has = pose_ok && r < R;
        float      ang = 0.0f, dx = 0.0f, dy = 0.0f;
        if (has)
        {
            ang = fmul(OK_DEG2RAD, fadd(ps.rot, __ldg(q.ray_deg + r)));
            sincosf(ang, dy, dx); // cosf/sinf of CollisionChecker.cu:47-48
        }
        int   seg     = -1;
        float t_known = 0.0f; // the winner's exact t when a beam key holds it (0 = recompute it)
        if (q.raycast_mode == OK_RAYCAST_BEAM)
        { // the beam kernel's decision: pass A's inline chunk, process_full's rest chunks, the grid walk
            const bool         cov = has && ps.row >= 0 && fabsf(ang) < kBeamMaxAngle;
            uint4              ent = make_uint4(0u, 0u, 0u, 0u);
            unsigned long long key = key_none;
            if (cov)
            {
                const int bin = __float2int_rd(fmul(ang, bv.bin_scale)) & (bv.nb - 1);
                OK_CHECK(static_cast<uint32_t>(ps.row) < bv.n_rows);
                ent = __ldg(bv.entries + static_cast<size_t>(ps.row) * bv.nb + bin);
                OK_CHECK(beam_meta_rest(ent.w) == 0 || ent.z + beam_meta_rest(ent.w) <= bv.n_chunks);
                key = beam_chunk_key(tv.seg, ent.x, ent.y, ps.ox, ps.oy, dx, dy, q.sensor_range, key_none, tv.n_seg);
            }
            const bool     undecided = has && !beam_settles(cov, key, beam_meta_d1(ent.w, bv.rb));
            const uint32_t nch       = (undecided && cov) ? beam_meta_rest(ent.w) : 0u; // chunks of the rest of the list
            if (__any_sync(0xffffffffu, nch > 0))
            { // process_full's dealing: chunk j of the warp's rest chunks goes to lane j % 32, results meet in a shared key
                const uint32_t inc   = warp_inclusive_scan(nch, lane);
                const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
                s_wray[tid]  = make_float4(ps.ox, ps.oy, dx, dy);
                s_wkey[tid]  = key;
                s_wchk[tid]  = nch > 0 ? bv.chunks + ent.z - (inc - nch) : nullptr; // chunk j of the warp is s_wchk[owner][j]
                s_wseg[tid]  = tv.seg;
                s_wnseg[tid] = tv.n_seg;
                __syncwarp();
                const int w0 = tid & ~31;
                for (uint32_t base = 0; base < total; base += 32)
                {
                    const uint32_t j     = base + lane;
                    const int      owner = w0 + chunk_owner(inc, j);
                    if (j < total)
                    {
                        const uint2               it = __ldg(s_wchk[owner] + j);
                        const float4              ry = s_wray[owner];
                        unsigned long long *const kp = s_wkey + owner;
                        // the ray's incumbent exact t (already in the key) bounds what is worth a division
                        const unsigned long long kc =
                            beam_chunk_key(s_wseg[owner], it.x, it.y, ry.x, ry.y, ry.z, ry.w, beam_key_t_at(kp), ~0ull, s_wnseg[owner]);
                        if (kc != ~0ull)
                            atomicMin(kp, kc);
                    }
                }
                __syncwarp();
                key = s_wkey[tid];
                __syncwarp(); // the next round rewrites the warp's slots
            }
            const float d_eff = beam_meta_d(ent.w, bv.rb);
            seg               = beam_key_seg(key);
            t_known           = beam_key_t(key); // the key holds the exact t of its segment
            if (undecided && !beam_settles(cov, key, d_eff))
            {
                seg     = beam_walk_rest(blob, ps.ox, ps.oy, dx, dy, q.sensor_range, cov, d_eff, key);
                t_known = 0.0f;
            }
        }
        else if (has && q.raycast_mode == OK_RAYCAST_GRID)
        {
            RayWalk w;
            if (walk_begin(tv, w, ps.ox, ps.oy, dx, dy, q.sensor_range))
            {
                while (walk_unit(tv, w))
                {
                }
                seg = w.best;
            }
        }
        else if (has)
            seg = cast_ray_brute(tv, ps.ox, ps.oy, dx, dy, q.sensor_range);
        if (!has)
            continue; // (uniform loop: nothing below is warp-collective)
        OK_CHECK(seg >= -1 && seg < tv.n_seg);
        const int64_t gi = k * R + r;
        // finish_ray's outputs, each only if asked for
        const float  t   = seg >= 0 ? (t_known != 0.0f ? t_known : exact_t(tv.seg[seg], ps.ox, ps.oy, dx, dy)) : q.sensor_range;
        const float2 hit = ray_hit(ps.ox, ps.oy, dx, dy, t);
        float        sq;
        const float2 rel = ray_rel(ps.ox, ps.oy, ps.rc, ps.rs, hit, sq);
        if (q.hit_seg)
            q.hit_seg[gi] = seg;
        if (q.hit_t)
            q.hit_t[gi] = t;
        if (q.hit_abs)
            reinterpret_cast<float2 *>(q.hit_abs)[gi] = hit;
        if (q.hit_rel)
            reinterpret_cast<float2 *>(q.hit_rel)[gi] = rel;
        if (q.obs)
            q.obs[gi] = ray_obs(sq, q.sensor_range);
        // min_dist2 of CollisionChecker.cu:150,162-165: `if (sq < min) min = sq` skips NaN
        if (sq == sq)
            m = fminf(m, sq);
    }
    if (pose_ok)
        smem_min(&s_min[local], __float_as_int(m));
    __syncthreads();

    // ---- one thread per pose: min_dist2 and the strict crash test of CollisionChecker.cu:167-171 ----
    if (tid < ppc && pose0 + tid < q.n)
    {
        const float min_d2 = __int_as_float(s_min[tid]);
        if (q.min_dist2)
            q.min_dist2[pose0 + tid] = min_d2;
        if (q.crashed)
            q.crashed[pose0 + tid] = min_d2 < q.collision_dist2;
    }
}

cudaError_t launch_lidar_query(const LidarQueryParams &q, cudaStream_t stream)
{
    const int     ppc    = lidar_poses_per_cta(q.rays);
    const int64_t blocks = (q.n + ppc - 1) / ppc;
    lidar_query_kernel<<<static_cast<unsigned>(blocks), kLidarBlock, 0, stream>>>(q);
    return cudaGetLastError();
}

cudaError_t violations_lidar_query(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
