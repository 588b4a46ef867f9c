// ok_kernels.cuh -- sm_100a kernels of the batched step loop.
//
// One fused kernel per tick (ok::step_kernel) replaces, per agent, the whole of
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
//   * the rays: kBeam = true reads precomputed candidate lists (ok_beam.hpp) -- warps pull groups of 32 rays, a ray's
//     first chunk of candidates is tested by its own lane, the rest is dealt evenly over the warp, results meet in a
//     64-bit atomicMin key per ray; kBeam = false walks a uniform grid ray by ray from a CTA-wide pool (or tests every
//     segment: the reference's loop);
//   * state is structure-of-arrays; per-ray outputs are written coalesced (lane = ray).
// The path is warp-issue bound, not HBM bound, and is not a contraction: no tensor cores (DESIGN.md section 4).
#pragma once

#include "ok_beam.hpp"
#include "ok_math.cuh"
#include "ok_schedule.hpp"
#include "ok_track.hpp"

#include <cfloat>

namespace ok
{

// Self-checks (the pool's compute-sanitizer is closed, profiles/r2_sanitizer_closed.log): a build with -DOK_CHECKED=1
// counts every index that leaves its array instead of using it (tools/checked_build.sh runs the parity suite on it and
// requires the count to stay zero).  Compiled out of the product build.
#ifndef OK_CHECKED
#define OK_CHECKED 0
#endif
static __device__ unsigned long long g_violations = 0; // one per translation unit (ok_capi.cu, ok_step_unstaged.cu)
#if OK_CHECKED
#define OK_CHECK(cond)                                                                                                 \
    do                                                                                                                 \
    {                                                                                                                  \
        if (!(cond))                                                                                                   \
            atomicAdd(&g_violations, 1ull);                                                                            \
    } while (0)
#else
#define OK_CHECK(cond) ((void)0)
#endif

struct TrackRef
{
    uint64_t offset;      // byte offset of the blob in the arena (128-byte aligned)
    uint32_t bytes;       // blob_bytes
    uint32_t has_beam;    // the track has a beam table
    uint64_t beam_offset; // device address of its beam table (ok_beam.hpp), its own allocation
    // the table's header, copied here by the host: a tile start reads this 64-byte record (L2 resident, 23 of them)
    // instead of chasing the header at the front of a multi-hundred-MB table that no cache holds
    float    bx0, by0, binv_h, bbin_scale, brb;
    int32_t  bnx, bny, bnb;
    uint32_t boff_rows, boff_entries, boff_items, bn_rows, bn_chunks;
    uint32_t seg_bytes;   // header + segments (+ the null segment) = the blob's prefix up to the grid words; no kernel reads it
    // what a crashed agent's auto-reset needs of the blob's header (phase 1 reads the GLOBAL blob: one trip to memory less)
    int32_t  n_points;
    uint32_t off_points, off_headings, pad;
};
static_assert(sizeof(TrackRef) == 96, "TrackRef layout");
// a CTA's FIRST tile with its track record next to it: one trip to memory instead of two before any work can start
struct FirstTile
{
    Tile     tile;
    TrackRef ref;
    uint32_t pad[4];
};
static_assert(sizeof(FirstTile) == 128, "FirstTile layout");

struct StepParams
{
    // agent state, structure of arrays
    float    *x, *y, *rot, *speed, *accel, *act_thr, *act_steer;
    uint8_t  *crashed, *timed_out, *done;
    uint32_t *ss_ctr;
    float    *ss_x, *ss_y;
    int32_t  *track_id;
    float    *hit_abs, *hit_rel, *obs, *hit_t, *min_dist2;
    int32_t  *hit_seg, *nearest, *prev;
    float    *reward, *fitness;
    int32_t  *reset_pt;
    float    *start_x, *start_y;
    // static inputs
    const float   *ray_deg;
    const uint8_t *arena;
    const TrackRef *tracks;
    const Tile    *tiles;
    const FirstTile *first; // nullable: tiles[b] and its track record for b < gridDim.x
    int64_t        n_agents;
    int32_t        n_tiles;
    int32_t        rays;
    int32_t        batch_agents;    // agents per tile (shared-memory scratch is sized for this many)
    uint32_t       smem_blob_bytes; // offset of the batch scratch behind the staged track
    uint32_t       actor_smem_off;  // kActor: offset of the policy weights in dynamic shared memory
    const uint16_t *ray_order;      // ray indices sorted by |angle|: pool order, long (central) rays first
    int32_t       *sched;           // {next tile, CTAs finished}: dynamic tile scheduler
    unsigned long long *stats;      // nullable: {rays cast, rays queued for pass B, rays sent to the grid walk} (beam kernel)
    unsigned long long *trace;      // nullable: per CTA and tile, globaltimer at the phase boundaries (profiling aid, beam kernel)
    int32_t             trace_tiles; // tiles per CTA the trace buffer has room for
    uint32_t           *tile_ns;     // nullable (beam kernel): per tile {ns in the ray phase, ns in the rest of the tile}: feedback for the host's tiling
    // this launch
    const float *ext_thr, *ext_steer; // nullable: actions supplied by the caller
    int32_t      ext_host;            // (host side only) they are pinned HOST arrays read through the mapping
    int32_t      action_source;       // 0 stored/ext, 1 philox
    uint32_t     seed;
    uint64_t     step;
    uint64_t     id_base;             // OkConfig::agent_id_base: global id of agent 0 (Philox counter)
    int32_t      do_move;             // 0: ok_cast_rays
    // optional mirrors in PINNED HOST memory (ok_step_host): the kernel stores results over PCIe as they are
    // produced, so the device->host transfer overlaps the tick instead of following it
    float   *host_obs, *host_reward;
    uint8_t *host_done;
    // ok_step_host_q16 (opt-in, lossy): the observations as 16-bit fixed point, q = rn(clamp(obs, 0, 1) * 65535), half the
    // bytes on the host link.  Excludes host_obs.
    uint16_t *host_obs_q16;
    // ok_step_host: a CTA's FIRST tile reads the caller's two action arrays through the host mapping; meanwhile the copy engine
    // brings both arrays to act_stage (device memory) on a side stream and then sets *act_ready = act_ready_target (a stream
    // memory operation), and every later tile reads the stage.  A mapped read issued after a tile's observations have been
    // flushed queues behind those posted writes (PCIe reads do not pass writes): 16-30 us per tile instead of 8, measured.
    float    *act_stage_thr, *act_stage_steer;
    uint32_t *act_ready;
    uint32_t  act_ready_target;
    // ok_step_host with flusher CTAs (obs_flush_kernel, launched next to this kernel): instead of copying a finished tile's
    // observations to the host itself, a CTA publishes flag[tile] = epoch and moves on to its next tile
    uint32_t *tile_flag;
    uint32_t  flag_epoch;
    // configuration
    int32_t  movement_mode, reward_mode, raycast_mode, auto_reset, auto_reset_stride;
    float    sensor_range, speed_limit, dt, collision_dist2, sensor_offset, standstill_thr2;
    uint32_t standstill_period;
};

// view of the staged blob
struct TrackView
{
    const float4   *seg;
    const uint2    *words;  // {occupancy bits, occupied-cell rank} per 32 cells
    const uint32_t *starts; // per occupied cell: first item | (one past the last) << 16
    const uint16_t *items;
    const float2   *pts;
    const float    *widths;
    const float    *headings;
    const float    *safe; // windowed nearest-point search, ok_track.hpp kNearestWindow
    int32_t         n_pts, n_seg, nx, ny;
    float           gx0, gy0, cell, inv_cell;
};

__device__ __forceinline__ TrackView make_view(const uint8_t *blob)
{
    const TrackHeader *h = reinterpret_cast<const TrackHeader *>(blob);
    TrackView          v;
    v.seg      = reinterpret_cast<const float4 *>(blob + h->off_segments);
    v.words    = reinterpret_cast<const uint2 *>(blob + h->off_words);
    v.starts   = reinterpret_cast<const uint32_t *>(blob + h->off_starts);
    v.items    = reinterpret_cast<const uint16_t *>(blob + h->off_items);
    v.pts      = reinterpret_cast<const float2 *>(blob + h->off_points);
    v.widths   = reinterpret_cast<const float *>(blob + h->off_widths);
    v.headings = reinterpret_cast<const float *>(blob + h->off_headings);
    v.safe     = reinterpret_cast<const float *>(blob + h->off_safe);
    v.n_pts = h->n_points, v.n_seg = h->n_segments, v.nx = h->grid_nx, v.ny = h->grid_ny;
    v.gx0 = h->grid_x0, v.gy0 = h->grid_y0, v.cell = h->cell, v.inv_cell = h->inv_cell;
    return v;
}

// ---------------------------------------------------------------------------------------------
// TMA bulk copy + mbarrier (PTX; SASS: UBLKCP / SYNCS)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "WAIT_%=:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@p bra DONE_%=;\n"
                 "bra WAIT_%=;\n"
                 "DONE_%=:\n"
                 "}" ::"r"(smem_u32(bar)),
                 "r"(phase)
                 : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared-memory atomic add as ONE instruction (ATOMS.ADD).  The CUDA atomicAdd() here sits behind `if (lane == 0)` inside
// a loop, and nvcc wraps it in its automatic warp aggregation (match / vote / popc / elect / shuffle, ~30 instructions for
// a single active lane): 9 % of the beam kernel's warp instructions in round 2's first profile.
__device__ __forceinline__ int smem_add(int *addr, int v)
{
    int old;
    asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(addr)), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ void smem_min(int *addr, int v)
{
    asm volatile("red.shared.min.s32 [%0], %1;" ::"r"(smem_u32(addr)), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------
// ray x segment: raySegmentIntersect, CollisionChecker.cu:8-35, with the running-minimum rule of
// castRaysToSegmentsKernel (CollisionChecker.cu:49-66).
//
// The reference walks the segments in ascending index and accepts t <= min_t, so its result is
// (smallest valid t, HIGHEST index among the segments attaining it): an order-independent rule,
// which lets the broadphase visit candidates in any order.  `best` is that index (-1 = none).
//
// Two IEEE divisions per pair is the reference's cost.  Here:
//  (1) a pair is first screened with comparisons on the numerators that are SUFFICIENT for the
//      reference's predicate to fail (proofs in DESIGN.md "exact early rejection").  With
//      a = tn*sign(denom), b = sn*sign(denom), ad = |denom| (t = a/ad, s = b/ad as reals):
//        b > ad              => RN(s) > 1            (RN(b/ad) <= 1 iff b <= ad for floats b, ad)
//        b < -2^-22          => RN(s) <= -2^-149 < 0 (|b/ad| > 2^-150 because ad < 2^128)
//        a < -2^-22          => RN(t) < 0            (same)
//        a > RN(RN(ad*m)*(1+2^-18)), RN(ad*m) >= 2^-100 => RN(t) > m(1+2^-21) >= incumbent
//  (2) the survivors (real crossings in front of the ray) are ranked on an APPROXIMATE quotient
//      tq = a * rcp(ad), |tq - RN(a/ad)| <= 2^-21 RN(a/ad): a candidate more than 2^-18 (relative)
//      away from the incumbent is decided without a division; only a candidate inside that band --
//      a near-tie -- is evaluated literally, against the incumbent's exact t.  The running value m
//      is therefore "exact t, or within 2^-21 of it"; the exact t of the winner is recomputed once
//      per ray in phase 3 (exact_t) from the same expression.
// NaN / non-finite operands fail every shortcut and reach the literal predicate, which rejects them.
// ---------------------------------------------------------------------------------------------
enum : uint32_t
{
    kWalkApprox  = 1u, // the running minimum is an approximate quotient (see test_segment)
    kWalkLaValid = 2u, // the look-ahead found the next occupied cell
    kWalkLaDone  = 4u  // the look-ahead ran past the limit: no further cell
};

__device__ __forceinline__ float exact_t(const float4 sg, const float ox, const float oy, const float dx, const float dy)
{
    const float ex    = fsub(sg.x, ox);
    const float ey    = fsub(sg.y, oy);
    const float denom = fsub(fmul(dx, sg.w), fmul(dy, sg.z));
    const float tn    = fsub(fmul(ex, sg.w), fmul(ey, sg.z));
    return __fdiv_rn(tn, denom);
}

__device__ __forceinline__ void test_segment(const float4 *segs, const int idx, const float ox, const float oy,
                                             const float dx, const float dy, float &m, int &best, uint32_t &flags)
{
    const float4   sg    = segs[idx];
    const float    ex    = fsub(sg.x, ox);
    const float    ey    = fsub(sg.y, oy);
    const float    denom = fsub(fmul(dx, sg.w), fmul(dy, sg.z));
    const float    sn    = fsub(fmul(ex, dy), fmul(ey, dx));
    const uint32_t db    = __float_as_uint(denom);
    const uint32_t adb   = db & 0x7fffffffu;
    const uint32_t sgn   = db & 0x80000000u;
    const float    ad    = __uint_as_float(adb);
    const float    b     = __uint_as_float(__float_as_uint(sn) ^ sgn);
    // most candidates end here: parallel (fabsf(denom) < 1e-8f), or the ray's line misses the segment
    if ((adb < 0x322BCC77u) | (b > ad) | (b < -0x1p-22f))
        return;
    // a segment registered in two cells along the ray comes back: it already is the incumbent (the literal
    // rule `idx > best` would reject it anyway, after two divisions)
    if (idx == best)
        return;
    const float tn = fsub(fmul(ex, sg.w), fmul(ey, sg.z));
    const float a  = __uint_as_float(__float_as_uint(tn) ^ sgn);
    if (a < -0x1p-22f)
        return;
    const float lim = fmul(ad, m);
    if ((lim >= 0x1p-100f) & (a > fmul(lim, 1.000003814697265625f))) // 1 + 2^-18
        return;
    // comfortably inside every edge: s in [0,1] needs no division (b in [0, ad], finite), t > 0
    if ((b >= 0.0f) & (adb < 0x5d800000u /* 2^60 */) & (a >= 0x1p-60f))
    {
        const float tq = __fdividef(a, ad);
        if (tq > fmul(m, 1.000003814697265625f))
            return;
        if (tq < fmul(m, 0.999996185302734375f)) // 1 - 2^-18
        {
            m    = tq;
            best = idx;
            flags |= kWalkApprox;
            return;
        }
    }
    // literal predicate of the reference, against the incumbent's exact t
    if (flags & kWalkApprox)
        m = exact_t(segs[best], ox, oy, dx, dy);
    flags &= ~kWalkApprox;
    const float t = __fdiv_rn(tn, denom);
    bool        s_ok = (b >= 0.0f) & (adb < 0x7f800000u);
    if (!s_ok)
    {
        const float s = __fdiv_rn(sn, denom);
        s_ok          = (s >= 0.0f) && (s <= 1.0f);
    }
    if (s_ok && (t >= 0.0f) && ((t < m) || ((t == m) && (idx > best))))
    {
        m    = t;
        best = idx;
    }
}

// every segment, ascending: the reference's own loop (OK_RAYCAST_BRUTE); returns the hit index
__device__ __forceinline__ int cast_ray_brute(const TrackView &tv, float ox, float oy, float dx, float dy, float range)
{
    float    m     = range;
    int      best  = -1;
    uint32_t flags = 0;
    for (int i = 0; i < tv.n_seg; ++i)
        test_segment(tv.seg, i, ox, oy, dx, dy, m, best, flags);
    return best;
}

// Uniform-grid broadphase: 2-D DDA over the cells the ray crosses, testing the segments
// registered in each cell, until the next cell starts beyond the current hit (+ slack).
// Exactness w.r.t. the brute-force loop is argued in DESIGN.md: segments are registered with a
// kGridMargin inflation that dominates every rounding error of this walk, and the per-pair
// arithmetic is the same function as above.
//
// The walk is a resumable state machine (begin / unit) because rays are NOT bound to lanes: the
// work per ray is heavy tailed (mean ~20 units, 1 ray in 32 needs 65+), so a lane that finishes
// its ray pulls the next one from a CTA-wide pool (see step_kernel phase 2).
//
// The grid carries a ring of empty cells around the clip box, so the walk needs no bounds checks:
// it stops at t1, the parameter at which the ray leaves the clip box (or its range).
#define OK_DDA_SLACK 0.5f
#ifndef OK_LA_STEPS
#define OK_LA_STEPS 2
#endif
#ifndef OK_TESTS
#define OK_TESTS 3
#endif
struct RayWalk
{
    float    ox, oy, dx, dy;
    float    min_t, t1;
    float    tmx, tmy, tdx, tdy;
    int      c, best;  // look-ahead cell (row-major index), incumbent segment
    uint32_t k, k_end; // items of the cell being tested
    uint32_t la_se;    // items of the look-ahead cell (first | end << 16), valid with kWalkLaValid
    float    la_t;     // ray parameter at which the look-ahead cell is entered
    uint32_t flags;
};

// item range of cell c, or 0 (empty range) when the cell is unoccupied
__device__ __forceinline__ uint32_t cell_items(const TrackView &tv, int c)
{
    const uint2 word = tv.words[c >> 5];
    if (!((word.x >> (c & 31)) & 1u))
        return 0u;
    const uint32_t r = word.y + __popc(word.x & ((1u << (c & 31)) - 1u));
    return tv.starts[r]; // first item | (one past the last item) << 16
}

// returns false when the ray cannot hit anything (result stays best = -1)
__device__ __forceinline__ bool walk_begin(const TrackView &tv, RayWalk &w, float ox, float oy, float dx, float dy,
                                           float range, float t_start = 0.0f)
{
    w.ox = ox, w.oy = oy, w.dx = dx, w.dy = dy;
    w.min_t = range;
    w.best  = -1;
    w.flags = 0;
    w.k = 0, w.k_end = 0;
    // a non-finite ray fails the reference predicate on every segment
    if (!(fabsf(ox) <= FLT_MAX && fabsf(oy) <= FLT_MAX && fabsf(dx) <= FLT_MAX && fabsf(dy) <= FLT_MAX))
        return false;
    // clip box = the grid without its one-cell ring (every segment lies >= 1 px inside it)
    const float bx0 = tv.gx0 + tv.cell, by0 = tv.gy0 + tv.cell;
    const float bx1 = tv.gx0 + (tv.nx - 1) * tv.cell, by1 = tv.gy0 + (tv.ny - 1) * tv.cell;
    float       t0 = t_start, t1 = range + OK_DDA_SLACK; // t_start > 0: everything nearer is already decided
    float       inv_dx = 0.0f, inv_dy = 0.0f;
    if (dx != 0.0f)
    {
        inv_dx         = __fdividef(1.0f, dx); // traversal only: any error here is covered by kGridMargin
        const float ta = (bx0 - ox) * inv_dx, tb = (bx1 - ox) * inv_dx;
        t0 = fmaxf(t0, fminf(ta, tb));
        t1 = fminf(t1, fmaxf(ta, tb));
    }
    else if (ox < bx0 || ox > bx1)
        return false;
    if (dy != 0.0f)
    {
        inv_dy         = __fdividef(1.0f, dy);
        const float ta = (by0 - oy) * inv_dy, tb = (by1 - oy) * inv_dy;
        t0 = fmaxf(t0, fminf(ta, tb));
        t1 = fminf(t1, fmaxf(ta, tb));
    }
    else if (oy < by0 || oy > by1)
        return false;
    if (!(t0 <= t1))
        return false; // the ray does not reach the clip box within range
    w.t1 = t1;

    const float px = ox + t0 * dx, py = oy + t0 * dy; // entry point
    int         ix = static_cast<int>(floorf((px - tv.gx0) * tv.inv_cell));
    int         iy = static_cast<int>(floorf((py - tv.gy0) * tv.inv_cell));
    ix             = min(max(ix, 1), tv.nx - 2);
    iy             = min(max(iy, 1), tv.ny - 2);
    const float inf = __int_as_float(0x7f800000);
    w.tmx = inf, w.tmy = inf, w.tdx = inf, w.tdy = inf;
    if (dx != 0.0f)
    {
        w.tmx = (tv.gx0 + (ix + (dx > 0.0f ? 1 : 0)) * tv.cell - ox) * inv_dx;
        w.tdx = tv.cell * fabsf(inv_dx);
    }
    if (dy != 0.0f)
    {
        w.tmy = (tv.gy0 + (iy + (dy > 0.0f ? 1 : 0)) * tv.cell - oy) * inv_dy;
        w.tdy = tv.cell * fabsf(inv_dy);
    }
    w.c = iy * tv.nx + ix;
    const uint32_t se = cell_items(tv, w.c);
    w.k = se & 0xffffu, w.k_end = se >> 16;
    return true;
}

// One unit of work = one DDA step of the LOOK-AHEAD (towards the next occupied cell) and one segment
// test in the CURRENT cell, so both halves of the code keep most lanes busy (a lane that alternates
// "step" and "test" units leaves each half of the warp's instruction stream half empty).  The
// look-ahead may run past the eventual hit; its cell is only adopted if it still starts within
// min_t + slack when the current cell is used up, so the set of tested cells is the one the plain
// walk would visit.  Returns false when the walk is over.
__device__ __forceinline__ bool walk_look_ahead(const TrackView &tv, RayWalk &w)
{ // one DDA step of the look-ahead; false = the walk left the grid (cannot happen, see walk_begin)
    if (!(w.flags & (kWalkLaValid | kWalkLaDone)))
    {
        const bool  step_x = w.tmx < w.tmy;
        const float t_next = step_x ? w.tmx : w.tmy;
        if (!(t_next <= fminf(w.min_t + OK_DDA_SLACK, w.t1)))
            w.flags |= kWalkLaDone;
        else
        {
            const int dcx = w.dx > 0.0f ? 1 : -1;
            const int dcy = w.dy > 0.0f ? tv.nx : -tv.nx;
            w.c += step_x ? dcx : dcy;
            if (static_cast<unsigned>(w.c) >= static_cast<unsigned>(tv.nx * tv.ny))
                return false; // keeps a rounding surprise from reading out of bounds
            w.tmx += step_x ? w.tdx : 0.0f;
            w.tmy += step_x ? 0.0f : w.tdy;
            const uint32_t se = cell_items(tv, w.c);
            if (se)
            {
                w.la_se = se;
                w.la_t  = t_next;
                w.flags |= kWalkLaValid;
            }
        }
    }
    return true;
}

__device__ __forceinline__ bool walk_unit(const TrackView &tv, RayWalk &w)
{
#pragma unroll
    for (int rep = 0; rep < OK_LA_STEPS; ++rep)
        if (!walk_look_ahead(tv, w))
            return false;
    if (w.k >= w.k_end)
    {
        if (w.flags & kWalkLaValid)
        {
            if (!(w.la_t <= w.min_t + OK_DDA_SLACK))
                return false;
            w.k = w.la_se & 0xffffu, w.k_end = w.la_se >> 16;
            w.flags &= ~kWalkLaValid;
        }
        else if (w.flags & kWalkLaDone)
            return false;
    }
#pragma unroll
    for (int rep = 0; rep < OK_TESTS; ++rep)
        if (w.k < w.k_end)
        {
            const int i = tv.items[w.k++];
            test_segment(tv.seg, i, w.ox, w.oy, w.dx, w.dy, w.min_t, w.best, w.flags);
        }
    return true;
}

// RaceTrack::findNearestTrackIndexBruteForce (RaceTrack.cpp:16-31), cooperatively by the `lpa`
// lanes of an agent: strict '<' keeps the lowest index on ties, so the combine is the
// lexicographic minimum of (distance, index) -- order independent, hence exact.
__device__ __forceinline__ int nearest_index(const TrackView &tv, float qx, float qy, int sub, int lpa, float &d2_out)
{
    float best = FLT_MAX;
    int   bi   = 0;
    for (int i = sub; i < tv.n_pts; i += lpa)
    {
        const float2 p  = tv.pts[i];
        const float  ddx = fsub(qx, p.x), ddy = fsub(qy, p.y);
        const float  d  = fadd(fmul(ddx, ddx), fmul(ddy, ddy)); // Vec2d::distanceSquared, Typedefs.h:40-43
        if (d < best)
        {
            best = d;
            bi   = i;
        }
    }
    for (int o = lpa >> 1; o > 0; o >>= 1)
    {
        const float od = __shfl_xor_sync(0xffffffffu, best, o);
        const int   oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (od < best || (od == best && oi < bi))
        {
            best = od;
            bi   = oi;
        }
    }
    d2_out = best;
    return bi;
}

// The same search by ONE thread with a hint (the agent's previous nearest index; phase 4 runs a thread per agent):
// the 32 points around the hint first; the rest only if the triangle inequality cannot rule them out
// (ok_track.hpp, kNearestWindow).  ok = true: every outside point is STRICTLY farther than the window's best, so the
// window's lexicographic (distance, index) minimum is the reference's result.  ok = false means "not proven": the
// caller runs the full search above.  Ties: lowest index, like the reference (the window wraps around the end of the
// centre line, so index order is not visiting order).
// kPostLanes = lanes that share one agent in phase 4 (4 for batches of up to 256 agents: every warp of the CTA gets
// work and the window scan is 4x shorter; 1 for the larger batches of large populations)
template <int kPostLanes>
__device__ __forceinline__ int nearest_index_window(const TrackView &tv, float qx, float qy, int hint, int lane, float &d2_out,
                                                    bool &ok)
{ // called by whole warps; kPostLanes consecutive lanes hold the same query and split the window between them
    const int n   = tv.n_pts;
    const int sub = lane & (kPostLanes - 1);
    constexpr int per = kNearestWindow / kPostLanes;
    ok          = false;
    d2_out      = FLT_MAX;
    if (n <= kNearestWindow)
        return 0;
    const int h    = min(max(hint, 0), n - 1);
    float     best = FLT_MAX, dh = FLT_MAX;
    int       bi   = 0;
    int       i    = h - kNearestWindow / 2 + sub * per;
    i += (i < 0) ? n : 0;
    i -= (i >= n) ? n : 0;
#pragma unroll
    for (int k = 0; k < per; ++k)
    {
        const float2 pt  = tv.pts[i];
        const float  ddx = fsub(qx, pt.x), ddy = fsub(qy, pt.y);
        const float  d   = fadd(fmul(ddx, ddx), fmul(ddy, ddy));
        dh               = (k == (kNearestWindow / 2) % per) ? d : dh; // the hint itself, in lane (window / 2) / per
        if (d < best || (d == best && d < FLT_MAX && i < bi))
        {
            best = d;
            bi   = i;
        }
        ++i;
        i = (i >= n) ? 0 : i;
    }
#pragma unroll
    for (int o = 1; o < kPostLanes; o <<= 1)
    {
        const float od = __shfl_xor_sync(0xffffffffu, best, o);
        const int   oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (od < best || (od == best && od < FLT_MAX && oi < bi))
        {
            best = od;
            bi   = oi;
        }
    }
    dh             = __shfl_sync(0xffffffffu, dh, (lane & ~(kPostLanes - 1)) + (kNearestWindow / 2) / per);
    const float rb = __fsqrt_rn(best), rh = __fsqrt_rn(dh);
    ok             = fsub(fsub(tv.safe[h], rh), rb) > fadd(fmul(1e-3f, fadd(rh, rb)), 1e-3f);
    d2_out         = best;
    return bi;
}

// ---------------------------------------------------------------------------------------------
// the tick
// ---------------------------------------------------------------------------------------------
// per-agent scratch in shared memory while its batch is in flight
struct AgentRec
{
    float    ox, oy, rc, rs; // lidar origin, cos/sin of the heading
    float    rot;            // heading after the move (degrees)
    uint32_t flags;
    int32_t  row;            // beam-table row of the lidar origin's cell, -1 = not covered (beam modes only)
    int      min_d2_bits;    // running min of the squared hit norms (as int: all values are >= +0)
    float    x, y;           // pose after the move
    float    rx, ry;         // where a reset put the agent (FLAG_RESET)
    int32_t  prev;           // prev_track_idx_ / accumulated fitness before this tick (phase 4 works from this record)
    float    fitness;
    int32_t  hint;           // where the nearest-centre-line search starts: last tick's index, or the reset point
    int32_t  pad;
};
static_assert(sizeof(AgentRec) == 64, "AgentRec layout");
enum : uint32_t
{
    kFlagCrashed = 1u,
    kFlagTimedOut = 2u,
    kFlagReset = 4u
};

// ---------------------------------------------------------------------------------------------
// Beam lists (ok_beam.hpp): the narrow phase reads, for the ray's start cell and direction bin, the
// precomputed list of segments it can reach, nearest first, and tests them -- no traversal.  The
// lists of a warp's 32 rays are cut into chunks of 4 candidates and dealt evenly to the 32 lanes
// (a lane finds the owner of its chunk by a shuffle binary search over the chunk prefix sums), so
// the heavy tail of the per-ray work does not idle lanes.  Results meet in a 64-bit key per ray in
// shared memory, (exact t bits) << 32 | (0x7fffffff - segment): atomicMin implements the
// reference's rule "smallest t, highest index among ties" (CollisionChecker.cu:49-66).
// ---------------------------------------------------------------------------------------------
struct BeamView
{
    const uint32_t *rows;
    const uint4    *entries; // {inline candidates 0-1, 2-3, first rest chunk, meta}: ok_beam.hpp
    const uint2    *chunks;  // rest lists: 4 x uint16 segment indices per chunk
    float           x0, y0, inv_h, bin_scale, rb;
    int32_t         nx, ny, nb;
    uint32_t        n_rows, n_chunks; // OK_CHECKED builds only
    bool            valid;
};

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

// row of the beam cell that contains (ox, oy), -1 = not covered (same arithmetic as ok::beam_lookup)
__device__ __forceinline__ int32_t beam_row(const BeamView &bv, float ox, float oy)
{
    if (!bv.valid)
        return -1;
    const float fx = fmul(fsub(ox, bv.x0), bv.inv_h), fy = fmul(fsub(oy, bv.y0), bv.inv_h);
    if (!(fx >= 0.0f && fy >= 0.0f && fx < static_cast<float>(bv.nx) && fy < static_cast<float>(bv.ny)))
        return -1;
    return static_cast<int32_t>(__ldg(bv.rows + static_cast<int>(fy) * bv.nx + static_cast<int>(fx)));
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

// hit point, unpack (CollisionChecker.cu:68-69,152-165) and the per-ray outputs of ray `gi`, whose nearest
// segment is `seg` (-1 = none); returns the squared norm of the relative hit
// t_known != 0: the winner's exact t is already at hand (the beam key holds it; a zero is recomputed because the
// key does not keep its sign)
// ok_step_host_q16's fixed point: round-to-nearest-even of clamp(obs, 0, 1) * 65535 (a NaN becomes 0)
__device__ __forceinline__ uint32_t obs_q16(const float ob)
{
    return __float2uint_rn(fmul(fminf(fmaxf(ob, 0.0f), 1.0f), 65535.0f));
}

template <bool kHostStore = true, typename Rec>
__device__ __forceinline__ float finish_ray(const StepParams &p, const float4 *segs, const Rec &rec, const int64_t gi,
                                            const float dx, const float dy, const int seg, const float t_known = 0.0f)
{
    float2 hit;
    if (!(rec.flags & kFlagCrashed))
    {
        // min_t of CollisionChecker.cu:49-66: the winner's t by the reference's expression
        const float t = seg >= 0 ? (t_known != 0.0f ? t_known : exact_t(segs[seg], rec.ox, rec.oy, dx, dy)) : p.sensor_range;
        p.hit_seg[gi] = seg;
        p.hit_t[gi]   = t;
        hit.x         = fadd(rec.ox, fmul(t, dx));
        hit.y         = fadd(rec.oy, fmul(t, dy));
        reinterpret_cast<float2 *>(p.hit_abs)[gi] = hit;
    }
    else
        hit = reinterpret_cast<const float2 *>(p.hit_abs)[gi]; // stale hit of a crashed agent
    OK_CHECK(gi >= 0 && seg >= -1);
    const float xt = fsub(hit.x, rec.ox), yt = fsub(hit.y, rec.oy);
    float2      rel;
    rel.x          = fsub(fmul(xt, rec.rc), fmul(yt, rec.rs));
    rel.y          = fadd(fmul(xt, rec.rs), fmul(yt, rec.rc));
    const float sq = fadd(fmul(rel.x, rel.x), fmul(rel.y, rel.y));
    reinterpret_cast<float2 *>(p.hit_rel)[gi] = rel;
    const float ob = __fdiv_rn(__fsqrt_rn(sq), p.sensor_range);
    p.obs[gi]      = ob;
    if (kHostStore && p.host_obs) // (the beam kernel copies a whole tile's observations at once, see its tile flush)
        p.host_obs[gi] = ob;
    if (kHostStore && p.host_obs_q16)
        p.host_obs_q16[gi] = static_cast<uint16_t>(obs_q16(ob));
    return sq;
}

__host__ __device__ inline size_t batch_smem_bytes(int agents, int rays)
{ // AgentRec + per ray float2 direction
    return static_cast<size_t>(agents) * (sizeof(AgentRec) + 8u * static_cast<size_t>(rays));
}
// beam mode: AgentRec only (the per-thread scratch is static shared memory)
__host__ __device__ inline size_t beam_smem_bytes(int agents)
{
    return (static_cast<size_t>(agents) * sizeof(AgentRec) + 15u) / 16u * 16u;
}

// Phase 1 for agent `a` (one thread): optional auto-reset, kinematics from the action, standstill timeout
// (Environment.cpp:128-143), lidar origin (CollisionChecker.cu:121-124).  Writes the agent's state buffers and
// returns the record the ray and reward phases work from.
// `gblob` is the track's blob in the GLOBAL arena: only a crashed agent's auto-reset reads it (centre line, headings),
// so phase 1 does not have to wait for the blob to be staged in shared memory.
__device__ __forceinline__ AgentRec agent_pre(const StepParams &p, const uint8_t *gblob, const TrackRef &tr, const BeamView &bv, const int64_t a,
                                              const bool act_staged = false, const float2 *s_action = nullptr)
{
    float    x = p.x[a], y = p.y[a], rot = p.rot[a], speed = p.speed[a], accel = p.accel[a];
    bool     crashed = p.crashed[a] != 0, timed_out = p.timed_out[a] != 0;
    // (auto-reset) the reset point is requested with the rest of the state, not after the crash flag has arrived
    const int32_t reset_pt0 = (p.auto_reset && p.do_move) ? p.reset_pt[a] : 0;
    // the standstill record is read up front with the rest of the state: a load issued only after the kinematics
    // would add a second trip to memory to the latency of this (latency-bound) phase
    const uint32_t ss_ctr0 = p.ss_ctr[a];
    const float    ss_x0 = p.ss_x[a], ss_y0 = p.ss_y[a];
#ifdef OK_PRE_PROBE // experiment build: where does a thread's phase 1 spend its time?  (slots 3-5 of the tile trace, thread 0)
#define OK_PROBE(slot, dep)                                                                                            \
    if (p.trace && threadIdx.x == 0)                                                                                   \
    {                                                                                                                  \
        unsigned long long t_;                                                                                         \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_) : "r"(__float_as_int(dep)) : "memory");                  \
        p.trace[static_cast<size_t>(blockIdx.x) * p.trace_tiles * 6 + (slot)] = t_;                                    \
    }
#else
#define OK_PROBE(slot, dep)
#endif
    uint32_t flags = 0;
    float    rx = 0.0f, ry = 0.0f;
    float    hs = 0.0f, hc = 0.0f; // sin / cos of the heading, when the move already computed them
    OK_PROBE(3, x + y + rot + speed + accel + (crashed ? 1.0f : 0.0f) + static_cast<float>(ss_ctr0) + ss_x0)
    bool     have_sc = false;
    int32_t  hint = p.nearest[a], prev_idx = 0;
    float    fitness = 0.0f;
    if (p.do_move)
    {
        prev_idx = p.prev[a];
        fitness  = p.fitness[a];
        float thr, steer;
        if (p.action_source == 1)
        { // synthetic stream: Philox4x32-10, counter (agent, step), key (seed, 0)
            uint32_t o[4];
            const uint64_t id = p.id_base + static_cast<uint64_t>(a);
            philox4x32_10(static_cast<uint32_t>(id), static_cast<uint32_t>(id >> 32),
                          static_cast<uint32_t>(p.step), static_cast<uint32_t>(p.step >> 32), p.seed, 0u, o);
            if (p.movement_mode == 1)
            { // GeneticAgent.hpp:22-24 action set
                const uint32_t ti = o[0] % 3u, si = o[1] % 5u;
                thr   = ti == 0 ? -0.3f : (ti == 1 ? 0.0f : 0.3f);
                steer = si == 0 ? -4.0f : (si == 1 ? -1.0f : (si == 2 ? 0.0f : (si == 3 ? 1.0f : 4.0f)));
            }
            else
            { // ReinforceAgent.hpp:92-93 ranges
                thr   = fmul(100.0f, fmul(static_cast<float>(o[0] >> 8), 0x1p-24f));
                steer = fsub(fmul(10.0f, fmul(static_cast<float>(o[1] >> 8), 0x1p-24f)), 5.0f);
            }
        }
        else if (p.ext_thr && act_staged)
        { // this launch's copy of the caller's arrays in device memory (see StepParams::act_ready)
            thr   = __ldcg(p.act_stage_thr + a);
            steer = __ldcg(p.act_stage_steer + a);
        }
        else if (p.ext_thr)
        {
            thr   = p.ext_thr[a];
            steer = p.ext_steer[a];
        }
        else if (s_action)
        { // the fused policy phase left it in shared memory (and in the action buffers)
            thr   = s_action->x;
            steer = s_action->y;
        }
        else
        {
            thr   = p.act_thr[a];
            steer = p.act_steer[a];
        }
        // app-side reset of a crashed agent before the tick (GuidedCostLearning/test.cpp:102-111):
        // Environment::resetAgent + Agent::reset, Environment.cpp:103-121 / Agent.cpp:123-135.
        // prev / nearest / fitness are finalised in phase 4 (they need a centre-line search).
        if (p.auto_reset && crashed)
        {
            const int32_t pt = static_cast<int32_t>((static_cast<int64_t>(reset_pt0) + p.auto_reset_stride) % tr.n_points);
            const float2  c  = reinterpret_cast<const float2 *>(gblob + tr.off_points)[pt];
            x = c.x, y = c.y, rot = reinterpret_cast<const float *>(gblob + tr.off_headings)[pt];
            accel = 0.0f, speed = 0.0f;
            crashed = false, timed_out = false;
            thr = 0.0f, steer = 0.0f; // Agent::reset zeroes current_action_
            rx = x, ry = y;
            flags |= kFlagReset;
            hint     = pt;
            prev_idx = 0;
            fitness  = 0.0f;
            p.reset_pt[a] = pt;
            p.start_x[a]  = x;
            p.start_y[a]  = y;
        }
        p.act_thr[a]   = thr;
        p.act_steer[a] = steer;
        if (!crashed)
        {
            rot = fadd(rot, steer);
            if (p.movement_mode == 1)
            { // moveViaAcceleration, Agent.cpp:82-98
                accel = fadd(accel, thr);
                speed = fadd(speed, fmul(accel, p.dt));
                speed = (speed < 0.0f) ? 0.0f : speed;
                speed = (speed > p.speed_limit) ? p.speed_limit : speed;
            }
            else
            { // moveViaVelocity, Agent.cpp:108-119
                speed = thr;
            }
            float ms, mc;
            sincosf(fmul(OK_DEG2RAD, rot), ms, mc);
            hs = ms, hc = mc, have_sc = true; // the lidar origin below uses the same heading
            x = fadd(x, fmul(fmul(mc, speed), p.dt));
            y = fadd(y, fmul(fmul(ms, speed), p.dt));
            // checkAndUpdateStandstill, Environment.cpp:16-39
            uint32_t ctr = ss_ctr0;
            bool     out = false;
            if (ctr == 0)
            {
                p.ss_x[a] = x;
                p.ss_y[a] = y;
                ctr       = 1;
            }
            else if (ctr >= p.standstill_period)
            {
                const float mx = fsub(x, ss_x0), my = fsub(y, ss_y0);
                out = fadd(fmul(mx, mx), fmul(my, my)) < p.standstill_thr2;
                ctr = 0;
            }
            else
                ++ctr;
            p.ss_ctr[a] = ctr;
            if (out)
            {
                crashed   = true;
                timed_out = true;
            }
        }
        p.x[a] = x, p.y[a] = y, p.rot[a] = rot, p.speed[a] = speed, p.accel[a] = accel;
        p.timed_out[a] = timed_out;
    }
    // lidar origin, CollisionChecker.cu:121-124
    float rs = hs, rc = hc;
    if (!have_sc)
        sincosf(fmul(OK_DEG2RAD, rot), rs, rc);
    AgentRec rec;
    rec.ox = fadd(x, fmul(p.sensor_offset, rc));
    rec.oy = fadd(y, fmul(p.sensor_offset, rs));
    rec.rc = rc, rec.rs = rs, rec.rot = rot, rec.x = x, rec.y = y, rec.rx = rx, rec.ry = ry;
    rec.min_d2_bits = __float_as_int(fmul(p.sensor_range, p.sensor_range));
    rec.flags       = flags | (crashed ? kFlagCrashed : 0u) | (timed_out ? kFlagTimedOut : 0u);
    OK_PROBE(4, rec.ox + rec.oy)
    rec.row         = beam_row(bv, rec.ox, rec.oy); // -1 when bv is not valid
    OK_PROBE(5, static_cast<float>(rec.row))
    rec.prev = prev_idx, rec.fitness = fitness, rec.hint = hint, rec.pad = 0;
    return rec;
}

// Phase 4 for agent `a` (kPostLanes consecutive lanes per agent, they split the centre-line window; the WHOLE warp must
// call this, lanes without an agent with valid = false):
// crash flag (CollisionChecker.cu:167-171), nearest centre-line index, progress / reward / done.
template <int kPostLanes>
__device__ __forceinline__ void agent_post(const StepParams &p, const TrackView &tv, const AgentRec &rec, const int64_t a,
                                           const bool valid, const int lane)
{
    const int  mode     = p.reward_mode;
    const bool need_idx = p.do_move && (mode == 1 || mode == 2 || mode == 6 || mode == 7);
            const float    min_d2 = __int_as_float(rec.min_d2_bits);
    bool           crashed = (rec.flags & kFlagCrashed) != 0;
    const bool     timed_out = (rec.flags & kFlagTimedOut) != 0;
    if (min_d2 < p.collision_dist2) // CollisionChecker.cu:167-171
        crashed = true;
    int32_t prev = rec.prev, near = 0;
    float   fitness = rec.fitness, near_d2 = 0.0f;
    // RaceTrack::findNearestTrackIndexBruteForce: the window around last tick's index first; the rare
    // agents it cannot prove (teleported by a buffer write, track folding back on itself) get the
    // full search, their warp's 32 lanes sharing it
    const bool leader     = (lane & (kPostLanes - 1)) == 0; // the lane that writes the agent's results
    const bool want_reset = valid && (rec.flags & kFlagReset) != 0;
    bool       ok_reset   = true;
    if (__any_sync(0xffffffffu, want_reset))
    { // prev_track_idx_ = nearest index of the post-reset pose (main_eigen.cpp:121-130)
        float     d2;
        bool      okw;
        const int r = nearest_index_window<kPostLanes>(tv, rec.rx, rec.ry, rec.hint, lane, d2, okw);
        if (want_reset)
        {
            prev     = r;
            ok_reset = okw;
        }
    }
    for (unsigned need = __ballot_sync(0xffffffffu, !ok_reset && leader); need; need &= need - 1)
    {
        const int src = __ffs(need) - 1;
        float     d2;
        const int r = nearest_index(tv, __shfl_sync(0xffffffffu, rec.rx, src), __shfl_sync(0xffffffffu, rec.ry, src), lane, 32, d2);
        if ((lane & ~(kPostLanes - 1)) == src)
            prev = r;
    }
    if (want_reset)
        near = prev;
    const bool want_near = valid && need_idx;
    bool       ok_near   = true;
    if (__any_sync(0xffffffffu, want_near))
    {
        float     d2;
        bool      okw;
        const int r = nearest_index_window<kPostLanes>(tv, rec.x, rec.y, want_reset ? prev : rec.hint, lane, d2, okw);
        if (want_near)
        {
            near    = r;
            near_d2 = d2;
            ok_near = okw;
        }
    }
    for (unsigned need = __ballot_sync(0xffffffffu, !ok_near && leader); need; need &= need - 1)
    {
        const int src = __ffs(need) - 1;
        float     d2;
        const int r = nearest_index(tv, __shfl_sync(0xffffffffu, rec.x, src), __shfl_sync(0xffffffffu, rec.y, src), lane, 32, d2);
        if ((lane & ~(kPostLanes - 1)) == src)
        {
            near    = r;
            near_d2 = d2;
        }
    }
    if (valid && leader)
    {
        if (p.do_move)
        {
            float reward = 0.0f;
            switch (mode)
            {
            case 1: // QAgent.hpp:150-168
                if (crashed)
                    reward = -200.0f;
                else
                {
                    const int32_t prog = near - prev;
                    prev               = near;
                    const int32_t ab = prog < 0 ? -prog : prog, len = tv.n_pts;
                    reward = static_cast<float>(ab > (len / 2) ? len - ab : ab);
                }
                break;
            case 2: // main_eigen.cpp:147-163
                if (!crashed)
                {
                    const int32_t prog = near - prev;
                    prev               = near;
                    reward             = static_cast<float>(prog < 0 ? -prog : prog);
                    fitness            = fadd(fitness, reward);
                }
                else if (timed_out)
                    fitness = 0.0f;
                break;
            case 3: reward = 1.0f; break; // ppo_sim.cpp:76
            case 4:                       // ReinforceContinuous/reinforce_sim.cpp:59-73
            {
                const float ddx = fsub(rec.x, p.start_x[a]), ddy = fsub(rec.y, p.start_y[a]);
                reward = crashed ? -5.0f : __fsqrt_rn(fadd(fmul(ddx, ddx), fmul(ddy, ddy)));
                break;
            }
            case 5: // DQAgent.hpp:161-180: min over rays of norm() == sqrt of the min squared norm
            {
                const float m = __fsqrt_rn(min_d2);
                reward        = crashed ? -200.0f : (p.sensor_range > m ? m : p.sensor_range);
                break;
            }
            case 6: reward = static_cast<float>(near); break; // MiscUtils.hpp:64-71
            case 7:                                           // WorldModelVaeRnn/main.cpp:336-342
                if (!crashed)
                {
                    reward  = fsub(1.0f, __fdiv_rn(__fsqrt_rn(near_d2), tv.widths[near])); // RaceTrack.cpp:53-72
                    fitness = fadd(fitness, reward);
                }
                else if (timed_out)
                    fitness = 0.0f;
                break;
            default: break;
            }
            p.reward[a]  = reward;
            if (p.host_reward)
                p.host_reward[a] = reward;
            p.fitness[a] = fitness;
            p.prev[a]    = prev;
            if (need_idx || (rec.flags & kFlagReset))
                p.nearest[a] = near;
        }
        p.crashed[a]   = crashed;
        p.done[a]      = crashed; // Agent::isDone, Agent.cpp:138-144 (completed_ is never set)
        if (p.host_done)
            p.host_done[a] = crashed;
        p.min_dist2[a] = min_d2;
    }
}

#ifndef OK_UNITS
#define OK_UNITS 4
#endif
constexpr int kUnitsPerRefill = OK_UNITS; // units of work a lane does between two looks at the pool
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
#ifndef OK_BEAM_PREFETCH
#define OK_BEAM_PREFETCH 0 // measured: an L2 prefetch of the queued rays' rest chunks costs 12 % (0.129 vs 0.115 ms)
#endif
#ifndef OK_BEAM_TILE
#define OK_BEAM_TILE 64 // agents per tile of the unstaged beam kernel
#endif
constexpr int kBeamBlockStaged   = 1024;
constexpr int kBeamBlockUnstaged = OK_BEAM_BLOCK;
// capacity of the CTA's queue of rays pass A leaves to pass B.  Tile-local ray indices are 16 bits, so a beam tile holds
// at most 65,535 rays (the host caps the batch); a full queue only costs speed (see pass A).
__host__ __device__ constexpr int beam_pend_cap(bool staged)
{
    return staged ? 8192 : 2048;
}
// static shared memory of the beam kernel besides the staged track and the agent records (host: batch sizing)
__host__ __device__ constexpr int beam_static_smem(bool staged)
{
    return (staged ? kBeamBlockStaged : kBeamBlockUnstaged) * (16 + 8) + 2 * beam_pend_cap(staged) + 4 * (beam_pend_cap(staged) / 32) + 128;
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
        if (kBeam && OK_TRACE_ON(slot) && p.trace && tid == 0 && n_done < p.trace_tiles)                                                    \
            p.trace[(static_cast<size_t>(blockIdx.x) * p.trace_tiles + n_done) * 6 + (slot)] = global_timer();         \
    } while (0)

// PPOAgent::updateAction + Actor::forward for every agent (RLRacers/PPO/PPOAgent.hpp:79-102, Actor.hpp:9-26): ONE
// kernel per tick does observation -> Linear(R, H) -> relu -> Linear(H, A) -> softmax -> clamp [1e-8, 1 - 1e-8] ->
// sample an action (torch::multinomial's distribution: inverse CDF of the clamped probabilities on a uniform draw) ->
// log-probability -> kActionMap lookup into the action buffers.  The weights are shared by all agents and staged in
// shared memory; kActorLanes lanes share an agent (each takes every kActorLanes-th hidden unit), logits meet by shuffles.
// It also records: the observation the action was chosen from, and the PREVIOUS tick's reward / done (so a rollout costs
// two launches per tick: this kernel and the step kernel).
struct ActorParams
{
    const float *w1, *b1, *w2, *b2; // torch Linear layouts: w1 [H][R], w2 [A][H]
    int32_t      hidden, n_actions;
    const float *table;   // [A][2] = (throttle, steering) per action, PPOAgent::kActionMap
    const float *uniform; // nullable: explicit draws in [0, 1), one per agent (tests); else Philox (id_base + a, step)
    int32_t      greedy;  // != 0: argmax instead of sampling
    int32_t     *action_out; // nullable outputs, one row of a rollout buffer each
    float       *log_prob_out, *probs_out, *obs_out;
    float       *prev_reward_out; // nullable: reward / done of the tick BEFORE this call (the env's buffers as they are)
    uint8_t     *prev_done_out;
    int32_t      act; // 0: only record prev_reward / prev_done (the flush after the last tick)
};
constexpr int kActorLanes   = 8;
constexpr int kActorMaxActs = 8;

// the weights of the actor, global -> shared memory (w1 | b1 | w2 | b2 | action table); the caller synchronises the CTA afterwards
__device__ __forceinline__ void actor_stage_weights(const ActorParams &q, const int R, float *s_w, const int tid, const int n_threads)
{
    const int H = q.hidden, A = q.n_actions;
    float    *s_w1 = s_w, *s_b1 = s_w1 + H * R, *s_w2 = s_b1 + H, *s_b2 = s_w2 + A * H;
    for (int i = tid; i < H * R; i += n_threads)
        s_w1[i] = q.w1[i];
    for (int i = tid; i < H; i += n_threads)
        s_b1[i] = q.b1[i];
    for (int i = tid; i < A * H; i += n_threads)
        s_w2[i] = q.w2[i];
    for (int i = tid; i < A; i += n_threads)
        s_b2[i] = q.b2[i];
    for (int i = tid; i < 2 * A; i += n_threads) // kActionMap behind the biases
        s_b2[A + i] = q.table[i];
}

// One agent's policy step by the kActorLanes lanes that share it (`sub` = the lane's place among them; `has` = the group holds
// an agent).  Warp-collective: all 32 lanes of a warp call it together.
__device__ __forceinline__ void actor_agent(const StepParams &p, const ActorParams &q, const float *s_w, const int64_t a, const bool has,
                                            const int sub, float2 *s_chosen = nullptr)
{ // s_chosen (fused instantiation): where the agent's own thread of the kinematics phase picks the action up (shared memory)
    const int    R = p.rays, H = q.hidden, A = q.n_actions;
    const float *s_w1 = s_w, *s_b1 = s_w1 + H * R, *s_w2 = s_b1 + H, *s_b2 = s_w2 + A * H;
    const int64_t ac  = has ? a : 0;
    if (has && sub == 0)
    { // the tick before this call
        if (q.prev_reward_out)
            q.prev_reward_out[a] = p.reward[a];
        if (q.prev_done_out)
            q.prev_done_out[a] = p.done[a];
    }
    if (!q.act)
        return;
    const float *obs = p.obs + ac * R;
    float        logit[kActorMaxActs];
#pragma unroll
    for (int k = 0; k < kActorMaxActs; ++k)
        logit[k] = 0.0f;
    // (plain loads of the observation: the fused instantiation rewrites p.obs later in the same launch.)  Fans of up to eight
    // rays -- the PPO racers' five -- are kept in registers: read in the loop they are eighty dependent L1 round trips per lane
    constexpr int kObsRegs = 8;
    const bool    in_regs  = R <= kObsRegs;
    float         ob[kObsRegs];
#pragma unroll
    for (int r = 0; r < kObsRegs; ++r)
        ob[r] = (in_regs && r < R) ? obs[r] : 0.0f;
    for (int h = sub; h < H; h += kActorLanes)
    {
        float        acc = s_b1[h];
        const float *row = s_w1 + h * R;
        if (in_regs)
        {
#pragma unroll
            for (int r = 0; r < kObsRegs; ++r)
                if (r < R)
                    acc = fmaf(row[r], ob[r], acc);
        }
        else
            for (int r = 0; r < R; ++r)
                acc = fmaf(row[r], obs[r], acc);
        acc = fmaxf(acc, 0.0f); // relu
#pragma unroll
        for (int k = 0; k < kActorMaxActs; ++k)
            if (k < A)
                logit[k] = fmaf(s_w2[k * H + h], acc, logit[k]);
    }
#pragma unroll
    for (int k = 0; k < kActorMaxActs; ++k)
        if (k < A) // (uniform)
#pragma unroll
            for (int o = kActorLanes >> 1; o > 0; o >>= 1)
                logit[k] += __shfl_xor_sync(0xffffffffu, logit[k], o);
    if (!has || sub != 0)
        return;
    // softmax (max-subtracted, as torch::softmax), clamp of PPOAgent.hpp:82-83 (the bounds narrow to float: 1e-8f, 1.0f)
    float mx = -FLT_MAX;
#pragma unroll
    for (int k = 0; k < kActorMaxActs; ++k)
        if (k < A)
        {
            logit[k] += s_b2[k];
            mx = fmaxf(mx, logit[k]);
        }
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < kActorMaxActs; ++k)
        if (k < A)
        {
            logit[k] = expf(logit[k] - mx);
            sum += logit[k];
        }
    float total = 0.0f;
#pragma unroll
    for (int k = 0; k < kActorMaxActs; ++k)
        if (k < A)
        {
            logit[k] = fminf(fmaxf(__fdiv_rn(logit[k], sum), 1e-8f), 1.0f);
            total += logit[k];
            if (q.probs_out)
                q.probs_out[a * A + k] = logit[k];
        }
    int act = 0;
    if (q.greedy)
    {
#pragma unroll
        for (int k = 1; k < kActorMaxActs; ++k)
            if (k < A && logit[k] > logit[act])
                act = k;
    }
    else
    { // torch::multinomial(probs, 1): index k with probability probs[k] / sum(probs)
        float u;
        if (q.uniform)
            u = q.uniform[a];
        else
        {
            uint32_t       o[4];
            const uint64_t id = p.id_base + static_cast<uint64_t>(a);
            philox4x32_10(static_cast<uint32_t>(id), static_cast<uint32_t>(id >> 32), static_cast<uint32_t>(p.step),
                          static_cast<uint32_t>(p.step >> 32), p.seed, 0x50504fu /* "PPO": a stream of its own */, o);
            u = static_cast<float>(o[0] >> 8) * 0x1p-24f;
        }
        const float target = u * total;
        float       cum    = 0.0f;
        act                = A - 1;
#pragma unroll
        for (int k = 0; k < kActorMaxActs; ++k)
            if (k < A)
            {
                cum += logit[k];
                if (target < cum && act == A - 1 && k < A - 1)
                    act = k;
            }
    }
    float pa = logit[0];
#pragma unroll
    for (int k = 1; k < kActorMaxActs; ++k)
        pa = (k == act) ? logit[k] : pa;
    if (q.action_out)
        q.action_out[a] = act;
    if (q.log_prob_out)
        q.log_prob_out[a] = logf(pa);
    if (q.obs_out)
        for (int r = 0; r < R; ++r)
            q.obs_out[a * R + r] = obs[r];
    const float thr = s_b2[A + 2 * act], steer = s_b2[A + 2 * act + 1]; // PPOAgent.hpp:95-96
    p.act_thr[a]   = thr;
    p.act_steer[a] = steer;
    if (s_chosen)
        *s_chosen = make_float2(thr, steer);
}

// the second kernel argument of step_kernel: the actor's parameters in the fused instantiation (kActor), nothing otherwise
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

// kActor (ok_ppo_actor_step): the PPO racers' policy step runs as phase 0 of every tile -- the tile's agents choose their
// actions from last tick's observations (actor_agent) and the kinematics read them from the action buffers -- so that a
// rollout tick is ONE launch: at a few thousand agents a tick is latency, and two kernels pay it twice.
template <int kBlock, bool kBeam, bool kStaged = true, bool kActor = false>
__global__ void __launch_bounds__(kBlock, (kBeam && !kStaged) ? OK_BEAM_MIN_CTAS : 1)
    step_kernel(const StepParams p, const typename ActorArg<kActor>::type q)
{
    static_assert(!kActor || kBeam, "the fused actor is built for the beam kernels");
    constexpr bool kStage   = !kBeam || kStaged; // the track is staged in shared memory with one TMA bulk copy
    constexpr int  kPendCap = beam_pend_cap(kStaged);
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint16_t                      s_order[kBeam ? 1 : 1024]; // pool order of the rays (p.ray_order)
    __shared__ __align__(8) uint64_t         bar;
    __shared__ int                           s_tile, s_pool, s_pool2, s_npend, s_adone, s_actdev;
    __shared__ int                           s_ready[kBeam ? kPendCap / 32 : 1]; // entries written, per 32-ray chunk of the queue
    __shared__ uint16_t                      s_pend[kBeam ? kPendCap : 1]; // tile-local indices of the rays pass A left open

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int     R      = p.rays;

    uint8_t  *blob    = smem;
    AgentRec *recs    = reinterpret_cast<AgentRec *>(smem + (kStage ? p.smem_blob_bytes : 0u));
    float2   *dirs    = reinterpret_cast<float2 *>(recs + p.batch_agents); // !kBeam
    // kBeam: per-thread ray parameters and result keys of the group a warp is working on
    __shared__ BeamHot                         s_hot;
    __shared__ unsigned long long              s_tns[3];
    __shared__ __align__(16) float4             s_wray[kBeam ? kBlock : 1];
    __shared__ __align__(8) unsigned long long s_wkey[kBeam ? kBlock : 1];

    if (kStage && tid == 0)
        mbar_init(&bar, 1);
    if (!kBeam)
        for (int i = tid; i < R; i += kBlock)
            s_order[i] = p.ray_order[i];
    __syncthreads();

    int      staged = -1;
    int      n_done = 0; // tiles this CTA has finished (trace slot)
    uint32_t phase  = 0;
    const float inv_R = 1.0f / static_cast<float>(R);
    // the first tile of a CTA is its own index: no trip to the global cursor before any work can start; and when the
    // grid covers every tile (the balanced tiling's single wave, small populations) the cursor is never touched
#ifndef OK_SINGLE_WAVE
#define OK_SINGLE_WAVE 1
#endif
    const bool single_wave = OK_SINGLE_WAVE && p.n_tiles <= static_cast<int>(gridDim.x);
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
        // ---- dynamic tile scheduler: tiles are batches of same-track agents, in agent order.  The next tile is
        // claimed as LATE as possible (after the rays of this batch): claiming it at the start of the batch hides
        // the atomic's latency but turns the schedule static -- measured 0.190 ms vs 0.150 ms per tick ----
        __syncthreads(); // everyone is done with the previous batch and its track; s_tile is published
        const int tile = s_tile;
        if (tile >= p.n_tiles)
            break;
        if (kBeam && p.trace && tid == 0 && n_done < p.trace_tiles)
        {
            unsigned smid;
            asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
            p.trace[(static_cast<size_t>(blockIdx.x) * p.trace_tiles + n_done) * 6] =
                static_cast<unsigned long long>(tile) | (static_cast<unsigned long long>(smid) << 32);
        }
        OK_TRACE(1);
        if (kBeam && p.tile_ns && tid == 0) // thread 0: this tile's cost, for the host's tiling (ok_balance_schedule); kept in shared memory
            s_tns[0] = global_timer();

        Tile     tl;
        TrackRef tr;
        if (p.first && n_done == 0)
        { // (the first tile of a CTA is its block index)
            tl = p.first[tile].tile;
            tr = p.first[tile].ref;
        }
        else
        {
            tl = p.tiles[tile];
            tr = p.tracks[tl.track];
        }
        // the bulk copy of the track runs under phase 1, which reads no staged data; it is awaited before the rays
        const uint8_t *gblob   = p.arena + tr.offset;
        const bool     restage = kStage && tl.track != staged;
        if (restage && tid == 0)
        {
            fence_proxy_async();
            mbar_expect_tx(&bar, tr.bytes);
            tma_bulk_g2s(blob, gblob, tr.bytes, &bar);
        }
        BeamView bv;
        bv.valid = false;
        if (kBeam && tr.has_beam)
            bv = make_beam_view(tr);
        const int       count    = tl.count;
        const int       n_rays   = count * R;
        const float     inv_cnt  = 1.0f / static_cast<float>(count);

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
            recs[tid] = agent_pre(p, gblob, tr, bv, tl.begin + tid, kBeam && n_done > 0 && s_actdev != 0, kActor ? s_actor_act + tid : nullptr);
        if (tid == 0)
        {
            s_pool = 0, s_pool2 = 0, s_npend = 0, s_adone = 0;
            if (kBeam)
            {
                s_hot.entries = bv.entries, s_hot.chunks = bv.chunks;
                s_hot.bin_scale = bv.bin_scale, s_hot.rb = bv.rb;
                s_hot.nb = bv.nb, s_hot.nb_mask = bv.nb - 1;
            }
        }
        if (kBeam)
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
        if (kBeam && p.tile_ns && tid == 0)
            s_tns[1] = global_timer();
        const uint8_t  *track    = kStage ? blob : gblob; // where this tile reads its track from
        const TrackView tv       = make_view(track);
        const int64_t   ray_base = tl.begin * R; // global index of the batch's first ray
        if (!kBeam)
        {

        // =====================================================================================
        // phase 1b -- one thread per ray: direction (cosf/sinf of CollisionChecker.cu:47-48)
        // =====================================================================================
        for (int q = tid; q < n_rays; q += kBlock)
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
        if (p.raycast_mode == 0)
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
            for (int q = tid; q < n_rays; q += kBlock)
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
        for (int q0 = 0; q0 < n_rays; q0 += kBlock)
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
                float2          hit;
                if (!(rec.flags & kFlagCrashed))
                {
                    const float2 d   = dirs[q];
                    const int    seg = p.hit_seg[gi]; // written in phase 2 by whichever lane cast this ray
                    // min_t of CollisionChecker.cu:49-66: the winner's t by the reference's expression
                    const float t = seg >= 0 ? exact_t(tv.seg[seg], rec.ox, rec.oy, d.x, d.y) : p.sensor_range;
                    p.hit_t[gi]   = t;
                    hit.x         = fadd(rec.ox, fmul(t, d.x));
                    hit.y          = fadd(rec.oy, fmul(t, d.y));
                    reinterpret_cast<float2 *>(p.hit_abs)[gi] = hit;
                }
                else
                    hit = reinterpret_cast<const float2 *>(p.hit_abs)[gi]; // stale hit of a crashed agent
                const float xt = fsub(hit.x, rec.ox), yt = fsub(hit.y, rec.oy);
                float2      rel;
                rel.x = fsub(fmul(xt, rec.rc), fmul(yt, rec.rs));
                rel.y = fadd(fmul(xt, rec.rs), fmul(yt, rec.rc));
                sq    = fadd(fmul(rel.x, rel.x), fmul(rel.y, rel.y));
                reinterpret_cast<float2 *>(p.hit_rel)[gi] = rel;
                const float ob = __fdiv_rn(__fsqrt_rn(sq), p.sensor_range);
                p.obs[gi]      = ob;
                if (p.host_obs)
                    p.host_obs[gi] = ob;
                if (p.host_obs_q16)
                    p.host_obs_q16[gi] = static_cast<uint16_t>(obs_q16(ob));
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
        } // !kBeam
        else
        {
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
            // claim the next batch now: late enough to keep the schedule dynamic (see the loop top), early enough
            // for the atomic's latency to hide behind the other warps' last groups and phase 4
            if (tid == 0)
            {
                s_tile = single_wave ? p.n_tiles : static_cast<int>(gridDim.x) + atomicAdd(p.sched, 1); // every thread read the old value before phase 1
                if (p.act_ready)
                { // have the staged actions arrived?  (Long since, normally; if not, the next tile reads the mapping.)
                    uint32_t c;
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(c) : "l"(p.act_ready) : "memory");
                    s_actdev = static_cast<int32_t>(c - p.act_ready_target) >= 0;
                }
            }
        }
        __syncthreads();
        OK_TRACE(4);
        if (kBeam && p.tile_ns && tid == 0)
            s_tns[2] = global_timer();
        if (kBeam && p.tile_flag)
        { // (every thread's stores of this tile happened before the barrier above; the fence makes them visible device-wide
          // before the flag, PTX fences being cumulative)
            if (tid == 0)
            {
                __threadfence();
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.tile_flag + tile), "r"(p.flag_epoch) : "memory");
            }
        }
        else if (kBeam && p.host_obs)
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
        else if (kBeam && p.host_obs_q16)
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
        if (kBeam && p.stats && tid == 0)
        {
            atomicAdd(p.stats, static_cast<unsigned long long>(n_rays));
            atomicAdd(p.stats + 1, static_cast<unsigned long long>(s_npend));
        }
        if (!kBeam && tid == 0)
            s_tile = single_wave ? p.n_tiles : static_cast<int>(gridDim.x) + atomicAdd(p.sched, 1); // every thread read the old value long ago; visible after the loop-top barrier

        // =====================================================================================
        // phase 4 -- four lanes (small batches) or one thread per agent: crash flag, centre-line search, reward, done
        // =====================================================================================
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
        OK_TRACE(5); // thread 0's own phase 4 (the CTA-wide end is the next tile's start)
        if (kBeam && p.tile_ns && tid == 0)
        {
            const unsigned long long t_end = global_timer(), rays_ns = s_tns[2] - s_tns[1];
            p.tile_ns[2 * tile]     = static_cast<uint32_t>(rays_ns);
            p.tile_ns[2 * tile + 1] = static_cast<uint32_t>((t_end - s_tns[0]) - rays_ns);
        }
        ++n_done;
    }

    // last CTA out re-arms the tile scheduler for the next launch on this stream
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


// Everything below is compiled into ok_capi.cu only.  ok_step_unstaged.cu (-DOK_STEP_KERNEL_ONLY) instantiates the
// unstaged beam kernel in a translation unit of its own: with both shapes in one unit ptxas shares the out-of-line
// device functions between them and the staged kernel lost a third of its speed (0.139 vs 0.095 ms per tick).
#ifndef OK_STEP_KERNEL_ONLY

// Environment::resetAgent (Environment.cpp:79-122) + Agent::reset (Agent.cpp:123-135), one thread
// per request, reading the track blobs from global memory.
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
    const uint8_t    *blob = p.arena + p.tracks[p.track_id[a]].offset;
    const TrackView   tv   = make_view(blob);
    int32_t           pt   = r.pt_idx[k];
    pt                     = min(max(pt, 0), tv.n_pts - 1);
    float sx, sy;
    if (r.lane_alpha)
    { // Environment.cpp:107-114; LI / RI points are the start points of the LI / RI segment chains
        const float   alpha = r.lane_alpha[k];
        const int32_t n     = tv.n_pts;
        float2        l, rr;
        if (pt < n - 1)
        {
            const float4 ls = tv.seg[pt], rs = tv.seg[2 * (n - 1) + pt];
            l = make_float2(ls.x, ls.y), rr = make_float2(rs.x, rs.y);
        }
        else
        { // the last point starts the closure segments
            const float4 ls = tv.seg[4 * (n - 1)], rs = tv.seg[4 * (n - 1) + 1];
            l = make_float2(ls.x, ls.y), rr = make_float2(rs.x, rs.y);
        }
        const float one_minus = fsub(1.0f, alpha);
        sx = fadd(fmul(l.x, alpha), fmul(rr.x, one_minus));
        sy = fadd(fmul(l.y, alpha), fmul(rr.y, one_minus));
    }
    else
    {
        const float2 c = tv.pts[pt];
        sx = c.x, sy = c.y;
    }
    const float off = r.heading_off ? r.heading_off[k] : 0.0f;
    p.x[a] = sx, p.y[a] = sy;
    p.rot[a]       = fadd(tv.headings[pt], off);
    p.accel[a]     = 0.0f;
    p.speed[a]     = 0.0f;
    p.crashed[a]   = 0;
    p.timed_out[a] = 0;
    p.done[a]      = 0;
    p.act_thr[a]   = 0.0f;
    p.act_steer[a] = 0.0f;
    p.reset_pt[a]  = pt;
    p.start_x[a]   = sx;
    p.start_y[a]   = sy;
    float   d2;
    int32_t near  = nearest_index(tv, sx, sy, 0, 1, d2);
    p.prev[a]     = near;
    p.nearest[a]  = near;
    p.fitness[a]  = 0.0f;
    p.reward[a]   = 0.0f;
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

#endif // OK_STEP_KERNEL_ONLY

// the unstaged beam kernel's launcher, occupancy and self-check counter (ok_step_unstaged.cu)
cudaError_t launch_step_unstaged(const StepParams &p, int grid, size_t smem_bytes, cudaStream_t stream);
// ok_step_actor.cu: the unstaged beam kernel with the policy step fused in
cudaError_t launch_step_actor(const StepParams &p, const ActorParams &q, int grid, size_t smem_bytes, cudaStream_t stream);
cudaError_t arm_step_actor(int smem_optin, int *max_dynamic);
cudaError_t occupancy_step_unstaged(size_t smem_bytes, int *ctas_per_sm);
cudaError_t violations_step_unstaged(unsigned long long *count);

} // namespace ok
