// ok_device.cuh -- device code shared by the step kernels (ok_step.cuh) and the auxiliary kernels (ok_kernels.cuh): the
// kernels' parameters, the staged track's layout, TMA and shared-memory helpers, the ray x segment test and the uniform-grid
// walk, the centre-line search, the per-agent phases 1 and 4 (agent_pre / agent_post), a ray's outputs (finish_ray) and the
// PPO racers' policy step (actor_agent).
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
static __device__ unsigned long long g_violations = 0; // one per translation unit: each step kernel's unit reports its own
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
// its ray pulls the next one from a CTA-wide pool (see grid_step_kernel, phase 2).
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

// ok_step_host_q16's fixed point: round-to-nearest-even of clamp(obs, 0, 1) * 65535 (a NaN becomes 0)
__device__ __forceinline__ uint32_t obs_q16(const float ob)
{
    return __float2uint_rn(fmul(fminf(fmaxf(ob, 0.0f), 1.0f), 65535.0f));
}

// hit point, unpack (CollisionChecker.cu:68-69,152-165) and the per-ray outputs of ray `gi`, whose nearest
// segment is `seg` (-1 = none); returns the squared norm of the relative hit
// t_known != 0: the winner's exact t is already at hand (the beam key holds it; a zero is recomputed because the
// key does not keep its sign)
// kGrid (the grid kernel's phase 3): phase 2 has already stored the hit index, and the per-ray host mirrors are stored
// here; the beam kernel stores the index here and copies a whole tile's observations to the host at once (its tile flush)
template <bool kGrid, typename Rec>
__device__ __forceinline__ float finish_ray(const StepParams &p, const float4 *segs, const Rec &rec, const int64_t gi,
                                            const float dx, const float dy, const int seg, const float t_known = 0.0f)
{
    float2 hit;
    if (!(rec.flags & kFlagCrashed))
    {
        // min_t of CollisionChecker.cu:49-66: the winner's t by the reference's expression
        const float t = seg >= 0 ? (t_known != 0.0f ? t_known : exact_t(segs[seg], rec.ox, rec.oy, dx, dy)) : p.sensor_range;
        if (!kGrid)
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
    if (kGrid && p.host_obs)
        p.host_obs[gi] = ob;
    if (kGrid && p.host_obs_q16)
        p.host_obs_q16[gi] = static_cast<uint16_t>(obs_q16(ob));
    return sq;
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

} // namespace ok
