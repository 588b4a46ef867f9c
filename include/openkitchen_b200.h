/*
 * openkitchen_b200.h -- C ABI of the B200-native batched step loop for OpenKitchen's racing
 * environment.  This is the drop-in boundary: plain pointers and sizes, no C++/torch types.
 *
 * The reference has no FFI layer; its seam is the C++ class surface of Environment/ and the
 * pybind module.  Each entry point below names the reference interface it replaces (file:line
 * relative to the reference repo root).  The C++ shim (openkitchen_b200/shim/) and the pybind
 * module (openkitchen_b200/pybind/) are written on top of exactly these functions; see
 * INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 (OK_SUCCESS) or a negative OkStatus; nothing throws or aborts
 *     across the ABI; ok_last_error() returns a thread-local message for the last failure;
 *   - `stream` arguments are cudaStream_t passed as void* (NULL = the legacy default stream);
 *     launches are asynchronous on that stream and never synchronise the device;
 *   - pointers named d_* are DEVICE pointers, h_* are HOST pointers;
 *   - agent buffers are owned by the OkEnv and stay valid until ok_alloc_agents is called again
 *     or the env is destroyed (borrowed by callers -- this is what DLPack exports);
 *   - one OkEnv per GPU; an env is thread-compatible (external synchronisation per env).
 */
#ifndef OPENKITCHEN_B200_H
#define OPENKITCHEN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OK_ABI_VERSION 2

typedef enum OkStatus {
    OK_SUCCESS            = 0,
    OK_ERR_INVALID_ARG    = -1,
    OK_ERR_CUDA           = -2,
    OK_ERR_IO             = -3,
    OK_ERR_STATE          = -4, /* e.g. stepping before ok_alloc_agents */
    OK_ERR_CAPACITY       = -5, /* a track does not fit the shared-memory staging area */
    OK_ERR_NO_DEVICE      = -6
} OkStatus;

/* Agent::MovementMode, Environment/Agent.h:20-25 (MANUAL is keyboard input: not supported) */
typedef enum OkMovementMode { OK_MOVE_VELOCITY = 0, OK_MOVE_ACCELERATION = 1 } OkMovementMode;

/* App-side progress/reward definitions (SURVEY.md section 8a row R) */
typedef enum OkRewardMode {
    OK_REWARD_NONE           = 0,
    OK_REWARD_Q_PROGRESS     = 1, /* RLRacers/Q_Learning/QAgent.hpp:150-168 */
    OK_REWARD_CMAES_PROGRESS = 2, /* CovarianceMatrixAdaptationEvolution/main_eigen.cpp:147-163 */
    OK_REWARD_CONSTANT       = 3, /* RLRacers/PPO/ppo_sim.cpp:76 */
    OK_REWARD_DISPLACEMENT   = 4, /* RLRacers/ReinforceContinuous/reinforce_sim.cpp:59-73 */
    OK_REWARD_MIN_RAY        = 5, /* RLRacers/Deep_Q_Learning/DQAgent.hpp:161-180 */
    OK_REWARD_TRACK_INDEX    = 6, /* EvolutionaryRacer/MiscUtils.hpp:64-71 */
    OK_REWARD_LANE_CENTER    = 7  /* WorldModelVaeRnn/main.cpp:336-342 */
} OkRewardMode;

typedef enum OkRaycastMode {
    OK_RAYCAST_GRID  = 0, /* uniform-grid broadphase: DDA walk over 8 px cells */
    OK_RAYCAST_BRUTE = 1, /* every ray x every segment, the reference's loop (CollisionChecker.cu:51-66) */
    OK_RAYCAST_BEAM  = 2  /* precomputed (start cell, direction bin) candidate lists, grid walk only for the rays a
                             list cannot decide; same results as the two modes above */
} OkRaycastMode;

/* Device buffers exported by ok_get_buffer.  N = agents, R = rays per agent. */
typedef enum OkBuffer {
    OK_BUF_POS_X = 0,    /* f32[N]     Agent::pos_.x                         Agent.h:56 */
    OK_BUF_POS_Y,        /* f32[N]     Agent::pos_.y */
    OK_BUF_ROT,          /* f32[N]     Agent::rot_ (degrees, never wrapped)  Agent.h:59 */
    OK_BUF_SPEED,        /* f32[N]     Agent::speed_                         Agent.h:57 */
    OK_BUF_ACCEL,        /* f32[N]     Agent::acceleration_                  Agent.h:58 */
    OK_BUF_ACT_THROTTLE, /* f32[N]     Agent::current_action_.throttle_delta Agent.h:78 */
    OK_BUF_ACT_STEER,    /* f32[N]     Agent::current_action_.steering_delta */
    OK_BUF_CRASHED,      /* u8[N]      Agent::crashed_                       Agent.h:72 */
    OK_BUF_TIMED_OUT,    /* u8[N]      Agent::timed_out_                     Agent.h:74 */
    OK_BUF_DONE,         /* u8[N]      Agent::isDone()                       Agent.cpp:138-144 */
    OK_BUF_SS_CTR,       /* u32[N]     DisplacementStats::displacement_ctr   Environment.h:23 */
    OK_BUF_SS_X,         /* f32[N]     DisplacementStats::init_pos.x         Environment.h:25 */
    OK_BUF_SS_Y,         /* f32[N]     DisplacementStats::init_pos.y */
    OK_BUF_TRACK_ID,     /* i32[N]     which track the agent drives on */
    OK_BUF_HIT_ABS,      /* f32[N,R,2] Ray_::hit_x/hit_y (window coords)     Typedefs.h:96-97 */
    OK_BUF_HIT_REL,      /* f32[N,R,2] Agent::sensor_hits_                   Agent.h:76 */
    OK_BUF_OBS,          /* f32[N,R]   sensor_hits_[i].norm()/sensor_range   PPOAgent.hpp:68-76 */
    OK_BUF_HIT_SEG,      /* i32[N,R]   index of the hit segment in TrackSegments order, -1 = none */
    OK_BUF_HIT_T,        /* f32[N,R]   ray parameter of the hit (min_t of CollisionChecker.cu:49) */
    OK_BUF_MIN_DIST2,    /* f32[N]     min_dist2 of CollisionChecker.cu:150 */
    OK_BUF_NEAREST_IDX,  /* i32[N]     RaceTrack::findNearestTrackIndexBruteForce(pos_) */
    OK_BUF_PREV_IDX,     /* i32[N]     prev_track_idx_ of the progress rewards */
    OK_BUF_REWARD,       /* f32[N]     per-tick reward of OkConfig::reward_mode */
    OK_BUF_FITNESS,      /* f32[N]     accumulated fitness (CMA-ES / lane-centre modes) */
    OK_BUF_RESET_PT,     /* i32[N]     centre-line index of the agent's last reset */
    OK_BUF_START_X,      /* f32[N]     pose at the start of the episode */
    OK_BUF_START_Y,      /* f32[N] */
    OK_BUF_COUNT
} OkBuffer;

typedef enum OkDType { OK_DTYPE_F32 = 0, OK_DTYPE_I32 = 1, OK_DTYPE_U32 = 2, OK_DTYPE_U8 = 3 } OkDType;

/* Track geometry arrays readable through ok_track_copy (host side, reference layout). */
typedef enum OkTrackArray {
    OK_TRACK_X = 0,     /* f32[P]   RaceTrack::track_data_points_.x_m (after fit-to-window) */
    OK_TRACK_Y,         /* f32[P] */
    OK_TRACK_W_RIGHT,   /* f32[P]   w_tr_right_m (clamped, scaled) */
    OK_TRACK_W_LEFT,    /* f32[P] */
    OK_TRACK_HEADING,   /* f32[P]   RaceTrack::headings_ (degrees) */
    OK_TRACK_LEFT_INNER,  /* f32[P,2] RaceTrack::left_bound_inner_ */
    OK_TRACK_LEFT_OUTER,  /* f32[P,2] */
    OK_TRACK_RIGHT_INNER, /* f32[P,2] */
    OK_TRACK_RIGHT_OUTER, /* f32[P,2] */
    OK_TRACK_SEGMENTS     /* f32[S,4] Segment2d in TrackSegments order, S = 4(P-1)+4 */
} OkTrackArray;

/* Constants the reference bakes in at compile time; defaults = reference values. */
typedef struct OkConfig {
    int32_t  device;               /* CUDA device ordinal */
    int32_t  movement_mode;        /* OkMovementMode; Agent.h:80 default VELOCITY */
    int32_t  reward_mode;          /* OkRewardMode */
    int32_t  raycast_mode;         /* OkRaycastMode */
    int32_t  auto_reset;           /* !=0: a crashed agent is reset at the start of the next step
                                      (GuidedCostLearning/test.cpp:102-111) to centre-line index
                                      (last_reset + auto_reset_stride) mod P, with a zero action; with reset
                                      draws on (ok_set_reset_draws) it is a drawn reset instead; with lap
                                      accounting on (ok_set_laps) a completed agent is reset too */
    int32_t  auto_reset_stride;    /* 97 */
    float    sensor_range;         /* Agent::kSensorRange 200        Agent.h:10 */
    float    speed_limit;          /* Agent::kSpeedLimit 100         Agent.h:11 */
    float    dt;                   /* kDt 0.016                      Agent.cpp:84,110 */
    float    collision_dist2;      /* 2.0 (strict <)                 CollisionChecker.cu:167 */
    float    sensor_offset;        /* Agent::sensor_offset_ 0        Agent.h:61 */
    uint32_t standstill_period;    /* DisplacementStats::kPeriod 200 Environment.h:19 */
    float    standstill_threshold; /* kDisplamentThreshold 20        Environment.h:20 */
    float    grid_cell;            /* broadphase cell size in px (8) */
    float    beam_cell;            /* OK_RAYCAST_BEAM: start-cell size in px (2); 0 = default */
    int32_t  beam_bins;            /* OK_RAYCAST_BEAM: direction bins, a power of two (256); 0 = default.  A track
                                      whose table would pass 4 GB (1 px x 1,024 bins on some tracks) fails at table
                                      time (ok_alloc_agents, ok_beam_lookup) with OK_ERR_INVALID_ARG */
    uint64_t agent_id_base;        /* global id of this env's agent 0 (multi-GPU: the first agent of the rank's slice).
                                      The synthetic Philox action stream is keyed by (agent_id_base + a, step), so a
                                      shard reproduces, bit for bit, its slice of the unsharded population */
} OkConfig;

typedef struct OkTrackInfo {
    int32_t n_points;
    int32_t n_segments;
    int32_t grid_nx, grid_ny;
    int32_t grid_items;   /* total (cell, segment) registrations */
    int32_t blob_bytes;   /* bytes staged into shared memory for this track */
    float   grid_x0, grid_y0, grid_cell;
} OkTrackInfo;

typedef struct OkEnv OkEnv;

/* ---- lifetime ------------------------------------------------------------------------------ */
int         ok_abi_version(void);
const char *ok_last_error(void);
void        ok_config_default(OkConfig *cfg);
/* Environment::Environment (Environment.cpp:42-62) minus raylib/visualizer/screen grabber. */
int  ok_create(const OkConfig *cfg, OkEnv **out);
void ok_destroy(OkEnv *env);
/* change the per-tick constants of a live env (everything except `device`, `grid_cell` and `beam_*`, which are fixed
 * at creation): e.g. Agent::setMovementMode (Agent.h:46-49), the reward definition, auto-reset */
int  ok_update_config(OkEnv *env, const OkConfig *cfg);
int  ok_get_config(const OkEnv *env, OkConfig *out);

/* ---- tracks: RaceTrack ctor chain (RaceTrack.cpp:3-14,127-307) + TrackSegments (TrackSegments.cu:6-76)
 *      + broadphase grid build + device upload. Must precede ok_alloc_agents. -------------------- */
/* the four raw CSV columns x_m,y_m,w_tr_right_m,w_tr_left_m (before clamp/scale) */
int ok_add_track(OkEnv *env, const float *h_x_m, const float *h_y_m, const float *h_w_right, const float *h_w_left,
                 int32_t n_points, int32_t *track_id_out);
/* RaceTrack::getTrackDataFromCsv, RaceTrack.cpp:127-164 */
int ok_load_track_csv(OkEnv *env, const char *path, int32_t *track_id_out);
int ok_num_tracks(const OkEnv *env);
int ok_track_info(const OkEnv *env, int32_t track_id, OkTrackInfo *out);
/* copies min(count, available) elements of the named array to h_out; returns elements available */
int64_t ok_track_copy(const OkEnv *env, int32_t track_id, int32_t which /*OkTrackArray*/, float *h_out, int64_t count);

/* ---- agents -------------------------------------------------------------------------------- */
/* replaces `std::vector<Agent*>` + CollisionChecker ctor (CollisionChecker.cu:76-86).  All agents
 * have `rays` rays (the reference assumes agents[0]'s count, CollisionChecker.cu:82) with angles
 * h_ray_deg[rays] relative to heading (Agent::sensor_ray_angles_).  h_track_id may be NULL (all on
 * track 0).  Every agent starts reset at RaceTrack::kStartingIdx (RaceTrack.h:18). Agents on the
 * same track should be contiguous for best performance. */
int     ok_alloc_agents(OkEnv *env, int64_t n_agents, int32_t rays, const float *h_ray_deg, const int32_t *h_track_id);
int64_t ok_num_agents(const OkEnv *env);
int32_t ok_num_rays(const OkEnv *env);

/* Environment::resetAgent (Environment.cpp:79-122) + Agent::reset (Agent.cpp:123-135) with the
 * random draws made explicit: agent d_agent_idx[k] (NULL = k) goes to centre-line index d_pt_idx[k];
 * d_lane_alpha (nullable) = the lane lerp alpha of Environment.cpp:107-114; d_heading_off (nullable)
 * = the heading offset of Environment.cpp:88-101.  Device pointers, asynchronous on `stream`. */
int ok_reset_agents(OkEnv *env, const int64_t *d_agent_idx, const int32_t *d_pt_idx, const float *d_lane_alpha,
                    const float *d_heading_off, int64_t n, void *stream);
/* same with HOST arrays, staged through the env's staging buffer (kept at its largest size until ok_destroy);
 * synchronises `stream` before it returns, on error too */
int ok_reset_agents_host(OkEnv *env, const int64_t *h_agent_idx, const int32_t *h_pt_idx, const float *h_lane_alpha,
                         const float *h_heading_off, int64_t n, void *stream);

/* Reset draws: Environment::resetAgent's random point, lane and heading (Environment.cpp:76-122) from a counter-based
 * stream keyed by device state, so that they run inside the step kernel (auto-reset), inside a CUDA graph, and come out the
 * same whatever the tiling, the kernel shape or the sharding.
 *
 * Every agent a has a device counter k[a] (u32, zero after ok_alloc_agents; ok_reset_draw_counts).  A DRAWN reset of a:
 *   1. o[0..3] = Philox4x32-10(counter = (lo32(id), hi32(id), k[a], 0), key = (seed, 0x525354 "RST")), id = agent_id_base + a
 *      (the key's second word keeps this stream apart from the action stream, 0, and the PPO stream, 0x50504f);
 *   2. U(o, m) = (uint32_t)(((uint64_t)o * m) >> 32): U{0..m-1}, each value's probability off by at most m / 2^32;
 *   3. centre-line index pt = U(o[0], P) with OK_RESET_DRAW_POINT; otherwise an auto-reset keeps the stride rule of
 *      OkConfig::auto_reset and an explicit reset uses RaceTrack::kStartingIdx (3, clamped to P - 1);
 *   4. with OK_RESET_DRAW_LANE the lane lerp alpha = (float)(10 + U(o[1], 81)) / 100.0f, correctly rounded
 *      (Environment.cpp:107-114); without it the agent starts on the centre line;
 *   5. with OK_RESET_DRAW_HEADING the heading offset off = s * (float)(45 + U(o[2], 46)), s = -1 for even k[a] and +1 for
 *      odd (the reference's alternating sign, Environment.cpp:88-101, per agent); without it off = 0;
 *   6. the agent is reset exactly as ok_reset_agents resets it with (pt, alpha, off), and k[a] += 1.
 * Resets that are not drawn (ok_reset_agents, the stride auto-reset with draws off) never touch k.  Draws are off by default. */
#define OK_RESET_DRAW_POINT   1
#define OK_RESET_DRAW_LANE    2
#define OK_RESET_DRAW_HEADING 4
typedef struct OkResetDraws {
    uint32_t seed;
    int32_t  flags; /* OK_RESET_DRAW_*; 0 = off */
} OkResetDraws;
/* d NULL = off; unknown flag bits: OK_ERR_INVALID_ARG.  With OkConfig::auto_reset != 0 and flags != 0, the auto-reset at the
 * start of a tick is a drawn reset (its tick still runs with a zero action) in every step entry point.  The settings are
 * read when a launch is enqueued: a CUDA graph keeps the settings it was captured with, and its replays continue the
 * stream, because the counters live on the device. */
int ok_set_reset_draws(OkEnv *env, const OkResetDraws *d);
int ok_get_reset_draws(const OkEnv *env, OkResetDraws *out);
/* a drawn reset of: the n agents d_agent_idx[0..n) (distinct indices) | every agent with d_mask[a] != 0 (u8[N], e.g. the
 * OK_BUF_DONE buffer) | every agent (both NULL).  With a mask or for all agents n must be ok_num_agents; passing both is
 * OK_ERR_INVALID_ARG.  With draws off the agents go to kStartingIdx and their counters still advance.  Device pointers;
 * asynchronous on `stream`, no host synchronisation: it can be captured into a CUDA graph. */
int ok_reset_agents_drawn(OkEnv *env, const int64_t *d_agent_idx, const uint8_t *d_mask, int64_t n, void *stream);
/* same with HOST arrays, staged through the env's staging buffer; synchronises `stream` before it returns, on error too */
int ok_reset_agents_drawn_host(OkEnv *env, const int64_t *h_agent_idx, const uint8_t *h_mask, int64_t n, void *stream);
/* the device counters k: u32[ok_num_agents], owned by the env like the agent buffers; writable (to restart or move a
 * stream) */
int ok_reset_draw_counts(OkEnv *env, uint32_t **d_counts);

/* Lap accounting: centre-line progress, laps and lap times per agent, and Agent::completed_ (Agent.h:73, ORed into
 * Agent::isDone, Agent.cpp:138-144) at a target lap count, inside the step.  A lap is P centre-line points (P = the
 * agent's track's point count) travelled from wherever the episode started, not a crossing of index 0.
 *
 * Every agent a has device state (zero after ok_alloc_agents allocates it, then restarted by its initial reset):
 *   lap_idx[a]   i32  the centre-line index at which progress was last measured
 *   progress[a]  i32  signed centre-line points travelled since the last restart
 *   laps[a]      i32  laps completed
 *   ticks[a]     u32  ticks the agent moved since the last restart
 *   lap_start[a] u32  the value of ticks when the current lap began
 *   last_lap[a]  u32  ticks of the last completed lap; 0 = none yet
 *   completed[a] u8   Agent::completed_
 * 1. RESTART of a: lap_idx = the nearest centre-line index of the agent's pose (RaceTrack::findNearestTrackIndexBruteForce,
 *    the value a reset writes to OK_BUF_PREV_IDX), every other field 0.  It happens at every reset of a by ok_reset_agents[_host],
 *    ok_reset_agents_drawn[_host] and ok_alloc_agents (with accounting on or off), at the auto-reset inside a tick with
 *    accounting on, and for every agent when ok_set_laps switches accounting from off to on.
 * 2. A TICK with accounting on, for every agent that moves in it (not crashed at the start of the tick, after the tick's
 *    auto-reset: the agents Environment.cpp:128-143 moves, one that crashes in this tick included), after the move:
 *    n = the nearest index of the new pose (written to OK_BUF_NEAREST_IDX, which is then updated every tick in every
 *    reward mode); d = n - lap_idx; if 2d > P then d -= P, else if 2d <= -P then d += P (so d lies in (-P/2, P/2]);
 *    progress += d; lap_idx = n; ticks += 1;
 *    if (int64)progress >= ((int64)laps + 1) * P: laps += 1, last_lap = ticks - lap_start, lap_start = ticks;
 *    if target > 0 and laps >= target: completed = 1.
 *    (Arithmetic on the 32-bit fields wraps in two's complement.)  At most one lap completes per tick; driving backwards
 *    lowers progress but never laps, and a lap regained after a reversal counts once progress passes the next multiple of P.
 *    OK_BUF_DONE = crashed || completed for every agent, and so is ok_step_host[_q16]'s host done mirror.
 * 3. A completed agent keeps driving and sensing (Environment::step moves every agent whose crashed_ is clear); completed
 *    stays set until the next restart.
 * 4. With OkConfig::auto_reset and accounting on, the auto-reset at the start of a tick resets every agent with crashed ||
 *    completed, by the same rule as for a crashed agent (the stride rule, or a drawn reset with reset draws on), and
 *    restarts its lap state.
 * 5. With accounting off, the tick neither reads nor writes lap state (its auto-reset does not restart it either: the
 *    switch to on restarts every agent); OK_BUF_DONE = crashed as before.  ok_cast_rays, which moves nothing, never
 *    touches it, and writes OK_BUF_DONE = crashed as it always has.
 * Accounting is off by default. */
typedef struct OkLaps {
    int32_t enabled; /* != 0: on */
    int32_t target;  /* laps at which completed is set; 0 = never */
} OkLaps;
/* l NULL = off; a negative target is OK_ERR_INVALID_ARG.  A switch from off to on enqueues the restart of every agent on
 * `stream` (asynchronous, no host synchronisation).  The settings are read when a step launch is enqueued: a CUDA graph
 * keeps the settings it was captured with, and its replays continue the lap state, which lives on the device. */
int ok_set_laps(OkEnv *env, const OkLaps *l, void *stream);
int ok_get_laps(const OkEnv *env, OkLaps *out);
typedef struct OkLapBuffers {
    int32_t  *lap_idx, *progress, *laps;
    uint32_t *ticks, *lap_start, *last_lap;
    uint8_t  *completed;
} OkLapBuffers;
/* device pointers to the seven arrays, [ok_num_agents] each, owned by the env like the agent buffers; writable (to plant
 * state) */
int ok_lap_buffers(OkEnv *env, OkLapBuffers *out);

/* Races: the cars of a group see each other in the lidar and crash on contact, in a pass after the tick.  The reference's
 * co-located agents never see each other; races depart from it on purpose, and only while they are on.
 *   - GROUPS.  Agent a (local index) belongs to race a / group: consecutive agents, the last race may be short.  Every agent
 *     is a car body, a disc of radius `radius` around (pos_x, pos_y), crashed or not.  Agent j is an OPPONENT of agent i when
 *     they are in the same race, on the same track_id, and j != i: cars on different tracks never meet.  For a sharded
 *     population, a shard's races equal the unsharded ones when its first agent (OkConfig::agent_id_base) is a multiple of
 *     `group`.
 *   - THE PASS runs after the step kernel of every call that casts the agents' rays: ok_cast_rays, ok_launch_step, every tick
 *     of ok_launch_steps_random and ok_ppo_actor_step (fused or as two launches), on the same stream.  It reads the tick's
 *     outputs and the poses.  Every agent i whose crashed flag is clear when the pass starts is processed; the others are
 *     left as they are.
 *   - SENSING (OK_RACE_SENSE).  For each ray r of i, (ox, oy) = the lidar origin and (dx, dy) = the ray's direction exactly
 *     as the tick computed them (the sensor-offset origin; the device sincosf of kDeg2Rad * (rot + ray_deg[r])).  For each
 *     opponent j, in binary32, every operation correctly rounded in this order, no contraction:
 *       wx = x_j - ox;  wy = y_j - oy;  b = wx*dx + wy*dy;  c = (wx*wx + wy*wy) - radius*radius;
 *     if c <= 0 then t = 0; else if b > 0 and q = b*b - c >= 0 then t = max(b - sqrt(q), 0); else j is missed.  j is hit
 *     when t <= sensor_range (a comparison with NaN is false: a NaN pose neither hits nor is hit).  The nearest car is the
 *     smallest t, the lowest j among ties.  It replaces the track hit only if t < hit_t[i,r] (strictly); then hit_t = t,
 *     hit_abs = (ox + t*dx, oy + t*dy), hit_seg = -1, hit_car[i,r] = j, and hit_rel and obs follow the unpack
 *     (CollisionChecker.cu:152-165) exactly as the tick writes them.  Rays whose track hit stands get hit_car = -1.  If a ray
 *     was replaced, min_dist2 is the unpack's minimum over all R rays again, and the agent crashes if it is < collision_dist2:
 *     the reference's lidar-derived crash rule applied to what the lidar now sees.
 *   - CONTACT (OK_RACE_CONTACT).  i crashes if some opponent j has (x_i - x_j)^2 + (y_i - y_j)^2 < (radius + radius)^2, in
 *     binary32 in that order (pos_, not the sensor origin).  The rule is symmetric.
 *   - A CRASH BY THE PASS writes crashed = 1, done = 1 and contact[i] = 1.  contact is 0 for every other agent and is
 *     rewritten by every pass.  timed_out, reward, fitness, prev_idx, nearest_idx and the lap state are never touched: the
 *     tick's reward stays the track-only reward.  The crash takes effect from the next tick: the car does not move, the
 *     auto-reset (stride or drawn) resets it, lap accounting restarts it.  A trainer that wants a penalty writes
 *     reward[contact] = ... itself.
 *   - ok_step_host, ok_step_host_q16 and ok_step_packed deliver their results from inside the step kernel and return
 *     OK_ERR_STATE while races are on.  ok_lidar_query, ok_bev_query and the resets do not see cars.  The settings are read
 *     when a launch is enqueued: a CUDA graph keeps the settings it was captured with.
 * Races are off by default. */
#define OK_RACE_SENSE   1
#define OK_RACE_CONTACT 2
typedef struct OkRaces {
    int32_t group;  /* agents per race, 2..1024; 0 = off */
    int32_t flags;  /* a non-empty set of OK_RACE_SENSE | OK_RACE_CONTACT */
    float   radius; /* car body radius in px, finite and > 0 */
} OkRaces;
/* r NULL or r->group == 0: off.  Otherwise a group outside 2..1024, a radius that is not finite and > 0, or flags that are
 * not a non-empty subset of the two: OK_ERR_INVALID_ARG.  Switching races on with agents allocated allocates the race
 * buffers (synchronously) if they do not exist yet. */
int ok_set_races(OkEnv *env, const OkRaces *r);
int ok_get_races(const OkEnv *env, OkRaces *out);
typedef struct OkRaceBuffers {
    int32_t *hit_car; /* i32[N,R]: the opponent a ray hit, -1 = none (also right after allocation) */
    uint8_t *contact; /* u8[N]: 1 = crashed by the last pass */
} OkRaceBuffers;
/* device pointers, owned by the env like the agent buffers: allocated when races are first switched on, or by
 * ok_alloc_agents while races are on.  Before that: OK_ERR_STATE. */
int ok_race_buffers(OkEnv *env, OkRaceBuffers *out);

/* ---- the tick ------------------------------------------------------------------------------ */
/* CollisionChecker::checkCollision (CollisionChecker.cu:96-100,113-174): lidar + crash flag on the
 * current poses, no movement. */
int ok_cast_rays(OkEnv *env, void *stream);
/* Environment::step stages 1-2 (Environment.cpp:125-146) + the app-side progress/reward/done:
 * one fused kernel.  d_act_* (nullable) are copied into the ACT_* buffers first; NULL = step with
 * the actions already stored there (what Agent::updateAction wrote). */
int ok_launch_step(OkEnv *env, const float *d_act_throttle, const float *d_act_steer, void *stream);
/* k consecutive ticks whose actions come from the counter-based Philox4x32-10 stream of
 * SURVEY.md 8(d) (key = seed, counter = (agent, first_step + i)), generated inside the step kernel. */
int ok_launch_steps_random(OkEnv *env, uint64_t first_step, int32_t k, uint32_t seed, void *stream);
/* write the Philox actions for `step` into the ACT_* buffers without stepping */
int ok_fill_random_actions(OkEnv *env, uint64_t step, uint32_t seed, void *stream);

/* Track queries for arbitrary points (the app-side reward code of WorldModelVaeRnn/main.cpp:336-337 and every
 * progress reward): RaceTrack::findNearestTrackIndexBruteForce (RaceTrack.cpp:16-31), getDistanceToLaneCenter
 * (RaceTrack.cpp:53-72) and getNearestDistanceToTrackBoundary (RaceTrack.cpp:33-51) for n points.  d_x, d_y f32[n];
 * d_track_id i32[n] or NULL (track 0); each output is nullable.  One warp per query; asynchronous on `stream`. */
int ok_track_query(OkEnv *env, const float *d_x, const float *d_y, const int32_t *d_track_id, int64_t n,
                   int32_t *d_nearest_idx, float *d_dist_lane_center, float *d_dist_boundary, void *stream);
/* same with HOST arrays, staged through the env's staging buffer (kept at its largest size until ok_destroy);
 * synchronises `stream` before it returns, on error too */
int ok_track_query_host(OkEnv *env, const float *h_x, const float *h_y, const int32_t *h_track_id, int64_t n,
                        int32_t *h_nearest_idx, float *h_dist_lane_center, float *h_dist_boundary, void *stream);

/* Lidar scans at arbitrary poses, with no agent state read or written (CollisionChecker::checkCollision's pack + kernel
 * + unpack, CollisionChecker.cu:115-172, for poses that are not agents).  Pose k = (x[k], y[k], rot[k]) on track
 * track_id[k] (NULL = track 0; out-of-range ids are clamped as in ok_track_query) casts the fan ray_deg[rays], angles in
 * degrees relative to the heading, 1 <= rays <= 1024.  ray_deg NULL = the env's fan from ok_alloc_agents, and then rays
 * must be ok_num_rays(env).  Uses the env's live OkConfig (sensor_range, sensor_offset, collision_dist2, raycast_mode);
 * every output is bit for bit what ok_cast_rays writes for an agent at that pose whose crash flag is clear, in the layout
 * of the agent buffer of the same name; every output is nullable.  crashed is the strict test min_dist2 <
 * collision_dist2.  Needs tracks only, not agents.  The first call of an env may build the track arena (in beam mode also
 * the device tables) synchronously; if that is still to do while `stream` is capturing, the call fails with OK_ERR_STATE:
 * call once outside the capture, later calls can be captured.  n == 0 is a no-op. */
typedef struct OkLidarQuery {
    const float   *x, *y, *rot;        /* f32[n]: Agent::pos_, rot_ (degrees) */
    const int32_t *track_id;           /* i32[n] or NULL */
    int64_t        n;
    const float   *ray_deg;            /* f32[rays] or NULL */
    int32_t        rays, reserved;
    float         *hit_abs, *hit_rel;  /* f32[n,R,2]: OK_BUF_HIT_ABS, OK_BUF_HIT_REL */
    float         *obs, *hit_t;        /* f32[n,R] */
    int32_t       *hit_seg;            /* i32[n,R], -1 = none */
    float         *min_dist2;          /* f32[n] */
    uint8_t       *crashed;            /* u8[n]: min_dist2 < collision_dist2 */
} OkLidarQuery;
/* device pointers; asynchronous on `stream` */
int ok_lidar_query(OkEnv *env, const OkLidarQuery *q, void *stream);
/* the same with HOST pointers (ray_deg included), staged through the env's staging buffer (kept at its largest size
 * until ok_destroy); synchronises `stream` before it returns, on error too */
int ok_lidar_query_host(OkEnv *env, const OkLidarQuery *q, void *stream);

/* Bird's-eye-view rasters at arbitrary poses, with no agent state read or written: the observation of the apps that read
 * the screen (ScreenGrabber), as a semantic image with an exact definition instead of raylib's RGB frame.
 * Regions: the four boundary polylines LI, LO, RI, RO (ok_track_copy), each closed by the edge from its last point to its
 * first -- the segments the lidar hits.  inside(L, p) is the even-odd (PNPOLY) rule over the edges (i, j = i - 1 cyclic)
 * of loop L: flip when (y_i > p_y) != (y_j > p_y) and p_x < ((x_j - x_i) * (p_y - y_i)) / (y_j - y_i) + x_i, in binary32,
 * every operation rounded in that order, no contraction.  k(p) = the sum over the four loops; the pixel's class is
 * OK_BEV_LANE for k == 2, OK_BEV_WALL for odd k (the 3 px band between an inner and an outer bound), OK_BEV_OFF for k == 0
 * or 4 (outside the track, or the infield).  Where an offset polyline folds on itself at a tight corner (most tracks have
 * such folds), the even-odd rule decides the class of the small pocket inside the fold; the lidar sees the same segments.
 * Sample points: pose k = (x[k], y[k], rot[k] degrees) on track track_id[k] (NULL = track 0; out-of-range ids are clamped
 * as in ok_track_query); pixel (r, c) of the height x width image is the point
 *   (rs, rc) = sincosf(kDeg2Rad * rot);  f = (0.5f*(H-1) - r) * scale + ahead;  l = (c - 0.5f*(W-1)) * scale;
 *   px = x + (f*rc - l*rs);  py = y + (f*rs + l*rc)
 * in binary32, rounded in that order: row 0 is ahead, column 0 on the agent's left (window y points down, so the right
 * is (-sin, cos), the ray at +90 degrees); rot = -90 gives a crop aligned with the window.  A NaN coordinate is OFF.
 * `scale` is track px per image pixel, `ahead` shifts the image forward.  The position is pos_, without the sensor
 * offset; raycast_mode does not matter.  Needs tracks only, not agents.  The first call after a track was added builds a
 * device table (per track, edge lists over 2 px bands of y) synchronously; if that is still to do while `stream` is
 * capturing, the call fails with OK_ERR_STATE: call once outside the capture, later calls can be captured.  n == 0 is a
 * no-op. */
#define OK_BEV_OFF 0
#define OK_BEV_WALL 1
#define OK_BEV_LANE 2
typedef struct OkBevQuery {
    const float   *x, *y, *rot;  /* f32[n]: Agent::pos_, rot_ (degrees) */
    const int32_t *track_id;     /* i32[n] or NULL (track 0) */
    int64_t        n;
    int32_t        height, width; /* 1..1024 each */
    float          scale, ahead;  /* scale finite and > 0; ahead finite */
    uint8_t       *out;          /* u8[n][height][width], row-major */
} OkBevQuery;
/* device pointers; asynchronous on `stream` */
int ok_bev_query(OkEnv *env, const OkBevQuery *q, void *stream);
/* the same with HOST pointers, staged through the env's staging buffer (kept at its largest size until ok_destroy);
 * synchronises `stream` before it returns, on error too */
int ok_bev_query_host(OkEnv *env, const OkBevQuery *q, void *stream);

/* The EvolutionaryRacer policy for the whole population (SURVEY.md 8f, N2): GeneticAgent::updateAction +
 * Network::infer (EvolutionaryRacer/GeneticAgent.hpp:37-50, Network.hpp:119-155).  Agent i has its own weights
 * d_w1[i] (f32 [R+2][hidden], inputs speed/100, normalizeAngleDeg(rot)/360, hits/200) and d_w2[i] (f32 [hidden][6]);
 * hidden = relu(x W1), out = sigmoid(hidden W2), actions decoded with the 0.5 activation limit into the ACT_*
 * buffers.  hidden <= 32.  One warp per agent; the kernel streams the weights once (HBM bound: 4*(R+2+6)*hidden
 * bytes per agent). */
int ok_genetic_policy(OkEnv *env, const float *d_w1, const float *d_w2, int32_t hidden, void *stream);

/* The CMA-ES racer's policy for the whole population (SURVEY.md 8f, N1): CmaEsAgent::updateAction + Controller::forward
 * (CovarianceMatrixAdaptationEvolution/main_torch.cpp:61-71, Controller.cpp:16-23).  Candidate i evaluates
 * tanh(fc3 tanh(fc2 tanh(fc1 obs_i))) with its OWN flat parameter vector d_params[i] (f32[n_params], torch parameters()
 * order: fc1.weight [16][R], fc1.bias, fc2.weight [8][16], fc2.bias, fc3.weight [1][8], fc3.bias; n_params = 16 R + 169)
 * and writes ACT_THROTTLE = throttle (100), ACT_STEER = steer_scale (5) * output.  hidden must be 16 (main_torch.cpp:19).
 * One warp per agent, weights streamed once: HBM bound at 4 * n_params bytes per agent. */
int ok_cmaes_controller(OkEnv *env, const float *d_params, int32_t n_params, int32_t hidden, float throttle, float steer_scale,
                        void *stream);

/* The PPO racers' policy step for every agent in ONE kernel (SURVEY.md 8f, N3): PPOAgent::updateAction + Actor::forward
 * (RLRacers/PPO/PPOAgent.hpp:79-102, Actor.hpp:9-26): probs = softmax(W2 relu(W1 obs + b1) + b2) clamped to
 * [1e-8, 1 - 1e-8]; an action index drawn with torch::multinomial's distribution (inverse CDF on one uniform per agent:
 * d_uniform[N] if given, else Philox keyed by (agent_id_base + a, step) with `seed`), or the argmax when greedy != 0;
 * log-probability of the choice; (throttle, steering) = d_action_table[action] into the ACT_* buffers
 * (PPOAgent::kActionMap).  Weights are device pointers in torch.nn.Linear layout, shared by all agents: d_w1 [hidden][R],
 * d_b1 [hidden], d_w2 [n_actions][hidden], d_b2 [n_actions]; n_actions <= 8.  Nullable outputs (rows of a rollout
 * buffer): d_action i32[N], d_log_prob f32[N], d_probs f32[N][n_actions], d_obs f32[N][R] (the observation the action
 * was chosen from), d_prev_reward f32[N] / d_prev_done u8[N] (REWARD / DONE of the tick before this call).
 * With d_w1 == NULL only the d_prev_* record is made (the flush after a rollout's last tick). */
typedef struct OkActorIO {
    const float *d_w1, *d_b1, *d_w2, *d_b2;
    int32_t      hidden, n_actions;
    const float *d_action_table;
    const float *d_uniform;
    int32_t      greedy, reserved;
    int32_t     *d_action;
    float       *d_log_prob, *d_probs, *d_obs;
    float       *d_prev_reward;
    uint8_t     *d_prev_done;
} OkActorIO;
int ok_ppo_actor(OkEnv *env, const OkActorIO *io, uint64_t step, uint32_t seed, void *stream);
/* ok_ppo_actor and the tick that consumes its actions (ok_launch_step with the stored actions) as ONE launch: the policy
 * step runs as phase 0 of every tile of the step kernel (ppo_sim.cpp:61-89's updateAction + env.step per tick).  At a few
 * thousand agents a tick is launch-to-completion latency, and two kernels pay it twice.  Same results as the two calls; falls
 * back to them when the env's kernel shape has no fused instantiation (grid / brute-force modes; the staged shapes of
 * populations of 65,536 rays per tick and more, whose tick is not latency). */
int ok_ppo_actor_step(OkEnv *env, const OkActorIO *io, uint64_t step, uint32_t seed, void *stream);
/* ExperienceBuffer::calculateDiscountedRewards (RLRacers/PPO/ExperienceBuffer.hpp:45-62) for all agents: d_rewards
 * f32[steps][N] -> d_out f32[steps][N], ret[t] = r[t] + gamma * ret[t + 1] in binary32 with the reference's operation
 * order; d_done u8[steps][N] (nullable) restarts the sum where an episode ended.  No env needed beyond its device. */
int ok_discounted_returns(OkEnv *env, const float *d_rewards, const uint8_t *d_done, float *d_out, int32_t steps, int64_t n,
                          float gamma, void *stream);

/* End-to-end host call (what the C++ shim's Environment::step and the reference-facing plugin
 * use): H2D of the two action arrays, one tick, D2H of obs / reward / done / crashed (each
 * nullable), then a stream synchronise.  Host buffers should be pinned (ok_host_alloc). */
int ok_step_host(OkEnv *env, const float *h_act_throttle, const float *h_act_steer, float *h_obs, float *h_reward,
                 uint8_t *h_done, void *stream);
/* ok_step_host with the observations as 16-bit fixed point -- OPT-IN AND LOSSY: h_obs_q16[a][r] =
 * round-to-nearest-even(clamp(obs, 0, 1) * 65535), obs being the binary32 value ok_step_host delivers
 * (|error| <= 0.5 / 65535 = 7.7e-6 of the sensor range, 0.0015 px at 200 px).  Half the bytes on the host link, which bounds the
 * end-to-end tick (DESIGN.md 4).  The device-side buffers (OK_BUF_OBS ...) keep the exact values; h_obs_q16 must be
 * pinned.  No counterpart in the reference (its consumers read Agent::sensor_hits_, Agent.h:66, as float). */
int ok_step_host_q16(OkEnv *env, const float *h_act_throttle, const float *h_act_steer, uint16_t *h_obs_q16, float *h_reward,
                     uint8_t *h_done, void *stream);
/* The object-model tick in ONE upload, one launch and two downloads (what the C++ shim's Environment::step and
 * CollisionChecker::checkCollision use; round 1 made ~24 synchronous buffer copies per tick).  The env's first thirteen
 * buffers (OK_BUF_POS_X .. OK_BUF_SS_Y: pose, speed, acceleration, action, flags, standstill record) are adjacent in
 * device memory; h_state is a byte-for-byte host image of that block (layout from ok_packed_layout).  The call copies
 * h_state to the device, runs one tick (move != 0: ok_launch_step with the actions in the block; 0: ok_cast_rays), copies
 * the block back into h_state and HIT_ABS + HIT_REL into h_hits, and synchronises `stream` once.  Pinned buffers
 * (ok_host_alloc) make the three copies asynchronous. */
typedef struct OkPackedLayout {
    size_t state_bytes;      /* bytes of the state block */
    size_t state_offset[13]; /* byte offset of OK_BUF_POS_X ... OK_BUF_SS_Y (enum order) inside it */
    size_t hits_bytes;       /* bytes of the hits block */
    size_t hit_abs_offset, hit_rel_offset;
} OkPackedLayout;
int ok_packed_layout(const OkEnv *env, OkPackedLayout *out);
int ok_step_packed(OkEnv *env, void *h_state, void *h_hits, int32_t move, void *stream);
int ok_host_alloc(void **h_ptr, size_t bytes); /* cudaMallocHost */
int ok_host_free(void *h_ptr);

/* ---- buffers ------------------------------------------------------------------------------- */
/* device pointer, shape (shape[1] = 0 for per-agent vectors; shape[2] = 2 for the xy buffers) and
 * OkDType of an agent buffer: the DLPack export of the Python layer is built from this. */
int ok_get_buffer(OkEnv *env, int32_t which /*OkBuffer*/, void **d_ptr, int64_t shape[3], int32_t *dtype);
/* convenience copies (synchronise `stream`) */
int ok_read_buffer(OkEnv *env, int32_t which, void *h_dst, size_t bytes, void *stream);
int ok_write_buffer(OkEnv *env, int32_t which, const void *h_src, size_t bytes, void *stream);
int ok_sync(OkEnv *env, void *stream);

/* ---- introspection (bench / profiling) ----------------------------------------------------- */
/* Population counters (SURVEY.md 5, metrics: what the reference's apps print per episode -- colony averages, how many
 * agents are still driving -- needs these): agents alive (= not crashed) / crashed / timed out / done in the env's buffers as
 * they are now, counted on the device.  Synchronises `stream`. */
typedef struct OkPopulationCounters {
    uint64_t agents, alive, crashed, timed_out, done;
} OkPopulationCounters;
int ok_population_counters(OkEnv *env, OkPopulationCounters *out, void *stream);
typedef struct OkLaunchStats {
    uint64_t kernel_launches; /* kernels launched by this env since creation */
    int32_t  grid_blocks, block_threads, smem_bytes, tiles;
} OkLaunchStats;
int ok_launch_stats(const OkEnv *env, OkLaunchStats *out);
/* Work counters of the beam kernel (profiling aid, off by default): out[0] = rays cast, out[1] = rays its first pass
 * could not settle from the table entry alone (queued for the second pass), out[2] = rays that fell back to the
 * uniform-grid walk, since the previous call.  Synchronises the device; enable != 0 keeps counting, 0 stops. */
int ok_debug_stats(OkEnv *env, uint64_t out[4], int32_t enable);
/* Index self-checks: a library built with -DOK_CHECKED=1 (tools/checked_build.sh) counts every table row, chunk,
 * segment, ray or agent index that would leave its array; *count is the total since the library was loaded (always 0 for
 * the product build, whose *checks_compiled_in is 0).  Synchronises the device. */
int ok_debug_violations(OkEnv *env, uint64_t *count, int32_t *checks_compiled_in);
/* Timeline of the beam kernel's last launch (profiling aid, off by default): per CTA and per tile it processed, six
 * 64-bit words {tile | smid << 32, then %globaltimer (ns) at: tile start, end of the thread-per-agent phase, end of the
 * first ray pass, end of the second ray pass, end of the reward phase}.  Copies min(words available, capacity_words) to
 * h_out (layout [grid_blocks][tiles_per_cta][6], zero = unused) and returns the count; then re-arms the trace with room
 * for `tiles_per_cta` tiles per CTA (0 = off).  Synchronises the device. */
int64_t ok_debug_trace(OkEnv *env, uint64_t *h_out, int64_t capacity_words, int32_t tiles_per_cta);
/* Feedback tiling of the staged beam kernels.  The kernel leaves every tile's time (ray phase / rest) in a small device
 * buffer; this call synchronises `stream`, reads it and re-cuts the tiles so that a tile's MEASURED cost -- not its agent
 * count -- is equal across the SMs (tracks differ by up to 15 % per agent).  Results never depend on the tiling.  The
 * library does this on its own after the 16th, 64th and 256th launch of an env and every 4,096 launches from then on
 * (never inside a stream capture; OK_AUTO_BALANCE=0 turns that off); call it yourself after a change of workload.
 * out[0] / out[1] (nullable): slowest tile over mean tile before (measured) and after (predicted). */
int ok_balance_schedule(OkEnv *env, void *stream, float out[2]);
/* The beam kernel's tiling of the population (profiling aid; ok_debug_trace's tile ids index it): copies up to `capacity`
 * tiles as {track, count, first agent} to h_out[capacity][3] and returns the number of tiles. */
int64_t ok_debug_tiles(OkEnv *env, int64_t *h_out, int64_t capacity);
/* evaluates the kernels' sincosf (the glibc-2.39 restatement, ok_math.cuh) on `n` host floats: lets a test
 * compare the DEVICE function with libm / the oracle directly (tests/test_gpu_math.py).  The arrays are staged through
 * the env's staging buffer (kept at its largest size until ok_destroy) on the legacy default stream, which the call
 * synchronises before it returns, on error too. */
int ok_eval_sincosf(OkEnv *env, const float *h_in, float *h_sin, float *h_cos, int64_t n);

/* Host-link probe (measurement only, no env needed): moves `bytes` between a pinned host buffer and device memory
 * `iters` times on one stream and returns the achieved GB/s in *gbps_out.  mode 0: device->host DMA copies; 1: a kernel
 * storing through the host mapping (what ok_step_host does with the lidar observations); 2: host->device DMA copies.
 * bench.py and tools/pcie_ceiling.py run it on all ranks at once to measure the box's ceiling for the end-to-end path. */
int ok_pcie_probe(int32_t device, size_t bytes, int32_t iters, int32_t mode, double *gbps_out);

/* OK_RAYCAST_BEAM's candidate table, host side (no device needed; built on first use, ok_beam.hpp): the
 * segments a ray starting at (x, y) with direction `angle_rad` can reach within *d_complete px, nearest first.
 * Copies min(count, capacity) indices to h_items and returns count; OK_BEAM_NOT_COVERED = the start cell is not
 * covered (the kernel then uses the grid walk); other negative values are OkStatus errors.  Test / inspection hook. */
#define OK_BEAM_NOT_COVERED (-100)
int32_t ok_beam_lookup(OkEnv *env, int32_t track_id, float x, float y, float angle_rad, uint16_t *h_items,
                       int32_t capacity, float *d_complete);
/* the same, also returning what the kernel's first pass works with: *n_inline = how many of the leading candidates are
 * carried in the table entry itself (at most 4), *d_inline = the distance up to which those are provably the ONLY
 * contenders (every other listed segment is met at a parameter >= *d_inline by every ray of the cell and bin) */
int32_t ok_beam_lookup_ex(OkEnv *env, int32_t track_id, float x, float y, float angle_rad, uint16_t *h_items,
                          int32_t capacity, float *d_complete, float *d_inline, int32_t *n_inline);
/* size of the track's beam table in bytes (builds it if needed) */
int64_t ok_beam_table_bytes(OkEnv *env, int32_t track_id);
/* Beam tables are shared between the envs of a process through a cache (host copies and, per device, the tables the
 * kernels read: ~250 MB per track at the default resolution).  This drops the cache's own references; a table is freed
 * when the last env that uses it is destroyed. */
void ok_release_caches(void);

#ifdef __cplusplus
}
#endif
#endif /* OPENKITCHEN_B200_H */
