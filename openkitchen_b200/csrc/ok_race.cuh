// ok_race.cuh -- the host's interface to the race pass (ok_race.cu): cars of a race see each other in the lidar and crash on
// contact, in a pass after the tick (OkRaces, include/openkitchen_b200.h).
#pragma once

#include "ok_device.cuh"

namespace ok
{
struct RaceParams
{
    // the tick's inputs and outputs, read and written only for the agent itself (the poses of the others are read)
    const float   *x, *y, *rot;
    const int32_t *track_id;
    uint8_t       *crashed, *done;
    float         *hit_abs, *hit_rel; // f32[n, rays, 2]
    float         *obs, *hit_t;       // f32[n, rays]
    int32_t       *hit_seg;           // i32[n, rays]
    float         *min_dist2;         // f32[n]
    // the pass's own outputs
    int32_t       *hit_car;           // i32[n, rays]: the car a ray hit, -1 = the track hit stands
    uint8_t       *contact;           // u8[n]: crashed by this pass
    const float   *ray_deg;           // f32[rays]
    int64_t        n;
    int32_t        rays, group, flags, n_tracks;
    float          radius, sensor_range, sensor_offset, collision_dist2;
    float          cull_d2; // a body whose centre is farther (squared) from the lidar origin cannot be hit; host-computed
};

constexpr int kRaceBlock = 256; // 8 warps, one agent each

cudaError_t launch_race_pass(const RaceParams &p, cudaStream_t stream);
cudaError_t violations_race(unsigned long long *count); // the unit's self-check counter (OK_CHECKED builds)
} // namespace ok
