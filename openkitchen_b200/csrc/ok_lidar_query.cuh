// ok_lidar_query.cuh -- the host's interface to the lidar query kernel (ok_lidar_query.cu): lidar scans at arbitrary
// poses, with no agent state read or written.
#pragma once

#include "ok_device.cuh"

namespace ok
{
struct LidarQueryParams
{
    const float   *x, *y, *rot; // f32[n]: pose (rot in degrees)
    const int32_t *track;       // nullable: track 0; out-of-range ids are clamped
    int64_t        n;
    const float   *ray_deg; // f32[rays], relative to the heading
    int32_t        rays, n_tracks;
    const uint8_t  *arena;
    const TrackRef *tracks;
    // nullable outputs, in the layouts of the agent buffers of the same name
    float   *hit_abs, *hit_rel; // f32[n, rays, 2]
    float   *obs, *hit_t;       // f32[n, rays]
    int32_t *hit_seg;           // i32[n, rays], -1 = none
    float   *min_dist2;         // f32[n]
    uint8_t *crashed;           // u8[n]: min_dist2 < collision_dist2
    float    sensor_range, sensor_offset, collision_dist2;
    int32_t  raycast_mode;      // OkRaycastMode
};

constexpr int kLidarBlock = 256;
#ifndef OK_LIDAR_MIN_CTAS
#define OK_LIDAR_MIN_CTAS 4 // 64 registers per thread fill the register file, as in the unstaged beam kernel
#endif
constexpr int kLidarMinCtas = OK_LIDAR_MIN_CTAS;
// threads that share one pose when rays > 32: whole warps, at most the CTA
__host__ __device__ constexpr int lidar_threads_per_pose(int rays)
{
    return ((rays + 31) / 32) * 32 < kLidarBlock ? ((rays + 31) / 32) * 32 : kLidarBlock;
}
// poses per CTA: floor(32 / rays) per warp up to 32 rays, else the CTA's share of whole-warp groups
__host__ __device__ constexpr int lidar_poses_per_cta(int rays)
{
    return rays <= 32 ? (kLidarBlock / 32) * (32 / rays) : kLidarBlock / lidar_threads_per_pose(rays);
}

cudaError_t launch_lidar_query(const LidarQueryParams &q, cudaStream_t stream);
cudaError_t violations_lidar_query(unsigned long long *count); // the unit's self-check counter (OK_CHECKED builds)
} // namespace ok
