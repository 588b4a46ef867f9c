// ok_bev.cuh -- the host's interface to the bird's-eye-view query (ok_bev.cu): semantic rasters of the track around
// arbitrary poses, with no agent state read or written.
//
// Pixel (r, c) of an H x W image at pose (x, y, rot) on track t is the point
//   f  = (0.5 (H-1) - r) scale + ahead,   l = (c - 0.5 (W-1)) scale,   (rs, rc) = sincosf(kDeg2Rad rot)
//   px = x + (f rc - l rs),               py = y + (f rs + l rc)
// in binary32, rounded in that order; k = the number of the four closed boundary loops LI, LO, RI, RO that contain it
// by the even-odd (PNPOLY) rule; the class is OK_BEV_LANE for k == 2, OK_BEV_WALL for odd k, OK_BEV_OFF otherwise.
//
// The table the kernel reads, per track: the y axis cut into bands of kBevBand px, and per (band, loop) the loop's
// edges whose y-range meets the band, sorted by their x bound xhi, descending.  A pixel reads only its band's lists.
#pragma once

#include <cstdint>
#include <vector>

#include <cuda_runtime.h>

namespace ok
{
struct Track;

constexpr float kBevBand    = 2.0f;  // band height (px)
constexpr float kBevInvBand = 0.5f;  // its inverse, a power of two: the band coordinate (y - y0) * kBevInvBand is monotone in y
constexpr int   kBevLoops   = 4;     // LI, LO, RI, RO

// one track's bands: lists of band b, loop L are entries [starts[off_starts + 4 b + L], starts[off_starts + 4 b + L + 1])
struct BevTrack
{
    float    y0;         // y of band 0's lower edge
    int32_t  n_bands;
    uint32_t off_starts; // into BevTableView::starts
    uint32_t pad;
};
static_assert(sizeof(BevTrack) == 16, "BevTrack layout");

// an edge (i, j = i - 1) of a loop, as the kernel tests it: a = {y_i, y_j, xlo, xhi}, b = {x_i, x_j}.  A point with
// (y_i > py) != (y_j > py) crosses the edge when px < xlo, does not when px >= xhi, and is decided by the exact PNPOLY
// expression in between (see xlo / xhi in ok_bev.cu for why the two bounds are exact).
struct BevTableView
{
    const BevTrack *tracks;
    const uint32_t *starts;
    const float4   *a;
    const float2   *b;
    uint32_t        n_starts, n_entries; // OK_CHECKED builds only
};

// the band lists of every track in one blob: [BevTrack x tracks][starts][pad to 16][float4 a][float2 b]
struct BevTableHost
{
    std::vector<uint8_t> bytes;
    size_t               off_starts{0}, off_a{0}, off_b{0};
    int32_t              n_tracks{0};
    size_t               entries{0};
};
void build_bev_table(const std::vector<Track> &tracks, BevTableHost &out);

struct BevQueryParams
{
    const float   *x, *y, *rot; // f32[n]: pose (rot in degrees)
    const int32_t *track;       // nullable: track 0; out-of-range ids are clamped
    int64_t        n;
    int32_t        height, width;
    float          scale, ahead;
    uint8_t       *out; // u8[n][height][width]
    int32_t        n_tracks;
    BevTableView   table;
};

constexpr int kBevBlock = 256;
constexpr int kBevBytes = 4; // output bytes per thread: one 32-bit store, a warp stores 128 consecutive bytes

cudaError_t launch_bev_query(const BevQueryParams &q, cudaStream_t stream);
cudaError_t violations_bev(unsigned long long *count); // the unit's self-check counter (OK_CHECKED builds)
} // namespace ok
