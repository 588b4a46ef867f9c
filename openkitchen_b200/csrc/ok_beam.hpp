// ok_beam.hpp -- "beam lists": the narrow phase's candidate table.
//
// For every cell of a fine uniform grid over the lane (`cell` px) and every direction bin (2*pi / `bins`)
// the table holds the segments a ray that STARTS in that cell with a direction in that bin can reach within
// a completeness distance d, nearest first:
//
//     list(C, b) = { S : dist(C, b, S) <= d(C, b) },
//     dist(C, b, S) = min { t >= 0 : p + t u(theta) in S, p in C, theta in b }.
//
// dist is computed exactly (up to binary64 rounding, which the inflation margins dominate): with
// H = S (+) (-C) (Minkowski sum, a convex hexagon), dist = Euclidean distance from the origin to
// H intersected with the bin's cone.  d(C, b) is chosen from a few sample rays as "a little beyond the
// farthest first hit"; it only decides how long the list is, never correctness: the kernel accepts
// a list-based result only if the hit parameter is <= d - slack, and otherwise continues with the
// uniform-grid walk from t = d - 1 (ok_kernels.cuh, "beam phase").  Hence
//     every segment whose true crossing parameter is <= d is in the list      (by construction)
//  => a ray whose nearest listed hit is at t <= d - slack has no nearer hit   (rounding << slack)
// which is the same exactness class as the grid walk (DESIGN.md "broadphase exactness").
//
// The reference has no counterpart: CollisionChecker.cu:51-66 tests every ray against every segment.
#pragma once

#include "ok_track.hpp"

#include <cstdint>
#include <string>
#include <vector>

namespace ok
{

// Header of a track's beam blob (device global memory).  Offsets in bytes from the blob start.
//
// An ENTRY is 16 bytes and carries the list's first four candidates INLINE, so that one 16-byte load (one 32-byte
// sector) gives the kernel everything most rays need:
//   x, y : the four nearest candidates (uint16 segment indices, nearest first, padded with the null segment)
//   z    : index of the first chunk of the REST of the list (candidates 5, 6, ...: chunks of four uint16, padded)
//   w    : meta = dq | d1q << 12 | n_rest_chunks << 24
//          dq  = floor(d * 16)  (12 bits, 0xfff = rb): the list is complete up to d
//          d1q = floor(d1 * 16) (12 bits): d1 = the lower bound dist(C, b, S) of the first candidate of the REST (= d
//                when there is no rest).  Every ray from the cell with a direction in the bin meets every segment of
//                the rest at a parameter >= d1, so a hit among the inline four at t <= d1 - slack is final WITHOUT
//                looking at the rest (the same argument, with d1 for d, as for the segments the list leaves out).
//          n_rest_chunks (8 bits): a longer list is cut and d lowered to the first candidate left out.
struct BeamHeader
{
    float    x0, y0;     // origin of the beam-cell grid
    float    inv_h, h;   // 1 / cell, cell
    int32_t  nx, ny;     // cells
    int32_t  nb;         // direction bins, a power of two
    float    bin_scale;  // nb / (2 pi): bin = floor(angle * bin_scale) & (nb - 1)
    float    rb;         // completeness distance of entries flagged complete (dq = 0xfff)
    uint32_t off_rows;   // uint32[nx * ny]: row of the cell in `entries`, 0xffffffff = not covered
    uint32_t off_entries; // uint4[n_rows * nb]
    uint32_t off_items;  // uint16[]: the rest lists, in chunks of 4, padded with n_segments (the blob's null segment)
    uint32_t n_rows;
    uint32_t n_chunks;
    uint32_t bytes;
    uint32_t tag;        // kBeamFormat << 16 | index of the null segment (= n_segments, the padding value)
};
static_assert(sizeof(BeamHeader) == 64, "BeamHeader must be 64 bytes");

constexpr uint32_t kBeamFormat      = 2;
constexpr uint32_t kBeamDistScale   = 16;    // quantisation of d and d1: 1/16 px, rounded DOWN (conservative)
constexpr uint32_t kBeamDistFull    = 0xfffu; // dq of a list that is complete up to rb
constexpr uint32_t kBeamMaxRest     = 255;   // chunks of a rest list
constexpr int      kBeamInline      = 4;     // candidates carried in the entry itself

#if defined(__CUDACC__)
#define OK_BEAM_HD __host__ __device__ inline
#else
#define OK_BEAM_HD inline
#endif
// meta word of an entry from the list's completeness distance d, the rest's lower bound d1 (both < rb unless `full`)
OK_BEAM_HD uint32_t beam_pack_meta(double d, double d1, bool full, uint32_t n_rest)
{
    const double   q  = d * kBeamDistScale, q1 = d1 * kBeamDistScale;
    uint32_t       dq = full ? kBeamDistFull : static_cast<uint32_t>(q < 0.0 ? 0.0 : (q > 4094.0 ? 4094.0 : q));
    const uint32_t d1q = static_cast<uint32_t>(q1 < 0.0 ? 0.0 : (q1 > 4094.0 ? 4094.0 : q1));
    return dq | (d1q << 12) | (n_rest << 24);
}
// the fields of a meta word w: chunks of the rest, d, d1 (rb = the table's completeness distance of full lists)
OK_BEAM_HD uint32_t beam_meta_rest(uint32_t w)
{
    return w >> 24;
}
OK_BEAM_HD float beam_meta_d(uint32_t w, float rb)
{
    const uint32_t q = w & 0xfffu;
    return q == kBeamDistFull ? rb : static_cast<float>(q) * (1.0f / kBeamDistScale);
}
OK_BEAM_HD float beam_meta_d1(uint32_t w, float rb)
{
    return beam_meta_d(w >> 12, rb);
}

struct BeamConfig
{
    float   cell{8.f};
    int32_t bins{64};
    float   range{200.f}; // Agent::kSensorRange; lists flagged complete cover range + 1
    float   pad{1.0f};    // px added to the farthest sampled first hit to get the completeness distance
    int32_t threads{0};   // 0 = std::thread::hardware_concurrency()
};

// bump when build_beam_table changes what it produces (the on-disk cache is keyed on it)
constexpr int    kBeamBuildVersion = 2;
constexpr double kBeamCellMargin  = 0.0625; // px: the cell is grown by this much on every side
constexpr double kBeamAngleMargin = 1e-4;   // rad: the bin's cone is widened by this much on both sides
constexpr float  kBeamSlack       = 0.25f;  // px: a list result is trusted up to d - slack
constexpr float  kBeamMaxAngle    = 100.0f; // rad: rays with a larger |angle| skip the table (bin rounding)

// The grid over the lane and the covered cells (shared by the host and the device builder).
struct BeamPlan
{
    double                x0{0}, y0{0}, h{0}, rb{0};
    int32_t               nx{0}, ny{0}, nb{0};
    std::vector<uint32_t> rows;    // per cell: row, 0xffffffff = not covered
    std::vector<uint32_t> covered; // per row: cell
};
bool beam_plan(const Track &t, const BeamConfig &cfg, BeamPlan &plan, std::string &err);
// section offsets of a table with n_items uint16 items
bool beam_layout(const BeamPlan &plan, const BeamConfig &cfg, size_t n_items, int32_t n_segments, BeamHeader &h, std::string &err);
// entries: 4 x uint32 per (row, bin) (see BeamHeader); items: the rest lists, uint16 chunks of 4
bool beam_assemble(const BeamPlan &plan, const BeamConfig &cfg, const uint32_t *entries, const uint16_t *items, size_t n_items,
                   int32_t n_segments, std::vector<uint8_t> &blob, std::string &err);

// Builds the blob on the host.  False (with err) if the configuration is unusable; never throws.
bool build_beam_table(const Track &t, const BeamConfig &cfg, std::vector<uint8_t> &blob, std::string &err);

// The same table built by a kernel on CUDA device `device` (ok_beam_gpu.cu): one CTA per covered cell.  Same
// construction, binary64 on the device; libm differences may move a list boundary by an ulp, never its validity.
// The blob is left in device memory (*d_blob, cudaMalloc'ed on `device`, owned by the caller).
bool build_beam_table_device(const Track &t, const BeamConfig &cfg, int device, uint8_t **d_blob, size_t *bytes, std::string &err);
// Several tables back to back, pipelined (the host sizes / allocates / assembles table i - 1 while the kernel of table i
// runs).  blobs[i] stays null for a track that needs the one-track path above (item array too small, any failure).
void build_beam_tables_device(const std::vector<const Track *> &tracks, const BeamConfig &cfg, int device, std::vector<uint8_t *> &blobs,
                              std::vector<size_t> &bytes);
// frees the device builder's scratch pool (kept between tracks)
void beam_builder_release();

// Host-side lookup used by the CPU tests: the list of (x, y, angle[rad]) -- the inline candidates (null padding removed)
// followed by the rest; returns false when the cell is not covered or the angle is out of range.  d_out = completeness
// distance, d1_out = lower bound of the rest (= d_out when the list has no rest), n_inline = candidates that came from
// the entry itself.
bool beam_lookup(const std::vector<uint8_t> &blob, float x, float y, float angle, std::vector<uint16_t> &items,
                 float &d_out, float *d1_out = nullptr, int32_t *n_inline = nullptr);

// Structural check of a table that did not come from this process's builders (the on-disk cache): sizes, offsets,
// row / chunk / segment indices all within bounds.  The kernels trust a table that passes.
bool beam_validate(const std::vector<uint8_t> &blob, int32_t n_segments, std::string &err);

} // namespace ok
