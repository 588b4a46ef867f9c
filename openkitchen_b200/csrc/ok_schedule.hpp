// ok_schedule.hpp -- how the agent range is cut into tiles (batches of same-track agents that the CTAs of the step kernel
// pull in list order).  Host-only and free of CUDA: every decision here is a pure function of host data, and
// ok_capi.cu uploads the result.
#pragma once

#include <cstdint>
#include <vector>

namespace ok
{

struct Tile
{
    int32_t track;
    int32_t count;
    int64_t begin;
};

// a maximal run of same-track agents, with what the cost-balanced tiling knows of it
struct TileRun
{
    int32_t track;
    int64_t begin, len, cap; // cap: most agents a tile of this run may hold
    double  w;               // measured cost per agent (ns in the ray phase), 1 before any measurement
    int64_t k;               // tiles
};

// the maximal same-track runs of track_id[0, n), each with tile cap `cap`, w = 1 and k = 0
std::vector<TileRun> track_runs(const int32_t *track_id, int64_t n, int64_t cap);

// Guided self-scheduling: every run cut into tiles of `big` agents, in order; with tail_div > 1 about half a big tile per
// CTA (at most half the agents) is taken from the end of every run, in proportion to its length, and cut into tiles
// 1 / tail_div the size that follow all the big ones and even out the finish.  tail_div <= 1: uniform tiles.
std::vector<Tile> guided_tiles(const int32_t *track_id, int64_t n, int big, int ctas, int tail_div);

// Balanced tiling (staged beam kernel).  The kernel's cost per ray is nearly uniform, but a tile pays ~15 us of serial
// latency (thread-per-agent phases, second ray pass, barriers) whatever its size: the fewer, larger and more equal the
// tiles, the better.  Tiles = CTAs x waves (at least min_waves, and as many as max_tile requires), dealt to the runs in
// proportion to their length (and, once the kernel has reported tile times, to their measured cost: reweigh_runs).
struct BalancedTiling
{
    std::vector<Tile> tiles;
    int64_t           target; // CTAs x waves
};
BalancedTiling balanced_tiles(std::vector<TileRun> &runs, int64_t max_tile, int ctas, int min_waves);

// Cost-aware balanced tiling.  A tile of `count` agents of run r costs about c0 + w_r * count (c0: the thread-per-agent
// phases and barriers, whatever the size; w_r: the ray phase, which differs from track to track by up to 15 %).  Tiles go
// to the runs greedily -- one more for the run whose tiles are the most expensive -- which minimises the slowest tile;
// every run is cut into equal parts, most expensive first (CTAs take tiles in list order).  With w = 1, c0 = 0 this is the
// plain balanced tiling by agent count.  Sets runs[].k; *slowest_over_mean (nullable): predicted slowest / mean tile cost.
std::vector<Tile> cost_balanced_tiles(std::vector<TileRun> &runs, int64_t target, double c0, float *slowest_over_mean);

// The feedback model of the beam tiling.  ns[2 i], ns[2 i + 1]: the ns tile i of `tiles` spent in the ray phase and in the
// rest, as the kernel left them.  Zero or wrapped (> 1e9) ray times carry no information; with fewer than half the tiles
// measured nothing changes and the result is false.  Otherwise every run's weight becomes its measured ray ns per agent --
// as measured in the first round (`weighted` false, then set), half way from the weight in use in later ones -- c0 the
// median of the measured tiles' other times, and `out` the cost-balanced re-cut with its predicted balance.
struct Reweighing
{
    std::vector<Tile> tiles;
    float             balance_before; // slowest / mean measured tile time of `tiles`
    float             balance_after;  // the same, predicted for the re-cut
};
bool reweigh_runs(std::vector<TileRun> &runs, const std::vector<Tile> &tiles, const uint32_t *ns, bool &weighted, int64_t target,
                  Reweighing &out);

} // namespace ok
