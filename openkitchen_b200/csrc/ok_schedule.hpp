// ok_schedule.hpp -- how large a population's batches are and which kernel shape runs it, and how the agent range is cut
// into tiles (batches of same-track agents that the CTAs of the step kernel pull in list order).  Host-only and free of
// CUDA: every decision here is a pure function of host data, and ok_capi.cu allocates and uploads the result.
#pragma once

#include <cstddef>
#include <cstdint>
#include <optional>
#include <string>
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

// ---- sizing of a population (ok_alloc_agents) ---------------------------------------------------------------------------

// The environment variables that steer the sizing, as ok_capi.cu reads them at every ok_alloc_agents (unset: empty).  Their
// defaults and bounds are applied here.
struct SizingKnobs
{
    enum class BeamKernel
    {
        Automatic,
        Staged,
        Unstaged
    };
    std::optional<int> batch_agents;                   // OK_BATCH_AGENTS: cap on the grid kernel's batch (default 256)
    BeamKernel         beam_kernel{BeamKernel::Automatic}; // OK_BEAM_KERNEL = staged | unstaged (anything else: automatic)
    std::optional<int> beam_batch_agents;              // OK_BEAM_BATCH_AGENTS: cap on the beam kernel's tile
    std::optional<int> beam_tail;                      // OK_BEAM_TAIL: guided beam tiling with this tail divisor
    std::optional<int> beam_waves;                     // OK_BEAM_WAVES: balanced tiling, tiles per CTA (default 1)
    std::optional<int> auto_balance;                   // OK_AUTO_BALANCE=0: keep the tiling by agent count
    std::optional<int> e2e_tiles;                      // OK_E2E_TILES: ok_step_host tiles per CTA (default 4)
    std::optional<int> e2e_tiles_q16;                  // OK_E2E_TILES_Q16: ok_step_host_q16's (default 3, or OK_E2E_TILES)
    std::optional<int> e2e_flushers;                   // OK_E2E_FLUSHERS: SMs left to obs_flush_kernel (at most half)
    std::optional<int> act_stage;                      // OK_ACT_STAGE=0: every tile reads the mapped actions
};

// What the step kernels need of shared memory, as plain numbers (ok_capi.cu fills it from ok_step.cuh)
struct StepFootprint
{
    int64_t agent_rec;          // sizeof(AgentRec): one per agent of a batch or tile
    int64_t grid_ray_bytes;     // batch_smem_bytes: bytes per ray of an agent of the grid kernel's batch
    int64_t beam_static_staged; // beam_static_smem(true)
    int32_t beam_block_staged, beam_block_unstaged; // beam_block(true / false)
    int32_t beam_tile;          // OK_BEAM_TILE: agents per tile of the unstaged beam kernel
};

// How a population runs: the kernel shapes and batch sizes (size_population), the unstaged beam kernel's occupancy
// (queried by the caller), the flusher count (tile_population) and the knob-derived flags.
struct Sizing
{
    int32_t batch_agents{0}; // the grid kernel's batch
    size_t  smem{0};         // ... and its dynamic shared memory
    bool    beam_staged{false};
    int32_t beam_block{0};
    int32_t batch_agents_beam{0};
    size_t  smem_beam{0};
    int32_t ctas_per_sm_beam{1};
    int32_t e2e_flushers{0};
    bool    auto_balance{true};
    bool    act_stage{true};
};

// Stage 1: the shape of a population of n agents x rays behind tracks of up to max_blob bytes, on a device of num_sms SMs
// and smem_optin bytes of shared memory per block.  False (with err) when shared memory cannot hold one agent's rays.
bool size_population(int64_t n, int32_t rays, int num_sms, int smem_optin, size_t max_blob, const StepFootprint &fp,
                     const SizingKnobs &knobs, Sizing &out, std::string &err);

// a tiling as it is uploaded: the table, room for `capacity` tiles (at least as many as there are), run by `ctas` CTAs at most
struct Tiling
{
    std::vector<Tile> tiles;
    size_t            capacity{0};
    int               ctas{0};
};

// Stage 2: every tiling of the population (track_id[0, n)) that s describes, s.ctas_per_sm_beam included.
struct PopulationTilings
{
    Tiling grid; // guided, the grid kernel's
    Tiling beam;
    bool   feedback{false};      // beam is the feedback tiling: re-cut from measured tile times (reweigh_runs) ...
    std::vector<TileRun> runs;   // ... of these runs ...
    int64_t              target{0}; // ... into this many tiles
    Tiling  e2e, q16;            // ok_step_host's and ok_step_host_q16's (staged beam kernel only)
    int32_t e2e_flushers{0};
};
PopulationTilings tile_population(const int32_t *track_id, int64_t n, const Sizing &s, int num_sms, const SizingKnobs &knobs);

} // namespace ok
