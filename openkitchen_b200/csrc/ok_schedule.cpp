// ok_schedule.cpp -- sizing of a population and tilings of the agent range (ok_schedule.hpp)
#include "ok_schedule.hpp"

#include <algorithm>

namespace ok
{

std::vector<TileRun> track_runs(const int32_t *track_id, int64_t n, int64_t cap)
{
    std::vector<TileRun> runs;
    for (int64_t i = 0; i < n;)
    {
        int64_t j = i;
        while (j < n && track_id[j] == track_id[i])
            ++j;
        runs.push_back({track_id[i], i, j - i, cap, 1.0, 0});
        i = j;
    }
    return runs;
}

std::vector<Tile> guided_tiles(const int32_t *track_id, int64_t n, int big, int ctas, int tail_div)
{
    const int     small       = std::max(1, big / std::max(1, tail_div));
    const int64_t tail_agents = tail_div > 1 ? std::min<int64_t>(n / 2, static_cast<int64_t>(ctas) * big / 2) : 0;
    std::vector<Tile> tiles, tail;
    for (const TileRun &r : track_runs(track_id, n, big))
    {
        const int64_t j        = r.begin + r.len;
        const int64_t run_tail = r.len * tail_agents / n; // this run's share of the small-tile tail
        const int64_t split    = j - run_tail;
        for (int64_t b = r.begin; b < j;)
        {
            const bool    in_tail = b >= split;
            const int64_t lim     = in_tail ? j : split;
            Tile          t{};
            t.track = r.track;
            t.begin = b;
            t.count = static_cast<int32_t>(std::min<int64_t>(in_tail ? small : big, lim - b));
            (in_tail ? tail : tiles).push_back(t);
            b += t.count;
        }
    }
    tiles.insert(tiles.end(), tail.begin(), tail.end());
    return tiles;
}

BalancedTiling balanced_tiles(std::vector<TileRun> &runs, int64_t max_tile, int ctas, int min_waves)
{
    int64_t n = 0, have = 0;
    for (const TileRun &r : runs)
        n += r.len, have += (r.len + r.cap - 1) / r.cap;
    const int64_t per_wave = static_cast<int64_t>(ctas) * max_tile;
    const int64_t waves    = std::max<int64_t>({static_cast<int64_t>(min_waves), (n + per_wave - 1) / per_wave, (have + ctas - 1) / ctas});
    BalancedTiling out;
    out.target = static_cast<int64_t>(ctas) * waves;
    out.tiles  = cost_balanced_tiles(runs, out.target, 0.0, nullptr);
    return out;
}

std::vector<Tile> cost_balanced_tiles(std::vector<TileRun> &runs, int64_t target, double c0, float *slowest_over_mean)
{
    int64_t have = 0;
    for (auto &r : runs)
    {
        r.k = std::max<int64_t>(1, (r.len + r.cap - 1) / r.cap);
        have += r.k;
    }
    auto cost = [&](const TileRun &r) { return c0 + r.w * static_cast<double>((r.len + r.k - 1) / r.k); };
    for (; have < target; ++have)
    {
        TileRun *best = nullptr;
        for (auto &r : runs)
            if (r.len > r.k && (!best || cost(r) > cost(*best)))
                best = &r;
        if (!best)
            break;
        best->k++;
    }
    struct Costed
    {
        Tile   t;
        double c;
    };
    std::vector<Costed> tiles;
    double              sum = 0.0, worst = 0.0;
    for (const auto &r : runs)
        for (int64_t t = 0; t < r.k; ++t)
        {
            const int64_t b0 = r.begin + r.len * t / r.k, b1 = r.begin + r.len * (t + 1) / r.k;
            if (b1 > b0)
            {
                const double c = c0 + r.w * static_cast<double>(b1 - b0);
                tiles.push_back({{r.track, static_cast<int32_t>(b1 - b0), b0}, c});
                sum += c, worst = std::max(worst, c);
            }
        }
    std::stable_sort(tiles.begin(), tiles.end(), [](const Costed &a, const Costed &b) { return a.c > b.c; });
    if (slowest_over_mean)
        *slowest_over_mean = tiles.empty() ? 1.0f : static_cast<float>(worst * static_cast<double>(tiles.size()) / sum);
    std::vector<Tile> out;
    out.reserve(tiles.size());
    for (const auto &t : tiles)
        out.push_back(t.t);
    return out;
}

bool reweigh_runs(std::vector<TileRun> &runs, const std::vector<Tile> &tiles, const uint32_t *ns, bool &weighted, int64_t target,
                  Reweighing &out)
{
    // per run: ns of ray phase per agent; c0: the median of what a tile spends outside the ray phase
    std::vector<double>   ray_ns(runs.size(), 0.0), agents(runs.size(), 0.0);
    std::vector<uint32_t> rest;
    for (size_t i = 0; i < tiles.size(); ++i)
    {
        if (ns[2 * i] == 0 || ns[2 * i] > 1000000000u) // never ran (or a wrapped timer): no information
            continue;
        const Tile &t = tiles[i];
        for (size_t r = 0; r < runs.size(); ++r)
            if (t.begin >= runs[r].begin && t.begin < runs[r].begin + runs[r].len)
            {
                ray_ns[r] += ns[2 * i], agents[r] += t.count;
                break;
            }
        rest.push_back(ns[2 * i + 1]);
    }
    if (rest.size() * 2 < tiles.size())
        return false; // too few tiles measured
    std::nth_element(rest.begin(), rest.begin() + rest.size() / 2, rest.end());
    const double c0 = rest[rest.size() / 2];
    double       w_sum = 0.0, a_sum = 0.0;
    for (size_t r = 0; r < runs.size(); ++r)
        w_sum += ray_ns[r], a_sum += agents[r];
    const double w_mean = a_sum > 0 ? w_sum / a_sum : 1.0;
    // what the CURRENT tiling costs under the measured model (for the report)
    {
        double sum = 0.0, worst = 0.0;
        for (size_t i = 0; i < tiles.size(); ++i)
        {
            const double c = static_cast<double>(ns[2 * i]) + ns[2 * i + 1];
            sum += c, worst = std::max(worst, c);
        }
        out.balance_before = sum > 0 ? static_cast<float>(worst * tiles.size() / sum) : 1.0f;
    }
    for (size_t r = 0; r < runs.size(); ++r)
    { // the first measurement as it is; later ones damped, half way from the weight in use to the measured one
        const double measured = agents[r] > 0 ? ray_ns[r] / agents[r] : w_mean;
        runs[r].w             = weighted ? 0.5 * (runs[r].w + measured) : measured;
    }
    weighted  = true;
    out.tiles = cost_balanced_tiles(runs, target, c0, &out.balance_after);
    return true;
}

bool size_population(int64_t n, int32_t rays, int num_sms, int smem_optin, size_t max_blob, const StepFootprint &fp,
                     const SizingKnobs &knobs, Sizing &out, std::string &err)
{
    out = Sizing{};
    // small populations: spread over all SMs rather than filling a few batches
    const int64_t spread = std::max<int64_t>(1, (n + num_sms - 1) / std::max(1, num_sms));
    // grid kernel: batch = the agents a CTA keeps in flight, as many as fit behind the largest staged track
    const size_t blob  = (max_blob + 127) / 128 * 128;
    const size_t avail = static_cast<size_t>(smem_optin) > blob + 4096 ? smem_optin - blob - 4096 : 0;
    const size_t per   = static_cast<size_t>(fp.agent_rec + fp.grid_ray_bytes * rays);
    int64_t      a     = static_cast<int64_t>(avail / per);
    if (avail < static_cast<size_t>(fp.beam_static_staged) + 4096)
        a = 0; // the beam kernel keeps per-thread scratch and its ray queue in static shared memory
    a = std::min<int64_t>(a, knobs.batch_agents ? std::max(1, *knobs.batch_agents) : 256);
    a = std::min<int64_t>(a, spread);
    if (a < 1)
    {
        err = "shared memory cannot hold one agent's rays next to the largest track";
        return false;
    }
    out.batch_agents = static_cast<int32_t>(a);
    out.smem         = blob + static_cast<size_t>(a) * per;
    // beam kernel: one AgentRec per agent; phases 1 / 4 run a thread per agent, so at most one block of agents.
    // Which shape (ok_step.cuh): the staged one for throughput, the unstaged one when the population is too small
    // to give every SM a worthwhile tile.
    // measured (tools/bench_small.py, tools/bench_c4.py): the unstaged shape is ahead below ~2,000 agents of 32 rays, and at
    // 4,096 agents of 5 rays (a PPO rollout tick: 0.0289 vs 0.0300 ms, 0.0262 with the policy step fused in), behind at
    // 8,192 agents of 5 rays (0.0376 vs 0.0318 ms)
    out.beam_staged = knobs.beam_kernel == SizingKnobs::BeamKernel::Automatic ? n >= 2048 && n * rays > 24576
                                                                                : knobs.beam_kernel == SizingKnobs::BeamKernel::Staged;
    out.beam_block = out.beam_staged ? fp.beam_block_staged : fp.beam_block_unstaged;
    int64_t ab;
    int64_t capb;
    if (out.beam_staged)
    { // one 1,024-thread CTA per SM behind the staged track: as many agents per tile as the shared memory behind the
      // largest track holds (the balanced tiling then sizes the tiles: about one per CTA and wave)
        ab   = static_cast<int64_t>((avail - static_cast<size_t>(fp.beam_static_staged)) / static_cast<size_t>(fp.agent_rec));
        capb = out.beam_block;
    }
    else
    { // several small CTAs per SM, nothing staged: small tiles, the SM's other CTAs hide a tile's serial phases
        ab   = out.beam_block;
        capb = fp.beam_tile;
    }
    ab = std::min<int64_t>(ab, 65535 / rays); // tile-local ray indices are 16 bits (the kernel's ray queue)
    if (knobs.beam_batch_agents)
        capb = std::max(1, *knobs.beam_batch_agents);
    ab = std::min<int64_t>({ab, capb, out.beam_block});
    if (!out.beam_staged)
        ab = std::min<int64_t>(ab, spread);
    out.batch_agents_beam = static_cast<int32_t>(std::max<int64_t>(1, ab));
    // beam_smem_bytes: the records, rounded up to 16 bytes
    out.smem_beam = (out.beam_staged ? blob : 0) + (static_cast<size_t>(out.batch_agents_beam * fp.agent_rec) + 15u) / 16u * 16u;
    out.auto_balance = knobs.auto_balance.value_or(1) != 0;
    out.act_stage    = knobs.act_stage.value_or(1) != 0;
    return true;
}

PopulationTilings tile_population(const int32_t *track_id, int64_t n, const Sizing &s, int num_sms, const SizingKnobs &knobs)
{
    PopulationTilings out;
    out.grid = {guided_tiles(track_id, n, s.batch_agents, num_sms, 4), 0, num_sms};
    // the balanced tiling of the beam kernel's batches over `ctas` CTAs, at least `waves` tiles per CTA; `runs` keeps the
    // track runs with their tile counts
    auto balanced = [&](int ctas, int waves, std::vector<TileRun> &runs) {
        runs = track_runs(track_id, n, s.batch_agents_beam);
        return balanced_tiles(runs, s.batch_agents_beam, ctas, waves);
    };
    const int beam_ctas = num_sms * s.ctas_per_sm_beam;
    // the unstaged beam kernel's small tiles cost about the same serial latency whatever their size (the thread-per-
    // agent phases, the second ray pass): shrinking them further only adds tiles
    const int tail_div = knobs.beam_tail.value_or(s.beam_staged ? -1 : 0); // -1: balanced tiling
    if (tail_div < 0)
    { // the feedback tiling: its table is allocated once, with room for every re-cut (rebalance_beam_tiles)
        BalancedTiling bt = balanced(beam_ctas, std::max(1, knobs.beam_waves.value_or(1)), out.runs);
        out.feedback      = true;
        out.target        = bt.target;
        out.beam          = {std::move(bt.tiles), 0, beam_ctas};
        out.beam.capacity = std::max<size_t>(out.beam.tiles.size(), static_cast<size_t>(bt.target));
    }
    else
        out.beam = {guided_tiles(track_id, n, s.batch_agents_beam, beam_ctas, tail_div), 0, beam_ctas};
    if (s.beam_staged)
    { // the end-to-end tilings (see ok_step_host).  OK_E2E_FLUSHERS = F > 0: F SMs are left to obs_flush_kernel, which
      // moves finished tiles to the host while the step kernel's CTAs carry on
        const int per_cta = std::max(1, knobs.e2e_tiles.value_or(4));
        out.e2e_flushers  = std::max(0, std::min(knobs.e2e_flushers.value_or(0), num_sms / 2));
        const int e2e_ctas = (num_sms - out.e2e_flushers) * s.ctas_per_sm_beam;
        std::vector<TileRun> runs;
        BalancedTiling       e2e = balanced(e2e_ctas, per_cta, runs);
        out.e2e                  = {std::move(e2e.tiles), static_cast<size_t>(e2e.target), e2e_ctas};
        // ok_step_host_q16: measured at the C3 shape 0.164 / 0.157 / 0.171 / 0.199 ms per tick with 2 / 3 / 4 / 6 tiles per CTA
        const int      per_cta_q16 = knobs.e2e_tiles_q16 ? std::max(1, *knobs.e2e_tiles_q16) : knobs.e2e_tiles ? per_cta : 3;
        const int      q16_ctas    = num_sms * s.ctas_per_sm_beam;
        BalancedTiling q16         = balanced(q16_ctas, per_cta_q16, runs);
        out.q16                    = {std::move(q16.tiles), static_cast<size_t>(q16.target), q16_ctas};
    }
    return out;
}

} // namespace ok
