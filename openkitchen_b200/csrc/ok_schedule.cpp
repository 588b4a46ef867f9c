// ok_schedule.cpp -- tilings of the agent range (ok_schedule.hpp)
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

} // namespace ok
