// ok_beam.cpp -- see ok_beam.hpp.  Host code, binary64 geometry.
#include "ok_beam.hpp"
#include "ok_beam_geom.hpp"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <thread>

namespace ok
{
namespace
{
using namespace beamgeom;

struct Cand
{
    double  lb;               // lower bound of the distance from any point of the cell to the segment
    int32_t seg;
    int32_t b_first, b_count; // direction bins the segment can be seen in from the cell (conservative)
    int32_t hull;             // index into Scratch::hulls, -1 = not computed yet
};

struct HullRec
{
    int n;
    V2  v[9];
};

struct Row
{
    std::vector<uint32_t> meta;   // per bin: beam_pack_meta
    std::vector<uint32_t> inl;    // per bin: 2 words = the four inline candidates
    std::vector<uint32_t> first;  // per bin: first item of the bin's REST within `items` (multiple of 4)
    std::vector<uint16_t> items;  // rest lists, chunks of 4
};

struct Scratch
{
    std::vector<Cand>                                    cands;
    std::vector<std::vector<int32_t>>                    by_bin;
    std::vector<HullRec>                                 hulls;
    std::vector<double>                                  sample_hit, dcomp;
    std::vector<std::pair<float, uint16_t>>              list;
};

struct Builder
{
    const Track &t;
    BeamConfig   cfg;
    double       x0, y0, h, rb;
    int32_t      nx, ny, nb;
    double       dth;
    std::vector<V2> edge_lo, edge_hi; // widened cone edges of every bin
    std::vector<V2> sample_dir;       // 2 * nb sample directions (bin edges and bin centres)
    std::vector<V2> seg_mid;          // per segment: midpoint
    std::vector<double> seg_half;     // per segment: half length

    void build_row(int32_t cx, int32_t cy, Row &row, Scratch &sc) const
    {
        const int32_t ns = t.n_segments();
        const double  m  = kBeamCellMargin;
        const double  bx0 = x0 + cx * h - m, bx1 = x0 + (cx + 1) * h + m;
        const double  by0 = y0 + cy * h - m, by1 = y0 + (cy + 1) * h + m;
        const double  ccx = 0.5 * (bx0 + bx1), ccy = 0.5 * (by0 + by1);
        const double  half_diag = 0.5 * std::hypot(bx1 - bx0, by1 - by0);
        const double  two_pi = 2.0 * M_PI, dbin = two_pi / nb;
        // candidates: segments within reach, with a lower bound of their distance from the cell and the
        // direction bins they can be seen in.  For p in the cell and q on the segment, q - p lies in the disc
        // of radius (half_diag + half length) around (midpoint - cell centre).
        auto &cands = sc.cands;
        cands.clear();
        for (int32_t s = 0; s < ns; ++s)
        {
            const double vx = seg_mid[s].x - ccx, vy = seg_mid[s].y - ccy;
            const double dist = std::hypot(vx, vy), rho = half_diag + seg_half[s];
            if (dist - rho > rb)
                continue;
            const float *g = &t.segments[4 * static_cast<size_t>(s)];
            const double d = point_segment_distance(ccx, ccy, g[0], g[1], g[2], g[3]) - half_diag;
            if (d > rb)
                continue;
            Cand c{std::max(0.0, d), s, 0, nb, -1};
            if (dist > rho * 1.0000001)
            {
                const double phi = std::atan2(vy, vx), alpha = std::asin(std::min(1.0, rho / dist)) + 2.0 * dth;
                const double f_lo = std::floor((phi - alpha) / dbin), f_hi = std::floor((phi + alpha) / dbin);
                c.b_count = static_cast<int32_t>(std::min<double>(nb, f_hi - f_lo + 1.0));
                c.b_first = static_cast<int32_t>(std::fmod(std::fmod(f_lo, nb) + nb, nb));
            }
            cands.push_back(c);
        }
        std::sort(cands.begin(), cands.end(), [](const Cand &a, const Cand &b) { return a.lb < b.lb || (a.lb == b.lb && a.seg < b.seg); });
        sc.by_bin.resize(nb);
        for (auto &v : sc.by_bin)
            v.clear();
        for (size_t i = 0; i < cands.size(); ++i)
            for (int32_t k = 0; k < cands[i].b_count; ++k)
                sc.by_bin[(cands[i].b_first + k) % nb].push_back(static_cast<int32_t>(i));

        // completeness distance per bin from sample rays: the four corners and the centre of the cell, the bin's
        // two edges and its centre.  Misses count as "beyond the range".
        const double ox[5] = {bx0, bx1, bx0, bx1, ccx}, oy[5] = {by0, by0, by1, by1, ccy};
        sc.sample_hit.assign(static_cast<size_t>(2 * nb), 0.0);
        for (int32_t j = 0; j < 2 * nb; ++j)
        {
            const V2 d   = sample_dir[j];
            double   far = 0.0;
            for (int o = 0; o < 5; ++o)
            {
                double best = 2.0 * rb; // miss
                for (const int32_t ci : sc.by_bin[j >> 1])
                {
                    const Cand &c = cands[ci];
                    if (c.lb > best)
                        break;
                    const float *g  = &t.segments[4 * static_cast<size_t>(c.seg)];
                    const double sx = static_cast<double>(g[2]) - g[0], sy = static_cast<double>(g[3]) - g[1];
                    const double den = d.x * sy - d.y * sx;
                    if (std::fabs(den) < 1e-12)
                        continue;
                    const double ex = g[0] - ox[o], ey = g[1] - oy[o];
                    const double tt = (ex * sy - ey * sx) / den, ss = (ex * d.y - ey * d.x) / den;
                    if (tt >= 0 && tt < best && ss >= 0 && ss <= 1)
                        best = tt;
                }
                far = std::max(far, best);
            }
            sc.sample_hit[j] = far;
        }
        sc.dcomp.resize(nb);
        for (int32_t b = 0; b < nb; ++b)
        {
            const double far =
                std::max(sc.sample_hit[2 * b], std::max(sc.sample_hit[2 * b + 1], sc.sample_hit[(2 * b + 2) % (2 * nb)]));
            double d = far + cfg.pad;
            if (far >= cfg.range || d >= rb)
                d = rb;
            sc.dcomp[b] = d;
        }

        // exact membership: distance from the origin to (S (+) -C) clipped to the bin's cone
        sc.hulls.clear();
        row.meta.assign(nb, 0);
        row.inl.assign(2 * static_cast<size_t>(nb), 0);
        row.first.assign(nb, 0);
        row.items.clear();
        for (int32_t b = 0; b < nb; ++b)
        {
            auto &l = sc.list;
            l.clear();
            const double dc = sc.dcomp[b];
            for (const int32_t ci : sc.by_bin[b])
            {
                Cand &c = cands[ci];
                if (c.lb > dc)
                    break;
                if (c.hull < 0)
                {
                    const float *g = &t.segments[4 * static_cast<size_t>(c.seg)];
                    V2           pts[8];
                    int          np = 0;
                    for (int e = 0; e < 2; ++e)
                        for (int k = 0; k < 4; ++k)
                            pts[np++] = {g[2 * e] - ((k & 1) ? bx1 : bx0), g[2 * e + 1] - ((k & 2) ? by1 : by0)};
                    HullRec hr;
                    hr.n   = convex_hull8(pts, np, hr.v);
                    c.hull = static_cast<int32_t>(sc.hulls.size());
                    sc.hulls.push_back(hr);
                }
                const HullRec &hr = sc.hulls[c.hull];
                V2             c1[12], c2[14];
                const int      n1  = clip_half_plane(hr.v, hr.n, edge_lo[b], c1);
                const V2       neg = {-edge_hi[b].x, -edge_hi[b].y};
                const int      n2  = clip_half_plane(c1, n1, neg, c2);
                const double   d   = origin_distance(c2, n2);
                if (d <= dc)
                    l.push_back({static_cast<float>(d), static_cast<uint16_t>(c.seg)});
            }
            std::sort(l.begin(), l.end());
            const size_t cap   = kBeamInline + 4 * static_cast<size_t>(kBeamMaxRest);
            const size_t count = std::min<size_t>(l.size(), cap);
            double       d     = dc;
            if (count < l.size())
                d = std::max(0.0, static_cast<double>(l[count].first) - 1e-3); // truncated: complete only up to here
            const uint16_t null_seg = static_cast<uint16_t>(t.n_segments());   // the blob's null segment
            uint16_t       in4[kBeamInline];
            for (int i = 0; i < kBeamInline; ++i)
                in4[i] = static_cast<size_t>(i) < count ? l[i].second : null_seg;
            row.inl[2 * b]     = in4[0] | (static_cast<uint32_t>(in4[1]) << 16);
            row.inl[2 * b + 1] = in4[2] | (static_cast<uint32_t>(in4[3]) << 16);
            row.first[b]       = static_cast<uint32_t>(row.items.size());
            for (size_t i = kBeamInline; i < count; ++i)
                row.items.push_back(l[i].second);
            while (row.items.size() % 4)
                row.items.push_back(null_seg);
            const uint32_t n_rest = static_cast<uint32_t>((row.items.size() - row.first[b]) / 4);
            const double   d1     = count > static_cast<size_t>(kBeamInline) ? std::min<double>(l[kBeamInline].first, d) : d;
            row.meta[b]           = beam_pack_meta(d, d1, d >= rb, n_rest);
        }
    }
};
} // namespace

bool beam_plan(const Track &t, const BeamConfig &cfg, BeamPlan &pl, std::string &err)
{
    if (!(cfg.cell >= 1.0f && cfg.cell <= 64.0f))
    {
        err = "beam cell must be in [1, 64] px";
        return false;
    }
    if (cfg.bins < 8 || cfg.bins > 1024 || (cfg.bins & (cfg.bins - 1)))
    {
        err = "beam bins must be a power of two in [8, 1024]";
        return false;
    }
    const int32_t n = t.n_points(), ns = t.n_segments();
    if (n < 2 || ns < 1)
    {
        err = "empty track";
        return false;
    }
    double lo_x = 1e300, lo_y = 1e300, hi_x = -1e300, hi_y = -1e300;
    for (int32_t s = 0; s < ns; ++s)
        for (int e = 0; e < 2; ++e)
        {
            lo_x = std::min<double>(lo_x, t.segments[4 * s + 2 * e]), hi_x = std::max<double>(hi_x, t.segments[4 * s + 2 * e]);
            lo_y = std::min<double>(lo_y, t.segments[4 * s + 2 * e + 1]), hi_y = std::max<double>(hi_y, t.segments[4 * s + 2 * e + 1]);
        }
    pl.h  = cfg.cell;
    pl.x0 = std::floor(lo_x - 1.0);
    pl.y0 = std::floor(lo_y - 1.0);
    pl.nx = std::max<int32_t>(1, static_cast<int32_t>(std::ceil((hi_x + 1.0 - pl.x0) / pl.h)));
    pl.ny = std::max<int32_t>(1, static_cast<int32_t>(std::ceil((hi_y + 1.0 - pl.y0) / pl.h)));
    pl.nb = cfg.bins;
    pl.rb = static_cast<double>(cfg.range) + 1.0;
    if (static_cast<int64_t>(pl.nx) * pl.ny > (1 << 24))
    {
        err = "beam grid has too many cells";
        return false;
    }
    // covered cells: everything within (lane half-width + 4 px) of a centre-line point
    pl.rows.assign(static_cast<size_t>(pl.nx) * pl.ny, 0xffffffffu);
    pl.covered.clear();
    for (int32_t i = 0; i < n; ++i)
    {
        const double r   = std::max(t.w_left[i], t.w_right[i]) + 4.0;
        const int32_t ix0 = std::max<int32_t>(0, static_cast<int32_t>(std::floor((t.x[i] - r - pl.x0) / pl.h)));
        const int32_t ix1 = std::min<int32_t>(pl.nx - 1, static_cast<int32_t>(std::floor((t.x[i] + r - pl.x0) / pl.h)));
        const int32_t iy0 = std::max<int32_t>(0, static_cast<int32_t>(std::floor((t.y[i] - r - pl.y0) / pl.h)));
        const int32_t iy1 = std::min<int32_t>(pl.ny - 1, static_cast<int32_t>(std::floor((t.y[i] + r - pl.y0) / pl.h)));
        for (int32_t iy = iy0; iy <= iy1; ++iy)
            for (int32_t ix = ix0; ix <= ix1; ++ix)
            { // cells that touch the disc
                const double qx = std::min(std::max<double>(t.x[i], pl.x0 + ix * pl.h), pl.x0 + (ix + 1) * pl.h);
                const double qy = std::min(std::max<double>(t.y[i], pl.y0 + iy * pl.h), pl.y0 + (iy + 1) * pl.h);
                if ((qx - t.x[i]) * (qx - t.x[i]) + (qy - t.y[i]) * (qy - t.y[i]) <= r * r)
                    pl.rows[static_cast<size_t>(iy) * pl.nx + ix] = 0;
            }
    }
    for (size_t c = 0; c < pl.rows.size(); ++c)
        if (pl.rows[c] == 0)
        {
            pl.rows[c] = static_cast<uint32_t>(pl.covered.size());
            pl.covered.push_back(static_cast<uint32_t>(c));
        }
    // the rows and entries alone already pass the 32-bit offsets of beam_layout: fail before any list is built
    if (sizeof(BeamHeader) + pl.rows.size() * 4 + pl.covered.size() * static_cast<size_t>(pl.nb) * 16 >= 0xffffffffull)
    {
        err = "beam table too large";
        return false;
    }
    return true;
}

bool beam_layout(const BeamPlan &pl, const BeamConfig &cfg, size_t n_items, int32_t n_segments, BeamHeader &h, std::string &err)
{
    if (n_segments < 1 || n_segments > 0xffff)
    {
        err = "beam tables index segments with 16 bits";
        return false;
    }
    if (n_items / 4 >= 0xffffffffull)
    {
        err = "beam table too large";
        return false;
    }
    h    = BeamHeader{};
    h.x0 = static_cast<float>(pl.x0), h.y0 = static_cast<float>(pl.y0);
    h.h = cfg.cell, h.inv_h = 1.0f / cfg.cell;
    h.nx = pl.nx, h.ny = pl.ny, h.nb = pl.nb;
    h.bin_scale = static_cast<float>(pl.nb / (2.0 * M_PI));
    h.rb        = static_cast<float>(pl.rb);
    h.tag       = (kBeamFormat << 16) | static_cast<uint32_t>(n_segments);
    h.n_rows    = static_cast<uint32_t>(pl.covered.size());
    h.n_chunks  = static_cast<uint32_t>(n_items / 4);
    size_t off  = sizeof(BeamHeader);
    h.off_rows  = static_cast<uint32_t>(off);
    off += (pl.rows.size() * 4 + 15) / 16 * 16;
    h.off_entries = static_cast<uint32_t>(off);
    off += pl.covered.size() * static_cast<size_t>(pl.nb) * 16;
    h.off_items = static_cast<uint32_t>(off);
    off += (n_items * 2 + 15) / 16 * 16;
    if (off >= 0xffffffffull)
    {
        err = "beam table too large";
        return false;
    }
    h.bytes = static_cast<uint32_t>(off);
    return true;
}

bool beam_assemble(const BeamPlan &pl, const BeamConfig &cfg, const uint32_t *entries, const uint16_t *items, size_t n_items,
                   int32_t n_segments, std::vector<uint8_t> &blob, std::string &err)
{
    BeamHeader h;
    if (!beam_layout(pl, cfg, n_items, n_segments, h, err))
        return false;
    blob.assign(h.bytes, 0);
    std::memcpy(blob.data(), &h, sizeof h);
    std::memcpy(blob.data() + h.off_rows, pl.rows.data(), pl.rows.size() * 4);
    std::memcpy(blob.data() + h.off_entries, entries, pl.covered.size() * static_cast<size_t>(pl.nb) * 16);
    if (n_items)
        std::memcpy(blob.data() + h.off_items, items, n_items * 2);
    return true;
}

bool build_beam_table(const Track &t, const BeamConfig &cfg, std::vector<uint8_t> &blob, std::string &err)
{
    BeamPlan pl;
    if (!beam_plan(t, cfg, pl, err))
        return false;
    const int32_t ns = t.n_segments();
    Builder b{t, cfg};
    b.h = pl.h, b.x0 = pl.x0, b.y0 = pl.y0, b.nx = pl.nx, b.ny = pl.ny, b.nb = pl.nb, b.rb = pl.rb;
    b.dth = kBeamAngleMargin;
    b.seg_mid.resize(ns), b.seg_half.resize(ns);
    for (int32_t s = 0; s < ns; ++s)
    {
        const float *g = &t.segments[4 * static_cast<size_t>(s)];
        b.seg_mid[s]   = {0.5 * (static_cast<double>(g[0]) + g[2]), 0.5 * (static_cast<double>(g[1]) + g[3])};
        b.seg_half[s]  = 0.5 * std::hypot(static_cast<double>(g[2]) - g[0], static_cast<double>(g[3]) - g[1]);
    }
    const double dbin = 2.0 * M_PI / b.nb;
    b.edge_lo.resize(b.nb), b.edge_hi.resize(b.nb), b.sample_dir.resize(2 * static_cast<size_t>(b.nb));
    for (int32_t k = 0; k < b.nb; ++k)
    {
        b.edge_lo[k] = {std::cos(k * dbin - b.dth), std::sin(k * dbin - b.dth)};
        b.edge_hi[k] = {std::cos((k + 1) * dbin + b.dth), std::sin((k + 1) * dbin + b.dth)};
        b.sample_dir[2 * k]     = {std::cos(k * dbin), std::sin(k * dbin)};
        b.sample_dir[2 * k + 1] = {std::cos((k + 0.5) * dbin), std::sin((k + 0.5) * dbin)};
    }
    const auto         &covered = pl.covered;
    std::vector<Row>    built(covered.size());
    std::atomic<size_t> next{0};
    unsigned            nthreads = cfg.threads > 0 ? static_cast<unsigned>(cfg.threads) : std::thread::hardware_concurrency();
    nthreads                     = std::max(1u, std::min(nthreads, 64u));
    auto worker = [&]() {
        Scratch sc;
        for (;;)
        {
            const size_t i = next.fetch_add(1);
            if (i >= covered.size())
                break;
            b.build_row(static_cast<int32_t>(covered[i] % b.nx), static_cast<int32_t>(covered[i] / b.nx), built[i], sc);
        }
    };
    if (nthreads == 1)
        worker();
    else
    {
        std::vector<std::thread> pool;
        for (unsigned k = 0; k < nthreads; ++k)
            pool.emplace_back(worker);
        for (auto &th : pool)
            th.join();
    }
    size_t n_items = 0;
    for (auto &r : built)
        n_items += r.items.size();
    std::vector<uint32_t> entries(covered.size() * static_cast<size_t>(b.nb) * 4);
    std::vector<uint16_t> items(n_items);
    size_t                cursor = 0;
    for (size_t r = 0; r < built.size(); ++r)
    {
        for (int32_t k = 0; k < b.nb; ++k)
        {
            uint32_t *e = &entries[4 * (r * b.nb + k)];
            e[0]        = built[r].inl[2 * k];
            e[1]        = built[r].inl[2 * k + 1];
            e[2]        = static_cast<uint32_t>((cursor + built[r].first[k]) / 4);
            e[3]        = built[r].meta[k];
        }
        if (!built[r].items.empty())
            std::memcpy(items.data() + cursor, built[r].items.data(), built[r].items.size() * 2);
        cursor += built[r].items.size();
    }
    return beam_assemble(pl, cfg, entries.data(), items.data(), n_items, ns, blob, err);
}

bool beam_lookup(const std::vector<uint8_t> &blob, float x, float y, float angle, std::vector<uint16_t> &out, float &d_out,
                 float *d1_out, int32_t *n_inline)
{
    out.clear();
    if (blob.size() < sizeof(BeamHeader))
        return false;
    BeamHeader h;
    std::memcpy(&h, blob.data(), sizeof h);
    // the device's arithmetic: binary32, same operation order (ok_kernels.cuh beam_row / beam_bin)
    const float fx = (x - h.x0) * h.inv_h, fy = (y - h.y0) * h.inv_h;
    if (!(fx >= 0.0f && fy >= 0.0f && fx < static_cast<float>(h.nx) && fy < static_cast<float>(h.ny)))
        return false;
    if (!(std::fabs(angle) < kBeamMaxAngle))
        return false;
    const int32_t ix = static_cast<int32_t>(fx), iy = static_cast<int32_t>(fy);
    uint32_t      row;
    std::memcpy(&row, blob.data() + h.off_rows + 4 * (static_cast<size_t>(iy) * h.nx + ix), 4);
    if (row == 0xffffffffu)
        return false;
    const int32_t bin = static_cast<int32_t>(std::floor(angle * h.bin_scale)) & (h.nb - 1);
    uint32_t      e[4];
    std::memcpy(e, blob.data() + h.off_entries + 16 * (static_cast<size_t>(row) * h.nb + bin), 16);
    const uint32_t n_rest = beam_meta_rest(e[3]);
    d_out                 = beam_meta_d(e[3], h.rb);
    if (d1_out)
        *d1_out = n_rest ? beam_meta_d1(e[3], h.rb) : d_out;
    if ((h.tag >> 16) != kBeamFormat)
        return false;
    const uint16_t null_seg = static_cast<uint16_t>(h.tag & 0xffffu); // padding value: the blob's null segment
    const uint16_t in4[4]   = {static_cast<uint16_t>(e[0] & 0xffffu), static_cast<uint16_t>(e[0] >> 16),
                               static_cast<uint16_t>(e[1] & 0xffffu), static_cast<uint16_t>(e[1] >> 16)};
    for (int i = 0; i < kBeamInline; ++i)
        if (in4[i] != null_seg)
            out.push_back(in4[i]);
    if (n_inline)
        *n_inline = static_cast<int32_t>(out.size());
    if (n_rest)
    {
        const uint16_t *src = reinterpret_cast<const uint16_t *>(blob.data() + h.off_items) + 4 * static_cast<size_t>(e[2]);
        for (size_t i = 0; i < 4 * static_cast<size_t>(n_rest); ++i)
            if (src[i] != null_seg)
                out.push_back(src[i]);
    }
    return true;
}

bool beam_validate(const std::vector<uint8_t> &blob, int32_t n_segments, std::string &err)
{
    auto bad = [&](const char *what) {
        err = std::string("beam table rejected: ") + what;
        return false;
    };
    if (blob.size() < sizeof(BeamHeader))
        return bad("too small");
    BeamHeader h;
    std::memcpy(&h, blob.data(), sizeof h);
    if ((h.tag >> 16) != kBeamFormat || static_cast<int32_t>(h.tag & 0xffffu) != n_segments)
        return bad("format or segment count");
    if (h.bytes != blob.size() || h.nx < 1 || h.ny < 1 || h.nb < 8 || h.nb > 1024 || (h.nb & (h.nb - 1)))
        return bad("header");
    const uint64_t cells = static_cast<uint64_t>(h.nx) * static_cast<uint64_t>(h.ny);
    if (cells > (1u << 24))
        return bad("grid");
    const uint64_t rows_end = static_cast<uint64_t>(h.off_rows) + 4 * cells;
    const uint64_t ent_end  = static_cast<uint64_t>(h.off_entries) + 16ull * h.n_rows * static_cast<uint64_t>(h.nb);
    const uint64_t item_end = static_cast<uint64_t>(h.off_items) + 8ull * h.n_chunks;
    if (h.off_rows < sizeof(BeamHeader) || rows_end > h.off_entries || ent_end > h.off_items || item_end > h.bytes ||
        (h.off_entries & 15u) || (h.off_items & 7u))
        return bad("section offsets");
    const uint32_t *rows = reinterpret_cast<const uint32_t *>(blob.data() + h.off_rows);
    for (uint64_t c = 0; c < cells; ++c)
        if (rows[c] != 0xffffffffu && rows[c] >= h.n_rows)
            return bad("row index");
    const uint32_t *ent = reinterpret_cast<const uint32_t *>(blob.data() + h.off_entries);
    const uint64_t  n_e = static_cast<uint64_t>(h.n_rows) * static_cast<uint64_t>(h.nb);
    for (uint64_t i = 0; i < n_e; ++i)
    {
        const uint32_t *e = ent + 4 * i;
        if ((e[0] & 0xffffu) > static_cast<uint32_t>(n_segments) || (e[0] >> 16) > static_cast<uint32_t>(n_segments) ||
            (e[1] & 0xffffu) > static_cast<uint32_t>(n_segments) || (e[1] >> 16) > static_cast<uint32_t>(n_segments))
            return bad("inline segment index");
        const uint32_t n_rest = beam_meta_rest(e[3]);
        if (n_rest && static_cast<uint64_t>(e[2]) + n_rest > h.n_chunks)
            return bad("chunk range");
    }
    const uint16_t *items = reinterpret_cast<const uint16_t *>(blob.data() + h.off_items);
    for (uint64_t i = 0; i < 4ull * h.n_chunks; ++i)
        if (items[i] > n_segments)
            return bad("segment index");
    return true;
}

} // namespace ok
