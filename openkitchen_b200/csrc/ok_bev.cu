// ok_bev.cu -- bird's-eye-view rasters at arbitrary poses (ok_bev_query): the semantic class of every pixel of a
// pose-aligned image (ok_bev.cuh states the sample points and the classes), in a translation unit of its own.
//
// The table.  Per track the y axis is cut into bands of kBevBand px from y0; per (band, loop) a list holds the loop's
// edges (i, j = i - 1 cyclic, the closing edge included, horizontal edges left out: they never satisfy the PNPOLY y
// test) whose y-range [min y, max y] meets the band.  A point is sent to band floor((py - y0) * kBevInvBand) in binary32
// on the device and in the builder alike; that map is monotone in py, so an edge whose y test can hold at py (min y <=
// py < max y) is listed in py's band, and a py outside every band fails every y test.  Each list is sorted by xhi,
// descending, so a pixel stops at the first entry with px >= xhi.
//
// Exactness of xlo / xhi.  When the y test holds, the PNPOLY abscissa is X = fl(fl(fl(fl(x_j - x_i) * fl(p_y - y_i)) /
// fl(y_j - y_i)) + x_i), and its exact counterpart X* = x_i + (x_j - x_i) t with t = (p_y - y_i) / (y_j - y_i) in [0, 1]
// lies in [min x, max x].  With u = 2^-24, D = |x_j - x_i| and M = max(|x_i|, |x_j|): each of the five roundings before
// the last one adds a relative error of at most u to a factor of D t, so the quotient is D t within 5.0002 u D; the last
// sum adds u (M + 5.0002 u D).  Underflow adds at most 2^-150 per rounding, which the division by |y_j - y_i| >= 2^-60
// magnifies to 2^-89.  So |X - X*| < m = 2^-19 (D + M) + 2^-80, and with xlo <= min x - m and xhi >= max x + m (rounded
// outwards to binary32): px < xlo implies px < X (the edge is crossed), px >= xhi implies px >= X (it is not).  Edges
// with |y_j - y_i| < 2^-60 (none on the 23 tracks) get xlo = -inf, xhi = +inf: always the exact expression.
//
// Mapping: a thread computes kBevBytes consecutive output bytes (consecutive columns of a row, or the end of one row
// and the start of the next) and stores them with one aligned 32-bit store, so a warp writes 128 consecutive bytes;
// the chunks are aligned to the output address, and only a chunk at either end of the output is stored byte by byte.
// Nothing is staged: the lists come through L1 / L2, and neighbouring pixels read the same ones.
#include "ok_bev.cuh"
#include "ok_device.cuh"
#include "ok_track.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace ok
{

namespace
{
// the band coordinate of y, on the host exactly as on the device: one binary32 subtraction, one exact scaling
float bev_band_coord(float y, float y0)
{
    return (y - y0) * kBevInvBand;
}
float round_down(double v)
{
    float f = static_cast<float>(v);
    return static_cast<double>(f) > v ? std::nextafter(f, -INFINITY) : f;
}
float round_up(double v)
{
    float f = static_cast<float>(v);
    return static_cast<double>(f) < v ? std::nextafter(f, INFINITY) : f;
}
struct Entry
{
    float4 a;
    float2 b;
};
} // namespace

void build_bev_table(const std::vector<Track> &tracks, BevTableHost &out)
{
    out           = BevTableHost{};
    out.n_tracks  = static_cast<int32_t>(tracks.size());
    std::vector<BevTrack> heads(tracks.size());
    std::vector<uint32_t> starts;
    std::vector<Entry>    entries;
    for (size_t t = 0; t < tracks.size(); ++t)
    {
        const Track              &tr      = tracks[t];
        const std::vector<float> *loops[] = {&tr.left_inner, &tr.left_outer, &tr.right_inner, &tr.right_outer};
        float                     ylo = INFINITY, yhi = -INFINITY;
        for (const std::vector<float> *p : loops)
            for (size_t i = 1; i < p->size(); i += 2)
                ylo = std::min(ylo, (*p)[i]), yhi = std::max(yhi, (*p)[i]);
        BevTrack &h  = heads[t];
        h.y0         = ylo - kBevBand;
        h.n_bands    = static_cast<int32_t>(bev_band_coord(yhi, h.y0)) + 1;
        h.off_starts = static_cast<uint32_t>(starts.size());
        h.pad        = 0;
        std::vector<std::vector<Entry>> lists(static_cast<size_t>(h.n_bands) * kBevLoops);
        for (int L = 0; L < kBevLoops; ++L)
        {
            const std::vector<float> &p = *loops[L];
            const int                 n = static_cast<int>(p.size() / 2);
            for (int i = 0; i < n; ++i)
            {
                const int   j  = i == 0 ? n - 1 : i - 1;
                const float xi = p[2 * i], yi = p[2 * i + 1], xj = p[2 * j], yj = p[2 * j + 1];
                if (yi == yj)
                    continue;
                const double d = std::fabs(static_cast<double>(xj) - xi), m = std::max(std::fabs(xi), std::fabs(xj));
                const double margin = std::ldexp(d + m, -19) + std::ldexp(1.0, -80);
                const bool   tiny   = std::fabs(static_cast<double>(yj) - yi) < std::ldexp(1.0, -60);
                Entry        e;
                e.a.x = yi, e.a.y = yj;
                e.a.z = tiny ? -INFINITY : round_down(std::min(xi, xj) - margin);
                e.a.w = tiny ? INFINITY : round_up(std::max(xi, xj) + margin);
                e.b   = make_float2(xi, xj);
                const int b0 = static_cast<int>(bev_band_coord(std::min(yi, yj), h.y0));
                const int b1 = static_cast<int>(bev_band_coord(std::max(yi, yj), h.y0));
                for (int b = b0; b <= b1; ++b)
                    lists[static_cast<size_t>(b) * kBevLoops + L].push_back(e);
            }
        }
        for (std::vector<Entry> &l : lists)
        {
            std::stable_sort(l.begin(), l.end(), [](const Entry &u, const Entry &v) { return u.a.w > v.a.w; });
            starts.push_back(static_cast<uint32_t>(entries.size()));
            entries.insert(entries.end(), l.begin(), l.end());
        }
        starts.push_back(static_cast<uint32_t>(entries.size())); // the end of the track's last list
    }
    out.entries = entries.size();
    const auto align16 = [](size_t v) { return (v + 15) / 16 * 16; };
    out.off_starts     = align16(sizeof(BevTrack) * heads.size());
    out.off_a          = align16(out.off_starts + sizeof(uint32_t) * starts.size());
    out.off_b          = out.off_a + sizeof(float4) * entries.size();
    out.bytes.assign(std::max<size_t>(out.off_b + sizeof(float2) * entries.size(), 16), 0);
    std::memcpy(out.bytes.data(), heads.data(), sizeof(BevTrack) * heads.size());
    std::memcpy(out.bytes.data() + out.off_starts, starts.data(), sizeof(uint32_t) * starts.size());
    for (size_t i = 0; i < entries.size(); ++i)
    {
        std::memcpy(out.bytes.data() + out.off_a + sizeof(float4) * i, &entries[i].a, sizeof(float4));
        std::memcpy(out.bytes.data() + out.off_b + sizeof(float2) * i, &entries[i].b, sizeof(float2));
    }
}

// the class of point (px, py) on the track whose bands are `bt`
__device__ __forceinline__ uint32_t bev_class(const BevTableView &tb, const BevTrack &bt, float px, float py)
{
    const float bc = fmul(fsub(py, bt.y0), kBevInvBand);
    if (!(bc >= 0.0f && bc < static_cast<float>(bt.n_bands))) // below or above every edge, or NaN: no y test holds
        return OK_BEV_OFF;
    const uint32_t *st = tb.starts + bt.off_starts + static_cast<uint32_t>(bc) * kBevLoops;
    OK_CHECK(bt.off_starts + static_cast<uint32_t>(bc) * kBevLoops + kBevLoops < tb.n_starts);
    int             k  = 0;
#pragma unroll 1
    for (int L = 0; L < kBevLoops; ++L)
    {
        const uint32_t end    = __ldg(st + L + 1);
        int            inside = 0;
        OK_CHECK(end <= tb.n_entries);
        for (uint32_t i = __ldg(st + L); i < end; ++i)
        {
            const float4 a = __ldg(tb.a + i); // y_i, y_j, xlo, xhi
            if (px >= a.w)
                break; // and so for every later entry of the list
            if ((a.x > py) != (a.y > py))
            {
                bool cross = px < a.z;
                if (!cross)
                {
                    const float2 b = __ldg(tb.b + i); // x_i, x_j
                    cross          = px < fadd(fdiv(fmul(fsub(b.y, b.x), fsub(py, a.x)), fsub(a.y, a.x)), b.x);
                }
                inside ^= cross;
            }
        }
        k += inside;
    }
    return k == 2 ? OK_BEV_LANE : (k & 1) ? OK_BEV_WALL : OK_BEV_OFF;
}

__global__ void __launch_bounds__(kBevBlock) bev_query_kernel(const BevQueryParams q)
{
    const int64_t hw    = static_cast<int64_t>(q.height) * q.width;
    const int64_t total = q.n * hw;
    const int     mis   = static_cast<int>(reinterpret_cast<uintptr_t>(q.out) & (kBevBytes - 1));
    const int64_t chunk = static_cast<int64_t>(blockIdx.x) * kBevBlock + threadIdx.x;
    const int64_t e0    = chunk * kBevBytes - mis; // output byte of the chunk's first byte (negative: before the output)
    if (e0 >= total)
        return;
    const int     j0 = e0 < 0 ? static_cast<int>(-e0) : 0;
    const int     j1 = static_cast<int>(min(static_cast<int64_t>(kBevBytes), total - e0));
    const int64_t e  = e0 + j0;
    int64_t       k  = e / hw;
    const int     rm = static_cast<int>(e - k * hw);
    int           r = rm / q.width, c = rm - r * q.width;
    const float   hc = fmul(0.5f, static_cast<float>(q.height - 1)), wc = fmul(0.5f, static_cast<float>(q.width - 1));
    int64_t       pk = -1;
    float         x = 0.0f, y = 0.0f, rs = 0.0f, rc = 0.0f;
    BevTrack      bt{};
    uint32_t      word = 0;
    for (int j = j0; j < j1; ++j)
    {
        if (k != pk)
        { // this pixel starts a new pose
            pk        = k;
            int32_t t = q.track ? q.track[k] : 0;
            t         = min(max(t, 0), q.n_tracks - 1);
            OK_CHECK(k < q.n);
            x = q.x[k], y = q.y[k];
            sincosf(fmul(OK_DEG2RAD, q.rot[k]), rs, rc);
            bt = q.table.tracks[t];
        }
        const float f  = fadd(fmul(fsub(hc, static_cast<float>(r)), q.scale), q.ahead); // forward
        const float l  = fmul(fsub(static_cast<float>(c), wc), q.scale);                 // to the right
        const float px = fadd(x, fsub(fmul(f, rc), fmul(l, rs)));
        const float py = fadd(y, fadd(fmul(f, rs), fmul(l, rc)));
        word |= bev_class(q.table, bt, px, py) << (8 * j);
        if (++c == q.width)
        {
            c = 0;
            if (++r == q.height)
                r = 0, ++k;
        }
    }
    if (j0 == 0 && j1 == kBevBytes)
        reinterpret_cast<uint32_t *>(q.out - mis)[chunk] = word;
    else
        for (int j = j0; j < j1; ++j)
            q.out[e0 + j] = static_cast<uint8_t>(word >> (8 * j));
}

cudaError_t launch_bev_query(const BevQueryParams &q, cudaStream_t stream)
{
    const int64_t total  = q.n * q.height * q.width;
    const int64_t mis    = static_cast<int64_t>(reinterpret_cast<uintptr_t>(q.out) & (kBevBytes - 1));
    const int64_t chunks = (total + mis + kBevBytes - 1) / kBevBytes;
    const int64_t blocks = (chunks + kBevBlock - 1) / kBevBlock;
    bev_query_kernel<<<static_cast<unsigned>(blocks), kBevBlock, 0, stream>>>(q);
    return cudaGetLastError();
}

cudaError_t violations_bev(unsigned long long *count)
{
    return cudaMemcpyFromSymbol(count, g_violations, sizeof *count);
}
} // namespace ok
