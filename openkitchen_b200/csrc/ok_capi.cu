// ok_capi.cu -- implementation of the C ABI (include/openkitchen_b200.h) over the sm_100a kernels.
// Host side of the product: owns device memory, uploads the tilings (ok_schedule.hpp), launches.  No CPU
// fallback exists: without a CUDA device every compute entry point returns OK_ERR_NO_DEVICE.
#include "../../include/openkitchen_b200.h"

#include "ok_beam.hpp"
#include "ok_kernels.cuh"
#include "ok_step.cuh"
#include "ok_track.hpp"

#include <nvtx3/nvToolsExt.h> // header-only; ranges only with OK_NVTX=1
#include <cuda.h> // types of the one driver entry point used (cuStreamWriteValue32), looked up at run time: libcuda is not linked

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <fcntl.h>
#include <map>
#include <sys/stat.h>
#include <thread>
#include <type_traits>
#include <unistd.h>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

namespace
{
thread_local std::string g_last_error;

int fail(int code, const std::string &msg)
{
    g_last_error = msg;
    return code;
}

#define OK_CUDA(expr)                                                                                                  \
    do                                                                                                                 \
    {                                                                                                                  \
        cudaError_t err__ = (expr);                                                                                    \
        if (err__ != cudaSuccess)                                                                                      \
            return fail(OK_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(err__));                           \
    } while (0)

// NVTX range around a library call (SURVEY 5, tracing): visible in Nsight Systems / Compute timelines; OK_NVTX=1 turns it on
struct NvtxRange
{
    bool on;
    explicit NvtxRange(const char *name)
    {
        static const bool enabled = [] {
            const char *v = std::getenv("OK_NVTX");
            return v && std::atoi(v) != 0;
        }();
        on = enabled;
        if (on)
            nvtxRangePushA(name);
    }
    ~NvtxRange()
    {
        if (on)
            nvtxRangePop();
    }
    NvtxRange(const NvtxRange &)            = delete;
    NvtxRange &operator=(const NvtxRange &) = delete;
};

struct DeviceGuard
{
    int  prev{-1};
    bool active{false};
    explicit DeviceGuard(int dev)
    {
        if (dev >= 0 && cudaGetDevice(&prev) == cudaSuccess && prev != dev)
        {
            cudaSetDevice(dev);
            active = true;
        }
    }
    ~DeviceGuard()
    {
        if (active)
            cudaSetDevice(prev);
    }
};

constexpr int kMaxBatchAgents = 256;

struct BufferDesc
{
    int32_t dtype;
    int32_t per_ray; // 0: [N], 1: [N,R], 2: [N,R,2]
};

BufferDesc describe(int which)
{
    switch (which)
    {
    case OK_BUF_CRASHED:
    case OK_BUF_TIMED_OUT:
    case OK_BUF_DONE: return {OK_DTYPE_U8, 0};
    case OK_BUF_SS_CTR: return {OK_DTYPE_U32, 0};
    case OK_BUF_TRACK_ID:
    case OK_BUF_NEAREST_IDX:
    case OK_BUF_PREV_IDX:
    case OK_BUF_RESET_PT: return {OK_DTYPE_I32, 0};
    case OK_BUF_HIT_ABS:
    case OK_BUF_HIT_REL: return {OK_DTYPE_F32, 2};
    case OK_BUF_OBS:
    case OK_BUF_HIT_T: return {OK_DTYPE_F32, 1};
    case OK_BUF_HIT_SEG: return {OK_DTYPE_I32, 1};
    default: return {OK_DTYPE_F32, 0};
    }
}

size_t dtype_size(int32_t dt)
{
    return dt == OK_DTYPE_U8 ? 1 : 4;
}
} // namespace

// a beam table in device memory, shared by every env of the process on that device
struct DeviceBlob
{
    uint8_t *ptr{nullptr};
    size_t   bytes{0};
    int      device{0};
    DeviceBlob(uint8_t *p, size_t b, int d) : ptr(p), bytes(b), device(d)
    {
    }
    DeviceBlob(const DeviceBlob &) = delete;
    DeviceBlob &operator=(const DeviceBlob &) = delete;
    ~DeviceBlob()
    {
        if (ptr)
        {
            DeviceGuard g(device);
            cudaFree(ptr); // an error after the runtime has shut down is harmless
        }
    }
};

namespace
{
// owners of the CUDA resources of an env: freed (destroyed) when the owner is reset or goes away
struct CudaFree
{
    void operator()(void *p) const
    {
        cudaFree(p);
    }
};
template <typename T> using DevPtr = std::unique_ptr<T, CudaFree>;
struct StreamDestroy
{
    void operator()(cudaStream_t s) const
    {
        cudaStreamDestroy(s);
    }
};
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
struct EventDestroy
{
    void operator()(cudaEvent_t ev) const
    {
        cudaEventDestroy(ev);
    }
};
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;

// replaces what `p` holds by `count` uninitialised elements of device memory (the old block is freed first)
template <typename T> cudaError_t dev_alloc(DevPtr<T> &p, size_t count)
{
    p.reset();
    T *raw = nullptr;
    const cudaError_t rc = cudaMalloc(&raw, sizeof(T) * count);
    p.reset(raw);
    return rc;
}

cudaError_t make_stream(Stream &s)
{
    cudaStream_t raw = nullptr;
    const cudaError_t rc = cudaStreamCreateWithFlags(&raw, cudaStreamNonBlocking);
    s.reset(raw);
    return rc;
}

cudaError_t make_event(Event &ev)
{
    cudaEvent_t raw = nullptr;
    const cudaError_t rc = cudaEventCreateWithFlags(&raw, cudaEventDisableTiming);
    ev.reset(raw);
    return rc;
}

// a tiling in device memory: the table the kernel reads, its length, and the grid that runs it
struct Schedule
{
    DevPtr<ok::Tile> d;
    int32_t          n{0}, grid{0};
};

// cost feedback for the beam tiling (ok_balance_schedule): the kernel leaves every tile's ray-phase / other time in
// d_tile_ns, and reweigh_runs re-cuts the tiles from them.  The table is allocated once, at `capacity` tiles, and
// rewritten in place: a CUDA graph captured earlier keeps reading it.
struct BeamFeedback
{
    std::vector<ok::TileRun> runs;
    std::vector<ok::Tile>    tiles; // host copy of the beam schedule's table
    bool                     weighted{false};
    int32_t                  target{0}, capacity{0};
    DevPtr<uint32_t>         d_tile_ns;
    uint64_t                 launches{0};
};

// everything ok_alloc_agents creates for one population: ok_alloc_agents and free_agents replace it as a whole
struct Agents
{
    DevPtr<uint8_t>  slab;
    DevPtr<float>    ray_deg;
    DevPtr<uint16_t> ray_order;
    DevPtr<int32_t>  sched;
    Schedule         tiles; // the grid-walk kernel's tiling
    // the beam kernel's batches are not limited by per-ray scratch: its own batch size, tiling and grid
    Schedule     beam;
    BeamFeedback feedback;
    DevPtr<ok::FirstTile> first_beam; // the first tile of every CTA with its track record (ok_device.cuh)
    int32_t               first_capacity{0};
    bool                  first_dirty{true};
    // ok_step_host's tiling: several tiles per CTA, so that a tile's observations cross PCIe while the next one is computed
    Schedule e2e;
    Schedule q16; // ok_step_host_q16's tiling: half the bytes per tile, fewer and larger tiles pay
    // ... with flusher CTAs (obs_flush_kernel) on SMs of their own
    DevPtr<uint32_t> tile_flag;
    // ok_step_host: device stage of the caller's two mapped action arrays, filled by the copy engine on act_stream next to
    // the running kernel, + the word the stream sets to this launch's target when both copies have landed
    DevPtr<float>    act_stage;
    DevPtr<uint32_t> act_ready;
    uint32_t         act_ready_target{0};
    DevPtr<unsigned long long> stats; // ok_debug_stats: allocated on first use
    DevPtr<unsigned long long> trace; // ok_debug_trace
    int32_t                    trace_tiles{0};
};
} // namespace

struct OkEnv
{
    OkConfig               cfg{};
    bool                   has_device{false};
    int                    num_sms{0};
    size_t                 max_blob{0};
    std::vector<ok::Track> tracks;
    // device track arena
    DevPtr<uint8_t>      d_arena;
    DevPtr<ok::TrackRef> d_track_refs;
    size_t        arena_bytes{0};
    size_t        max_blob_used{0};
    bool          arena_dirty{true};
    // beam tables (OK_RAYCAST_BEAM): one blob per track in global memory
    std::vector<std::shared_ptr<const std::vector<uint8_t>>> beams;     // host copies (host-only envs, ok_beam_lookup)
    std::vector<std::shared_ptr<const struct DeviceBlob>>    beams_dev; // what the kernels read; shared between envs
    bool          arena_has_beams{false};
    std::vector<ok::TrackRef> h_track_refs; // host copy of d_track_refs
    // agents
    int64_t              n_agents{0};
    int32_t              rays{0};
    Agents               ag;
    void                *d_buf[OK_BUF_COUNT]{};
    size_t               buf_off[OK_BUF_COUNT]{}; // offsets of the buffers inside the slab
    int32_t              batch_agents{0};
    int                  auto_balance{1};
    float                balance_before{0.0f}, balance_after{0.0f}; // predicted slowest-tile / mean-tile cost of the last rebalancing
    int32_t              e2e_flushers{0};
    uint32_t             flag_epoch{0};
    bool                 act_stage_on{true}; // OK_ACT_STAGE=0: every tile reads the mapping (A/B)
    int                  actor_dyn_max{0};   // dynamic shared memory the fused actor + step kernel may use
    int32_t              batch_agents_beam{0};
    int32_t              ctas_per_sm_beam{1};
    bool                 beam_staged{true}; // which shape of the beam kernel this population runs (ok_step.cuh)
    int32_t              beam_block{1024};
    int                  smem_optin{0};
    std::vector<int32_t> h_track_id;
    // created on first use, kept until ok_destroy
    DevPtr<uint8_t>            d_stage; // staging for the *_host entry points
    size_t                     stage_bytes{0};
    DevPtr<unsigned long long> d_counters; // ok_population_counters
    Stream                     act_stream; // ok_step_host's action copies
    Event                      ev_act;
    Stream                     flush_stream; // the flusher CTAs' side stream and its fork / join events
    Event                      ev_fork, ev_join;
    // stats
    uint64_t launches{0};
    size_t   smem{0}, smem_beam{0};
};

namespace
{
size_t buffer_bytes(const OkEnv *e, int which)
{
    const BufferDesc d = describe(which);
    size_t           n = static_cast<size_t>(e->n_agents);
    if (d.per_ray >= 1)
        n *= static_cast<size_t>(e->rays);
    if (d.per_ray == 2)
        n *= 2;
    return n * dtype_size(d.dtype);
}

void free_agents(OkEnv *e)
{
    e->ag = Agents{};
    for (auto &b : e->d_buf)
        b = nullptr;
    e->n_agents = 0, e->rays = 0;
}

// Beam tables are pure functions of (segments, cell, bins, range) and take ~0.1-1 s of host time per track.
// Two caches: one per process (envs over the same tracks share a table), and one on disk
// ($OK_BEAM_CACHE_DIR, default $TMPDIR/openkitchen_b200-cache-<uid>; OK_BEAM_CACHE=0 disables it) so that the ranks
// of one box -- which all need every table -- build each table once between them instead of once each.
uint64_t fnv1a(const void *ptr, size_t n, uint64_t h = 1469598103934665603ull)
{
    const uint8_t *b = static_cast<const uint8_t *>(ptr);
    for (size_t i = 0; i < n; ++i)
        h = (h ^ b[i]) * 1099511628211ull;
    return h;
}

std::string beam_cache_dir()
{
    if (const char *off = std::getenv("OK_BEAM_CACHE"))
        if (std::atoi(off) == 0)
            return "";
    std::string dir;
    if (const char *d = std::getenv("OK_BEAM_CACHE_DIR"))
        dir = d;
    else
    {
        const char *tmp = std::getenv("TMPDIR");
        dir             = std::string(tmp && *tmp ? tmp : "/tmp") + "/openkitchen_b200-cache-" + std::to_string(getuid());
    }
    ::mkdir(dir.c_str(), 0700);
    // the tables loaded from here steer device reads: only a real directory that belongs to this user and that nobody
    // else can write is trusted; anything else (a planted directory or symlink in a shared /tmp) disables the cache
    struct stat st
    {
    };
    if (::lstat(dir.c_str(), &st) != 0 || !S_ISDIR(st.st_mode) || st.st_uid != getuid() || (st.st_mode & (S_IWGRP | S_IWOTH)))
        return "";
    return dir;
}

struct BeamFileHeader
{
    char     magic[8]; // "OKBEAM02"
    uint64_t bytes, checksum;
};

bool beam_file_load(const std::string &path, std::vector<uint8_t> &blob, int32_t n_segments)
{
    FILE *f = std::fopen(path.c_str(), "rb");
    if (!f)
        return false;
    BeamFileHeader h{};
    bool           ok = std::fread(&h, sizeof h, 1, f) == 1 && std::memcmp(h.magic, "OKBEAM02", 8) == 0 && h.bytes >= sizeof(ok::BeamHeader) &&
              h.bytes < (1ull << 32);
    if (ok)
    {
        blob.resize(h.bytes);
        ok = std::fread(blob.data(), 1, h.bytes, f) == h.bytes && fnv1a(blob.data(), blob.size()) == h.checksum;
        // the kernels trust a table's indices: one that did not come from this process is checked structurally first
        std::string why;
        ok = ok && ok::beam_validate(blob, n_segments, why);
    }
    std::fclose(f);
    if (!ok)
        blob.clear();
    return ok;
}

void beam_file_save(const std::string &path, const std::vector<uint8_t> &blob)
{
    const std::string tmp = path + ".tmp." + std::to_string(getpid());
    FILE             *f   = std::fopen(tmp.c_str(), "wb");
    if (!f)
        return;
    BeamFileHeader h{};
    std::memcpy(h.magic, "OKBEAM02", 8);
    h.bytes    = blob.size();
    h.checksum = fnv1a(blob.data(), blob.size());
    const bool ok = std::fwrite(&h, sizeof h, 1, f) == 1 && std::fwrite(blob.data(), 1, blob.size(), f) == blob.size();
    std::fclose(f);
    if (ok && std::rename(tmp.c_str(), path.c_str()) == 0)
        return;
    std::remove(tmp.c_str());
}

std::string beam_key(const ok::Track &t, const ok::BeamConfig &cfg)
{
    uint64_t h = fnv1a(t.segments.data(), t.segments.size() * sizeof(float));
    h          = fnv1a(t.x.data(), t.x.size() * sizeof(float), h);
    h          = fnv1a(t.y.data(), t.y.size() * sizeof(float), h);
    h          = fnv1a(t.w_left.data(), t.w_left.size() * sizeof(float), h);
    h          = fnv1a(t.w_right.data(), t.w_right.size() * sizeof(float), h);
    char key[128];
    std::snprintf(key, sizeof key, "v%d-%016llx-%zu-%g-%d-%g", ok::kBeamBuildVersion, static_cast<unsigned long long>(h),
                  t.segments.size(), static_cast<double>(cfg.cell), cfg.bins, static_cast<double>(cfg.range));
    return key;
}

std::mutex                                                          g_beam_mu;
std::map<std::string, std::shared_ptr<const std::vector<uint8_t>>> g_beam_cache;

std::shared_ptr<const std::vector<uint8_t>> beam_cached(const std::string &key)
{
    std::lock_guard<std::mutex> lock(g_beam_mu);
    auto                        it = g_beam_cache.find(key);
    return it == g_beam_cache.end() ? nullptr : it->second;
}

std::shared_ptr<const std::vector<uint8_t>> beam_remember(const std::string &key, std::shared_ptr<std::vector<uint8_t>> blob)
{
    std::lock_guard<std::mutex> lock(g_beam_mu);
    size_t                      held = blob->size();
    for (auto &kv : g_beam_cache)
        held += kv.second->size();
    if (held > (size_t{12} << 30)) // envs keep their own references; this only bounds what the cache itself pins
        g_beam_cache.clear();
    g_beam_cache[key] = blob;
    return blob;
}

// `wait` = false: return nullptr (no error) when another process holds the track's build lock, so that the caller
// can build other tracks in the meantime; `wait` = true: wait for that process's file, or build after a timeout.
std::shared_ptr<const std::vector<uint8_t>> beam_table_for(const ok::Track &t, const ok::BeamConfig &cfg, bool wait, std::string &err)
{
    const std::string key = beam_key(t, cfg);
    if (auto hit = beam_cached(key))
        return hit;
    auto              blob = std::make_shared<std::vector<uint8_t>>();
    const std::string dir  = beam_cache_dir();
    const std::string path = dir.empty() ? "" : dir + "/beam-" + key + ".bin", lock = path + ".lock";
    bool              locked = false;
    if (!path.empty())
    {
        if (beam_file_load(path, *blob, t.n_segments()))
            return beam_remember(key, blob);
        const int fd = ::open(lock.c_str(), O_CREAT | O_EXCL | O_WRONLY, 0600);
        if (fd >= 0)
        {
            ::close(fd);
            locked = true;
        }
        else
        {
            struct stat st
            {
            };
            const bool stale = ::stat(lock.c_str(), &st) == 0 && std::time(nullptr) - st.st_mtime > 300;
            if (stale)
                std::remove(lock.c_str());
            else if (!wait)
                return nullptr; // someone else is building it
            else
                for (int i = 0; i < 2400 && ::stat(lock.c_str(), &st) == 0; ++i) // up to two minutes
                {
                    std::this_thread::sleep_for(std::chrono::milliseconds(50));
                    if (beam_file_load(path, *blob, t.n_segments()))
                        return beam_remember(key, blob);
                }
            if (beam_file_load(path, *blob, t.n_segments()))
                return beam_remember(key, blob);
        }
    }
    const bool built = ok::build_beam_table(t, cfg, *blob, err);
    if (built && !path.empty())
        beam_file_save(path, *blob);
    if (locked)
        std::remove(lock.c_str());
    if (!built)
    {
        if (err.empty())
            err = "beam table build failed";
        return nullptr;
    }
    return beam_remember(key, blob);
}

// never destroyed: at process exit the CUDA runtime may already be gone when static destructors run
std::map<std::string, std::shared_ptr<const DeviceBlob>> &g_beam_dev_cache = *new std::map<std::string, std::shared_ptr<const DeviceBlob>>();

// The track's table in the memory of `device`: built there by the kernel builder (ok_beam_gpu.cu); OK_BEAM_BUILDER=cpu
// (or a failure of the device builder) builds it on the host instead and uploads it.  `wait` as in beam_table_for.
std::shared_ptr<const DeviceBlob> beam_device_table_for(const ok::Track &t, const ok::BeamConfig &cfg, int device, bool wait,
                                                        std::string &err)
{
    const std::string key = beam_key(t, cfg) + "@" + std::to_string(device);
    {
        std::lock_guard<std::mutex> lock(g_beam_mu);
        auto                        it = g_beam_dev_cache.find(key);
        if (it != g_beam_dev_cache.end())
            return it->second;
    }
    std::shared_ptr<const DeviceBlob> out;
    const char                       *force = std::getenv("OK_BEAM_BUILDER");
    if (!(force && std::strcmp(force, "cpu") == 0))
    {
        uint8_t    *d = nullptr;
        size_t      bytes = 0;
        std::string gerr;
        if (ok::build_beam_table_device(t, cfg, device, &d, &bytes, gerr))
            out = std::make_shared<DeviceBlob>(d, bytes, device);
        else if (force && std::strcmp(force, "gpu") == 0)
        {
            err = "device builder: " + gerr;
            return nullptr;
        }
    }
    if (!out)
    {
        auto host = beam_table_for(t, cfg, wait, err);
        if (!host)
            return nullptr;
        DeviceGuard g(device);
        uint8_t    *d = nullptr;
        if (cudaMalloc(reinterpret_cast<void **>(&d), host->size()) != cudaSuccess ||
            cudaMemcpy(d, host->data(), host->size(), cudaMemcpyHostToDevice) != cudaSuccess)
        {
            err = std::string("beam table upload: ") + cudaGetErrorString(cudaGetLastError());
            if (d)
                cudaFree(d);
            return nullptr;
        }
        out = std::make_shared<DeviceBlob>(d, host->size(), device);
    }
    std::lock_guard<std::mutex> lock(g_beam_mu);
    size_t                      held = out->bytes;
    for (auto &kv : g_beam_dev_cache)
        held += kv.second->bytes;
    if (held > (size_t{24} << 30)) // envs keep their own references; this only bounds what the cache itself pins
        g_beam_dev_cache.clear();
    g_beam_dev_cache[key] = out;
    return out;
}

ok::BeamConfig beam_config(const OkEnv *e)
{
    ok::BeamConfig c;
    c.cell  = e->cfg.beam_cell;
    c.bins  = e->cfg.beam_bins;
    c.range = 200.0f; // Agent::kSensorRange; a larger OkConfig::sensor_range stays exact through the grid walk
    if (const char *env = std::getenv("OK_BEAM_THREADS"))
        c.threads = std::atoi(env);
    else if (const char *lws = std::getenv("LOCAL_WORLD_SIZE")) // torchrun: the ranks of a box share its cores
        c.threads = std::max(1, static_cast<int>(std::thread::hardware_concurrency()) / std::max(1, std::atoi(lws)));
    return c;
}

int ensure_arena(OkEnv *e)
{
    const bool want_beams = e->cfg.raycast_mode == OK_RAYCAST_BEAM;
    if (!e->arena_dirty && (!want_beams || e->arena_has_beams))
        return OK_SUCCESS;
    e->d_arena.reset(), e->d_track_refs.reset();
    std::vector<ok::TrackRef> refs;
    size_t                    total = 0;
    e->max_blob_used                = 0;
    e->beams_dev.resize(e->tracks.size());
    const bool verbose = std::getenv("OK_BEAM_VERBOSE") != nullptr;
    const auto t_0     = std::chrono::steady_clock::now();
    if (want_beams)
    {
        { // the tables nobody has built yet in this process, all at once: the device builder pipelines them
            const char *force = std::getenv("OK_BEAM_BUILDER");
            std::vector<const ok::Track *> todo;
            std::vector<std::string>       keys;
            if (!(force && std::strcmp(force, "cpu") == 0))
            {
                std::lock_guard<std::mutex> lock(g_beam_mu);
                for (size_t i = 0; i < e->tracks.size(); ++i)
                {
                    const std::string key = beam_key(e->tracks[i], beam_config(e)) + "@" + std::to_string(e->cfg.device);
                    if (!e->beams_dev[i] && !g_beam_dev_cache.count(key) && std::find(keys.begin(), keys.end(), key) == keys.end())
                        todo.push_back(&e->tracks[i]), keys.push_back(key);
                }
            }
            if (todo.size() > 1)
            {
                std::vector<uint8_t *> blobs;
                std::vector<size_t>    sizes;
                ok::build_beam_tables_device(todo, beam_config(e), e->cfg.device, blobs, sizes);
                std::lock_guard<std::mutex> lock(g_beam_mu);
                for (size_t k = 0; k < todo.size(); ++k)
                    if (blobs[k])
                        g_beam_dev_cache[keys[k]] = std::make_shared<DeviceBlob>(blobs[k], sizes[k], e->cfg.device);
            }
        }
        // (host-built tables only) first every table nobody else is building, then the ones other ranks were busy with
        for (int pass = 0; pass < 2; ++pass)
            for (size_t i = 0; i < e->tracks.size(); ++i)
                if (!e->beams_dev[i])
                {
                    std::string err;
                    e->beams_dev[i] = beam_device_table_for(e->tracks[i], beam_config(e), e->cfg.device, pass == 1, err);
                    if (!e->beams_dev[i] && (pass == 1 || !err.empty()))
                        return fail(OK_ERR_INVALID_ARG, "beam table: " + err);
                }
        const auto t_1 = std::chrono::steady_clock::now();
        ok::beam_builder_release(); // the device builder's scratch pool (kept from track to track) is no longer needed
        if (verbose)
            std::fprintf(stderr, "[ensure_arena] tables %.1f ms, pool release %.1f ms\n", std::chrono::duration<double, std::milli>(t_1 - t_0).count(),
                         std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_1).count());
    }
    for (size_t i = 0; i < e->tracks.size(); ++i)
    {
        const ok::Track &t = e->tracks[i];
        ok::TrackRef     r{};
        r.offset = total;
        r.bytes  = static_cast<uint32_t>(t.blob.size());
        if (want_beams)
        {
            r.has_beam    = 1;
            r.beam_offset = reinterpret_cast<uint64_t>(e->beams_dev[i]->ptr); // absolute: the table is its own allocation
            ok::BeamHeader h{};
            OK_CUDA(cudaMemcpy(&h, e->beams_dev[i]->ptr, sizeof h, cudaMemcpyDeviceToHost));
            r.bx0 = h.x0, r.by0 = h.y0, r.binv_h = h.inv_h, r.bbin_scale = h.bin_scale, r.brb = h.rb;
            r.bnx = h.nx, r.bny = h.ny, r.bnb = h.nb;
            r.boff_rows = h.off_rows, r.boff_entries = h.off_entries, r.boff_items = h.off_items;
            r.bn_rows = h.n_rows, r.bn_chunks = h.n_chunks;
        }
        {
            const ok::TrackHeader *th = reinterpret_cast<const ok::TrackHeader *>(t.blob.data());
            r.seg_bytes = th->off_words; // header + segments
            r.n_points = th->n_points, r.off_points = th->off_points, r.off_headings = th->off_headings;
        }
        refs.push_back(r);
        total += (t.blob.size() + 127) / 128 * 128;
        e->max_blob_used = std::max(e->max_blob_used, t.blob.size());
    }
    e->arena_has_beams = want_beams;
    std::vector<uint8_t> host(total, 0);
    for (size_t i = 0; i < e->tracks.size(); ++i)
        std::memcpy(host.data() + refs[i].offset, e->tracks[i].blob.data(), e->tracks[i].blob.size());
    OK_CUDA(dev_alloc(e->d_arena, std::max<size_t>(total, 128)));
    OK_CUDA(dev_alloc(e->d_track_refs, std::max<size_t>(refs.size(), 1)));
    OK_CUDA(cudaMemcpy(e->d_arena.get(), host.data(), total, cudaMemcpyHostToDevice));
    OK_CUDA(cudaMemcpy(e->d_track_refs.get(), refs.data(), sizeof(ok::TrackRef) * refs.size(), cudaMemcpyHostToDevice));
    e->h_track_refs   = refs;
    e->ag.first_dirty = true;
    e->arena_bytes = total;
    e->arena_dirty = false;
    return OK_SUCCESS;
}

ok::StepParams base_params(OkEnv *e)
{
    ok::StepParams p{};
    p.x         = static_cast<float *>(e->d_buf[OK_BUF_POS_X]);
    p.y         = static_cast<float *>(e->d_buf[OK_BUF_POS_Y]);
    p.rot       = static_cast<float *>(e->d_buf[OK_BUF_ROT]);
    p.speed     = static_cast<float *>(e->d_buf[OK_BUF_SPEED]);
    p.accel     = static_cast<float *>(e->d_buf[OK_BUF_ACCEL]);
    p.act_thr   = static_cast<float *>(e->d_buf[OK_BUF_ACT_THROTTLE]);
    p.act_steer = static_cast<float *>(e->d_buf[OK_BUF_ACT_STEER]);
    p.crashed   = static_cast<uint8_t *>(e->d_buf[OK_BUF_CRASHED]);
    p.timed_out = static_cast<uint8_t *>(e->d_buf[OK_BUF_TIMED_OUT]);
    p.done      = static_cast<uint8_t *>(e->d_buf[OK_BUF_DONE]);
    p.ss_ctr    = static_cast<uint32_t *>(e->d_buf[OK_BUF_SS_CTR]);
    p.ss_x      = static_cast<float *>(e->d_buf[OK_BUF_SS_X]);
    p.ss_y      = static_cast<float *>(e->d_buf[OK_BUF_SS_Y]);
    p.track_id  = static_cast<int32_t *>(e->d_buf[OK_BUF_TRACK_ID]);
    p.hit_abs   = static_cast<float *>(e->d_buf[OK_BUF_HIT_ABS]);
    p.hit_rel   = static_cast<float *>(e->d_buf[OK_BUF_HIT_REL]);
    p.obs       = static_cast<float *>(e->d_buf[OK_BUF_OBS]);
    p.hit_t     = static_cast<float *>(e->d_buf[OK_BUF_HIT_T]);
    p.min_dist2 = static_cast<float *>(e->d_buf[OK_BUF_MIN_DIST2]);
    p.hit_seg   = static_cast<int32_t *>(e->d_buf[OK_BUF_HIT_SEG]);
    p.nearest   = static_cast<int32_t *>(e->d_buf[OK_BUF_NEAREST_IDX]);
    p.prev      = static_cast<int32_t *>(e->d_buf[OK_BUF_PREV_IDX]);
    p.reward    = static_cast<float *>(e->d_buf[OK_BUF_REWARD]);
    p.fitness   = static_cast<float *>(e->d_buf[OK_BUF_FITNESS]);
    p.reset_pt  = static_cast<int32_t *>(e->d_buf[OK_BUF_RESET_PT]);
    p.start_x   = static_cast<float *>(e->d_buf[OK_BUF_START_X]);
    p.start_y   = static_cast<float *>(e->d_buf[OK_BUF_START_Y]);
    p.ray_deg   = e->ag.ray_deg.get();
    p.arena     = e->d_arena.get();
    p.tracks    = e->d_track_refs.get();
    p.tiles     = e->ag.tiles.d.get();
    p.n_tiles   = e->ag.tiles.n;
    p.n_agents  = e->n_agents;
    p.rays      = e->rays;
    p.batch_agents      = e->batch_agents;
    p.smem_blob_bytes   = static_cast<uint32_t>((e->max_blob_used + 127) / 128 * 128);
    p.ray_order         = e->ag.ray_order.get();
    p.sched             = e->ag.sched.get();
    p.stats             = e->ag.stats.get();
    p.trace             = e->ag.trace.get();
    p.trace_tiles       = e->ag.trace_tiles;
    p.movement_mode     = e->cfg.movement_mode;
    p.reward_mode       = e->cfg.reward_mode;
    p.raycast_mode      = e->cfg.raycast_mode;
    p.auto_reset        = e->cfg.auto_reset;
    p.auto_reset_stride = e->cfg.auto_reset_stride;
    p.sensor_range      = e->cfg.sensor_range;
    p.speed_limit       = e->cfg.speed_limit;
    p.dt                = e->cfg.dt;
    p.collision_dist2   = e->cfg.collision_dist2;
    p.sensor_offset     = e->cfg.sensor_offset;
    p.standstill_thr2   = e->cfg.standstill_threshold * e->cfg.standstill_threshold; // Environment.cpp:26
    p.standstill_period = e->cfg.standstill_period;
    p.id_base           = e->cfg.agent_id_base;
    return p;
}

int check_ready(OkEnv *e)
{
    if (!e)
        return fail(OK_ERR_INVALID_ARG, "env is NULL");
    if (!e->has_device)
        return fail(OK_ERR_NO_DEVICE, "this env was created without a CUDA device (device = -1): no compute entry point is available");
    if (e->n_agents <= 0)
        return fail(OK_ERR_STATE, "ok_alloc_agents has not been called");
    return OK_SUCCESS;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize of the grid, staged and actor step kernels = everything the device allows.
// Idempotent.
int arm_shared_memory_limit(OkEnv *e)
{
    int max_dynamic = 0;
    OK_CUDA(ok::arm_step_grid(e->smem_optin, &max_dynamic));
    OK_CUDA(ok::arm_step_staged(e->smem_optin, &max_dynamic));
    OK_CUDA(ok::arm_step_actor(e->smem_optin, &e->actor_dyn_max));
    return OK_SUCCESS;
}

// Uploads `tiles` as schedule `s`, in a table of room for `capacity` tiles (at least as many as there are), run by
// `ctas` CTAs at most.
int upload_schedule(Schedule &s, const std::vector<ok::Tile> &tiles, size_t capacity, int ctas)
{
    OK_CUDA(dev_alloc(s.d, std::max(capacity, tiles.size())));
    OK_CUDA(cudaMemcpy(s.d.get(), tiles.data(), sizeof(ok::Tile) * tiles.size(), cudaMemcpyHostToDevice));
    s.n    = static_cast<int32_t>(tiles.size());
    s.grid = std::max(1, std::min(ctas, s.n));
    return OK_SUCCESS;
}

// The CTAs' first tiles with their track records side by side (ok::FirstTile), rebuilt whenever the tiling or the arena
// changes.  Synchronises `s`: a launch in flight may still read the old records.
int upload_first_tiles(OkEnv *e, cudaStream_t s)
{
    Agents       &ag = e->ag;
    const int32_t nf = std::min<int32_t>(ag.beam.grid, static_cast<int32_t>(ag.feedback.tiles.size()));
    if (nf <= 0 || e->h_track_refs.empty())
        return OK_SUCCESS;
    OK_CUDA(cudaStreamSynchronize(s));
    if (nf > ag.first_capacity)
    {
        ag.first_capacity = 0;
        OK_CUDA(dev_alloc(ag.first_beam, static_cast<size_t>(nf)));
        ag.first_capacity = nf;
    }
    std::vector<ok::FirstTile> first(static_cast<size_t>(nf));
    for (int32_t i = 0; i < nf; ++i)
    {
        first[i].tile = ag.feedback.tiles[i];
        first[i].ref  = e->h_track_refs[ag.feedback.tiles[i].track];
        std::memset(first[i].pad, 0, sizeof first[i].pad);
    }
    OK_CUDA(cudaMemcpy(ag.first_beam.get(), first.data(), sizeof(ok::FirstTile) * first.size(), cudaMemcpyHostToDevice));
    ag.first_dirty = false;
    return OK_SUCCESS;
}

// Re-cuts the beam tiling from the per-tile times the last launch on `s` left in d_tile_ns (ok::reweigh_runs), in place.
// Results do not depend on the tiling (tests/test_gpu_properties.py); only the finish times of the SMs do.  Synchronises `s`.
int rebalance_beam_tiles(OkEnv *e, cudaStream_t s)
{
    Agents       &ag = e->ag;
    BeamFeedback &fb = ag.feedback;
    if (!fb.d_tile_ns || fb.tiles.empty() || fb.runs.empty())
        return OK_SUCCESS;
    OK_CUDA(cudaStreamSynchronize(s));
    std::vector<uint32_t> ns(2 * fb.tiles.size());
    OK_CUDA(cudaMemcpy(ns.data(), fb.d_tile_ns.get(), sizeof(uint32_t) * ns.size(), cudaMemcpyDeviceToHost));
    ok::Reweighing rw;
    if (!ok::reweigh_runs(fb.runs, fb.tiles, ns.data(), fb.weighted, fb.target, rw))
        return OK_SUCCESS;
    e->balance_before = rw.balance_before, e->balance_after = rw.balance_after;
    if (rw.tiles.empty() || static_cast<int32_t>(rw.tiles.size()) > fb.capacity)
        return OK_SUCCESS;
    OK_CUDA(cudaMemcpy(ag.beam.d.get(), rw.tiles.data(), sizeof(ok::Tile) * rw.tiles.size(), cudaMemcpyHostToDevice));
    OK_CUDA(cudaMemset(fb.d_tile_ns.get(), 0, sizeof(uint32_t) * 2 * static_cast<size_t>(fb.capacity)));
    fb.tiles       = std::move(rw.tiles);
    ag.first_dirty = true;
    ag.beam.n      = static_cast<int32_t>(fb.tiles.size());
    ag.beam.grid   = std::max(1, std::min(e->num_sms * e->ctas_per_sm_beam, ag.beam.n));
    // at once, not at the next launch: a CUDA graph captured earlier reads both arrays at every replay, and they must agree
    return ag.first_beam ? upload_first_tiles(e, s) : OK_SUCCESS;
}

// cuStreamWriteValue32 through the runtime's driver-entry-point lookup (the library does not link libcuda); nullptr if absent
using StreamWriteValue32Fn = CUresult (*)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
StreamWriteValue32Fn stream_write_value32()
{
    static const StreamWriteValue32Fn fn = [] {
        void                            *f  = nullptr;
        cudaDriverEntryPointQueryResult  qr = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &f, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess)
        {
            cudaGetLastError();
            f = nullptr;
        }
        return reinterpret_cast<StreamWriteValue32Fn>(f);
    }();
    return fn;
}

int launch_step(OkEnv *e, ok::StepParams &p, cudaStream_t s, const ok::ActorParams *actor = nullptr, size_t actor_smem = 0)
{
    NvtxRange range(actor ? "ok::step (actor + tick)" : "ok::step");
    int rc = ensure_arena(e);
    if (rc)
        return rc;
    p.arena      = e->d_arena.get();
    p.tracks     = e->d_track_refs.get();
    Agents &ag   = e->ag;
    if (e->cfg.raycast_mode == OK_RAYCAST_BEAM)
    {
        const bool e2e = (p.host_obs || p.host_obs_q16) && ag.e2e.d;
        if (!e2e && e->auto_balance && ag.feedback.d_tile_ns)
        { // feedback tiling: re-cut the tiles from the measured tile times, a few times early on, then now and then
            const uint64_t k = ag.feedback.launches++;
            if (k == 16 || k == 64 || k == 256 || (k & 4095) == 4095)
            {
                cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
                if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone)
                    if (int rc2 = rebalance_beam_tiles(e, s))
                        return rc2;
            }
        }
        p.tiles        = ag.beam.d.get();
        p.n_tiles      = ag.beam.n;
        p.batch_agents = e->batch_agents_beam;
        p.tile_ns      = e2e ? nullptr : ag.feedback.d_tile_ns.get();
        int grid       = ag.beam.grid;
        p.first        = nullptr;
        if (!e2e && !ag.feedback.tiles.empty())
        { // the CTAs' first tiles with their track records side by side (rebuilt when the tiling or the arena changed)
            if (ag.first_dirty)
            {
                cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
                if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone)
                    if (int rc2 = upload_first_tiles(e, s))
                        return rc2;
            }
            if (!ag.first_dirty)
                p.first = ag.first_beam.get();
        }
        if (e2e)
        { // results stream to a host buffer: several tiles per CTA, each flushed while the next is computed
            const Schedule &sch = p.host_obs_q16 && ag.q16.d ? ag.q16 : ag.e2e;
            p.tiles             = sch.d.get();
            p.n_tiles           = sch.n;
            grid                = sch.grid;
            if (p.ext_host && ag.act_stage && p.n_tiles > grid && e->act_stage_on && stream_write_value32())
            { // tiles after a CTA's first read the actions from a device copy (StepParams::act_ready)
                p.act_stage_thr    = ag.act_stage.get();
                p.act_stage_steer  = ag.act_stage.get() + e->n_agents;
                p.act_ready        = ag.act_ready.get();
                p.act_ready_target = ++ag.act_ready_target;
            }
        }
        const bool flushers = e2e && p.host_obs && e->e2e_flushers > 0 && ag.tile_flag && e->beam_staged;
        if (flushers)
        { // fork: the flusher CTAs start next to the step kernel, on the side stream
            p.tile_flag  = ag.tile_flag.get();
            p.flag_epoch = ++e->flag_epoch;
            OK_CUDA(cudaEventRecord(e->ev_fork.get(), s));
            OK_CUDA(cudaStreamWaitEvent(e->flush_stream.get(), e->ev_fork.get(), 0));
            ok::obs_flush_kernel<<<e->e2e_flushers, 1024, 0, e->flush_stream.get()>>>(ag.e2e.d.get(), ag.e2e.n, ag.tile_flag.get(), p.flag_epoch,
                                                                                      static_cast<const float *>(e->d_buf[OK_BUF_OBS]), p.host_obs, e->rays);
            OK_CUDA(cudaGetLastError());
            OK_CUDA(cudaEventRecord(e->ev_join.get(), e->flush_stream.get()));
        }
        if (actor)
        { // the policy step as phase 0 of every tile (ok_ppo_actor_step): its weights sit behind the kernel's own shared memory
            p.actor_smem_off = static_cast<uint32_t>((e->smem_beam + 15) & ~static_cast<size_t>(15));
            OK_CUDA(ok::launch_step_actor(p, *actor, ag.beam.grid, p.actor_smem_off + actor_smem, s));
        }
        else if (e->beam_staged)
            OK_CUDA(ok::launch_step_staged(p, grid, e->smem_beam, s));
        else
            OK_CUDA(ok::launch_step_unstaged(p, ag.beam.grid, e->smem_beam, s));
    }
    else
        OK_CUDA(ok::launch_step_grid(p, ag.tiles.grid, e->smem, s));
    if (p.act_ready)
    { // enqueued AFTER the launch: the kernel is already running its first tiles while the host issues these
        const size_t bytes = sizeof(float) * static_cast<size_t>(e->n_agents);
        OK_CUDA(cudaMemcpyAsync(p.act_stage_thr, p.ext_thr, bytes, cudaMemcpyHostToDevice, e->act_stream.get()));
        OK_CUDA(cudaMemcpyAsync(p.act_stage_steer, p.ext_steer, bytes, cudaMemcpyHostToDevice, e->act_stream.get()));
        if (stream_write_value32()(e->act_stream.get(), reinterpret_cast<CUdeviceptr>(ag.act_ready.get()), p.act_ready_target, 0) != CUDA_SUCCESS)
            return fail(OK_ERR_CUDA, "cuStreamWriteValue32 failed");
        OK_CUDA(cudaEventRecord(e->ev_act.get(), e->act_stream.get()));
        OK_CUDA(cudaStreamWaitEvent(s, e->ev_act.get(), 0)); // join: nothing of this tick outlives the caller's stream
    }
    if (p.tile_flag) // join: the tick is complete when the last tile has reached the host
        OK_CUDA(cudaStreamWaitEvent(s, e->ev_join.get(), 0));
    e->launches++;
    return OK_SUCCESS;
}
} // namespace

namespace
{
int alloc_agents_impl(OkEnv *e, int64_t n, int32_t rays, const float *h_ray_deg, const int32_t *h_track_id);
// device-visible alias of a pinned (cudaMallocHost / cudaHostRegister) host pointer, or nullptr if pageable
template <typename T> T *pinned_alias(T *h)
{
    if (!h)
        return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, h) != cudaSuccess)
    {
        cudaGetLastError();
        return nullptr;
    }
    return at.type == cudaMemoryTypeHost ? static_cast<T *>(at.devicePointer) : nullptr;
}
} // namespace

extern "C"
{
int ok_abi_version(void)
{
    return OK_ABI_VERSION;
}

const char *ok_last_error(void)
{
    return g_last_error.c_str();
}

void ok_config_default(OkConfig *c)
{
    if (!c)
        return;
    std::memset(c, 0, sizeof *c);
    c->device               = 0;
    c->movement_mode        = OK_MOVE_VELOCITY;
    c->reward_mode          = OK_REWARD_NONE;
    c->raycast_mode         = OK_RAYCAST_BEAM;
    c->auto_reset           = 0;
    c->auto_reset_stride    = 97;
    c->sensor_range         = 200.0f;
    c->speed_limit          = 100.0f;
    c->dt                   = static_cast<float>(0.016);
    c->collision_dist2      = 2.0f;
    c->sensor_offset        = 0.0f;
    c->standstill_period    = 200u;
    c->standstill_threshold = 20.0f;
    c->grid_cell            = 8.0f;
    c->beam_cell            = 2.0f;
    c->beam_bins            = 256;
}

int ok_create(const OkConfig *cfg, OkEnv **out)
{
    if (!out)
        return fail(OK_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    OkConfig c;
    if (cfg)
        c = *cfg;
    else
        ok_config_default(&c);
    if (c.movement_mode != OK_MOVE_VELOCITY && c.movement_mode != OK_MOVE_ACCELERATION)
        return fail(OK_ERR_INVALID_ARG, "movement_mode must be VELOCITY or ACCELERATION");
    if (c.reward_mode < OK_REWARD_NONE || c.reward_mode > OK_REWARD_LANE_CENTER)
        return fail(OK_ERR_INVALID_ARG, "unknown reward_mode");
    if (c.raycast_mode < OK_RAYCAST_GRID || c.raycast_mode > OK_RAYCAST_BEAM)
        return fail(OK_ERR_INVALID_ARG, "unknown raycast_mode");
    if (!(c.grid_cell >= 1.0f && c.grid_cell <= 512.0f))
        return fail(OK_ERR_INVALID_ARG, "grid_cell must be in [1, 512] px");
    if (c.beam_cell == 0.0f)
        c.beam_cell = 2.0f;
    if (c.beam_bins == 0)
        c.beam_bins = 256;
    if (!(c.beam_cell >= 1.0f && c.beam_cell <= 64.0f) || c.beam_bins < 8 || c.beam_bins > 1024 ||
        (c.beam_bins & (c.beam_bins - 1)))
        return fail(OK_ERR_INVALID_ARG, "beam_cell must be in [1, 64] px and beam_bins a power of two in [8, 1024]");
    auto e = new OkEnv();
    e->cfg = c;
    if (c.device >= 0)
    {
        int         count = 0;
        cudaError_t err   = cudaGetDeviceCount(&count);
        if (err != cudaSuccess || count <= 0 || c.device >= count)
        {
            delete e;
            return fail(OK_ERR_NO_DEVICE, std::string("no usable CUDA device ") + std::to_string(c.device) + " (" +
                                              (err != cudaSuccess ? cudaGetErrorString(err) : "device count 0") +
                                              "); there is no CPU fallback");
        }
        DeviceGuard g(c.device);
        int         sms = 0, optin = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c.device);
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, c.device);
        e->has_device = true;
        e->num_sms    = sms;
        e->smem_optin = optin;
        e->max_blob   = optin > 65536 ? static_cast<size_t>(optin) - 40960 : 0; // room for the batch scratch
    }
    else
    {
        e->max_blob = 227 * 1024 - 40960; // host-only env: tracks can be built and inspected, nothing else
    }
    *out = e;
    return OK_SUCCESS;
}

int ok_update_config(OkEnv *e, const OkConfig *cfg)
{
    if (!e || !cfg)
        return fail(OK_ERR_INVALID_ARG, "NULL argument");
    if (cfg->movement_mode != OK_MOVE_VELOCITY && cfg->movement_mode != OK_MOVE_ACCELERATION)
        return fail(OK_ERR_INVALID_ARG, "movement_mode must be VELOCITY or ACCELERATION");
    if (cfg->reward_mode < OK_REWARD_NONE || cfg->reward_mode > OK_REWARD_LANE_CENTER)
        return fail(OK_ERR_INVALID_ARG, "unknown reward_mode");
    if (cfg->raycast_mode < OK_RAYCAST_GRID || cfg->raycast_mode > OK_RAYCAST_BEAM)
        return fail(OK_ERR_INVALID_ARG, "unknown raycast_mode");
    OkConfig c   = *cfg;
    c.device     = e->cfg.device;
    c.grid_cell  = e->cfg.grid_cell;
    c.beam_cell  = e->cfg.beam_cell;
    c.beam_bins  = e->cfg.beam_bins;
    e->cfg       = c;
    return OK_SUCCESS;
}

int ok_get_config(const OkEnv *e, OkConfig *out)
{
    if (!e || !out)
        return fail(OK_ERR_INVALID_ARG, "NULL argument");
    *out = e->cfg;
    return OK_SUCCESS;
}

void ok_destroy(OkEnv *e)
{
    if (!e)
        return;
    DeviceGuard g(e->has_device ? e->cfg.device : -1); // the env's members free their device resources on that device
    delete e;
}

int ok_add_track(OkEnv *e, const float *x, const float *y, const float *wr, const float *wl, int32_t n, int32_t *id_out)
{
    if (!e)
        return fail(OK_ERR_INVALID_ARG, "env is NULL");
    if (e->n_agents > 0)
        return fail(OK_ERR_STATE, "add every track before ok_alloc_agents (the batch size depends on the largest track)");
    ok::Track   t;
    std::string err;
    if (!ok::build_track(x, y, wr, wl, n, e->cfg.grid_cell, e->max_blob, t, err))
        return fail(err.find("fit") != std::string::npos ? OK_ERR_CAPACITY : OK_ERR_INVALID_ARG, err);
    e->tracks.push_back(std::move(t));
    e->arena_dirty = true;
    if (id_out)
        *id_out = static_cast<int32_t>(e->tracks.size()) - 1;
    return OK_SUCCESS;
}

int ok_load_track_csv(OkEnv *e, const char *path, int32_t *id_out)
{
    if (!e || !path)
        return fail(OK_ERR_INVALID_ARG, "env or path is NULL");
    std::vector<float> cols[4];
    std::string        err;
    if (!ok::read_track_csv(path, cols, err))
        return fail(OK_ERR_IO, err);
    return ok_add_track(e, cols[0].data(), cols[1].data(), cols[2].data(), cols[3].data(),
                        static_cast<int32_t>(cols[0].size()), id_out);
}

int ok_num_tracks(const OkEnv *e)
{
    return e ? static_cast<int>(e->tracks.size()) : 0;
}

int ok_track_info(const OkEnv *e, int32_t id, OkTrackInfo *out)
{
    if (!e || !out || id < 0 || id >= static_cast<int32_t>(e->tracks.size()))
        return fail(OK_ERR_INVALID_ARG, "bad track id");
    const ok::Track &t = e->tracks[id];
    out->n_points      = t.n_points();
    out->n_segments    = t.n_segments();
    out->grid_nx       = t.grid_nx;
    out->grid_ny       = t.grid_ny;
    out->grid_items    = static_cast<int32_t>(t.items.size());
    out->blob_bytes    = static_cast<int32_t>(t.blob.size());
    out->grid_x0       = t.grid_x0;
    out->grid_y0       = t.grid_y0;
    out->grid_cell     = t.cell;
    return OK_SUCCESS;
}

int64_t ok_track_copy(const OkEnv *e, int32_t id, int32_t which, float *h_out, int64_t count)
{
    if (!e || id < 0 || id >= static_cast<int32_t>(e->tracks.size()))
        return fail(OK_ERR_INVALID_ARG, "bad track id");
    const ok::Track          &t = e->tracks[id];
    const std::vector<float> *v = nullptr;
    switch (which)
    {
    case OK_TRACK_X: v = &t.x; break;
    case OK_TRACK_Y: v = &t.y; break;
    case OK_TRACK_W_RIGHT: v = &t.w_right; break;
    case OK_TRACK_W_LEFT: v = &t.w_left; break;
    case OK_TRACK_HEADING: v = &t.heading; break;
    case OK_TRACK_LEFT_INNER: v = &t.left_inner; break;
    case OK_TRACK_LEFT_OUTER: v = &t.left_outer; break;
    case OK_TRACK_RIGHT_INNER: v = &t.right_inner; break;
    case OK_TRACK_RIGHT_OUTER: v = &t.right_outer; break;
    case OK_TRACK_SEGMENTS: v = &t.segments; break;
    default: return fail(OK_ERR_INVALID_ARG, "unknown track array");
    }
    if (h_out && count > 0)
        std::memcpy(h_out, v->data(), sizeof(float) * static_cast<size_t>(std::min<int64_t>(count, v->size())));
    return static_cast<int64_t>(v->size());
}

int ok_alloc_agents(OkEnv *e, int64_t n, int32_t rays, const float *h_ray_deg, const int32_t *h_track_id)
{
    if (!e)
        return fail(OK_ERR_INVALID_ARG, "env is NULL");
    if (!e->has_device)
        return fail(OK_ERR_NO_DEVICE, "this env was created without a CUDA device (device = -1)");
    if (n <= 0 || rays <= 0 || !h_ray_deg)
        return fail(OK_ERR_INVALID_ARG, "n_agents and rays must be positive and ray angles given");
    if (rays > 1024)
        return fail(OK_ERR_INVALID_ARG, "at most 1024 rays per agent");
    if (e->tracks.empty())
        return fail(OK_ERR_STATE, "add at least one track before allocating agents");
    for (int64_t i = 0; h_track_id && i < n; ++i)
        if (h_track_id[i] < 0 || h_track_id[i] >= static_cast<int32_t>(e->tracks.size()))
            return fail(OK_ERR_INVALID_ARG, "track id out of range for agent " + std::to_string(i));
    DeviceGuard g(e->cfg.device);
    const bool  verbose = std::getenv("OK_BEAM_VERBOSE") != nullptr;
    const auto  t_0     = std::chrono::steady_clock::now();
    // everything that can fail without touching the current agents comes first
    int rc0 = ensure_arena(e);
    if (rc0)
        return rc0;
    const auto t_1 = std::chrono::steady_clock::now();
    free_agents(e);
    const int rc1 = alloc_agents_impl(e, n, rays, h_ray_deg, h_track_id);
    if (verbose)
    {
        cudaDeviceSynchronize();
        const auto t_2 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[ok_alloc_agents] tables + arena %.1f ms, agents + tiles + reset %.1f ms\n",
                     std::chrono::duration<double, std::milli>(t_1 - t_0).count(), std::chrono::duration<double, std::milli>(t_2 - t_1).count());
    }
    if (rc1)
    { // never leave a half-built set behind: n_agents = 0 makes every entry point report OK_ERR_STATE
        const std::string msg = g_last_error;
        free_agents(e);
        cudaGetLastError();
        g_last_error = msg;
    }
    return rc1;
}
} // extern "C"

namespace
{
int alloc_agents_impl(OkEnv *e, int64_t n, int32_t rays, const float *h_ray_deg, const int32_t *h_track_id)
{
    NvtxRange range("ok_alloc_agents (tiling, buffers)");
    Agents   &ag = e->ag;
    e->n_agents  = n;
    e->rays      = rays;
    // batch = the agents a CTA keeps in flight: as many as fit behind the largest staged track
    {
        const size_t blob  = (e->max_blob_used + 127) / 128 * 128;
        const size_t avail = static_cast<size_t>(e->smem_optin) > blob + 4096 ? e->smem_optin - blob - 4096 : 0;
        const size_t per   = ok::batch_smem_bytes(1, rays);
        int64_t      a     = static_cast<int64_t>(avail / per);
        if (avail < static_cast<size_t>(ok::beam_static_smem(true)) + 4096)
            a = 0; // the beam kernel keeps per-thread scratch and its ray queue in static shared memory
        int          cap   = kMaxBatchAgents;
        if (const char *env = std::getenv("OK_BATCH_AGENTS"))
            cap = std::max(1, std::atoi(env));
        a = std::min<int64_t>(a, cap);
        // small populations: spread over all SMs rather than filling a few batches
        a = std::min<int64_t>(a, std::max<int64_t>(1, (n + e->num_sms - 1) / std::max(1, e->num_sms)));
        if (a < 1)
            return fail(OK_ERR_CAPACITY, "shared memory cannot hold one agent's rays next to the largest track");
        e->batch_agents = static_cast<int32_t>(a);
        e->smem         = blob + ok::batch_smem_bytes(e->batch_agents, rays);
        // beam kernel: one 64-byte record per agent; phases 1 / 4 run a thread per agent, so at most one block of agents.
        // Which shape (ok_step.cuh): the staged one for throughput, the unstaged one when the population is too small
        // to give every SM a worthwhile tile (OK_BEAM_KERNEL = staged | unstaged overrides).
        // measured (tools/bench_small.py, tools/bench_c4.py): the unstaged shape is ahead below ~2,000 agents of 32 rays, and at
        // 4,096 agents of 5 rays (a PPO rollout tick: 0.0289 vs 0.0300 ms, 0.0262 with the policy step fused in), behind at
        // 8,192 agents of 5 rays (0.0376 vs 0.0318 ms)
        e->beam_staged = n >= 2048 && n * rays > 24576;
        if (const char *env = std::getenv("OK_BEAM_KERNEL"))
            e->beam_staged = std::strcmp(env, "unstaged") != 0 && (std::strcmp(env, "staged") == 0 || e->beam_staged);
        e->beam_block = ok::beam_block(e->beam_staged);
        int64_t ab;
        int     capb;
        if (e->beam_staged)
        { // one 1,024-thread CTA per SM behind the staged track: as many agents per tile as the shared memory behind the
          // largest track holds (the balanced tiling then sizes the tiles: about one per CTA and wave)
            ab   = static_cast<int64_t>((avail - ok::beam_static_smem(true)) / sizeof(ok::AgentRec));
            capb = e->beam_block;
        }
        else
        { // several small CTAs per SM, nothing staged: small tiles, the SM's other CTAs hide a tile's serial phases
            ab   = e->beam_block;
            capb = OK_BEAM_TILE;
        }
        ab = std::min<int64_t>(ab, 65535 / rays); // tile-local ray indices are 16 bits (the kernel's ray queue)
        if (const char *env = std::getenv("OK_BEAM_BATCH_AGENTS"))
            capb = std::max(1, std::atoi(env));
        ab = std::min<int64_t>({ab, capb, e->beam_block});
        if (!e->beam_staged) // small populations: spread over all SMs rather than filling a few tiles
            ab = std::min<int64_t>(ab, std::max<int64_t>(1, (n + e->num_sms - 1) / std::max(1, e->num_sms)));
        e->batch_agents_beam = static_cast<int32_t>(std::max<int64_t>(1, ab));
        e->smem_beam         = (e->beam_staged ? blob : 0) + ok::beam_smem_bytes(e->batch_agents_beam);
        // The limit is an attribute of the FUNCTION on this device, not of the env: it is raised to the opt-in maximum
        // (minus the kernel's static shared memory), so that envs of different sizes can interleave their launches.
        if (int rc = arm_shared_memory_limit(e))
            return rc;
    }

    // one slab, 256-byte aligned sub-buffers
    size_t offs[OK_BUF_COUNT], total = 0;
    for (int b = 0; b < OK_BUF_COUNT; ++b)
    {
        offs[b] = total;
        total += (buffer_bytes(e, b) + 255) / 256 * 256;
    }
    OK_CUDA(dev_alloc(ag.slab, total));
    OK_CUDA(cudaMemset(ag.slab.get(), 0, total));
    for (int b = 0; b < OK_BUF_COUNT; ++b)
    {
        e->d_buf[b]   = ag.slab.get() + offs[b];
        e->buf_off[b] = offs[b];
    }
    OK_CUDA(dev_alloc(ag.ray_deg, static_cast<size_t>(rays)));
    OK_CUDA(cudaMemcpy(ag.ray_deg.get(), h_ray_deg, sizeof(float) * rays, cudaMemcpyHostToDevice));
    e->h_track_id.assign(static_cast<size_t>(n), 0);
    if (h_track_id)
        std::copy(h_track_id, h_track_id + n, e->h_track_id.begin());
    OK_CUDA(cudaMemcpy(e->d_buf[OK_BUF_TRACK_ID], e->h_track_id.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice));
    OK_CUDA(cudaMemset(e->d_buf[OK_BUF_HIT_SEG], 0xff, buffer_bytes(e, OK_BUF_HIT_SEG))); // -1 = no hit yet

    // pool order of the rays: by |angle|, the fan's centre (long) rays first
    {
        std::vector<uint16_t> order(rays);
        for (int i = 0; i < rays; ++i)
            order[i] = static_cast<uint16_t>(i);
        std::stable_sort(order.begin(), order.end(),
                         [&](uint16_t x, uint16_t y) { return std::fabs(h_ray_deg[x]) < std::fabs(h_ray_deg[y]); });
        OK_CUDA(dev_alloc(ag.ray_order, static_cast<size_t>(rays)));
        OK_CUDA(cudaMemcpy(ag.ray_order.get(), order.data(), sizeof(uint16_t) * rays, cudaMemcpyHostToDevice));
        OK_CUDA(dev_alloc(ag.sched, 512));
        OK_CUDA(cudaMemset(ag.sched.get(), 0, sizeof(int32_t) * 512));
    }

    // tilings (ok_schedule.hpp)
    const int32_t *track_id = e->h_track_id.data();
    // the balanced tiling of the beam kernel's batches over `ctas` CTAs, at least `waves` tiles per CTA; `runs` keeps the
    // track runs with their tile counts
    auto balanced = [&](int ctas, int waves, std::vector<ok::TileRun> &runs) {
        runs = ok::track_runs(track_id, n, e->batch_agents_beam);
        return ok::balanced_tiles(runs, e->batch_agents_beam, ctas, waves);
    };
    {
        int per_sm = 1;
        if (!e->beam_staged)
            OK_CUDA(ok::occupancy_step_unstaged(e->smem_beam, &per_sm));
        e->ctas_per_sm_beam = std::max(1, per_sm);
    }
    if (int rc = upload_schedule(ag.tiles, ok::guided_tiles(track_id, n, e->batch_agents, e->num_sms, 4), 0, e->num_sms))
        return rc;
    {
        const int beam_ctas = e->num_sms * e->ctas_per_sm_beam;
        // the unstaged beam kernel's small tiles cost about the same serial latency whatever their size (the thread-per-
        // agent phases, the second ray pass): shrinking them further only adds tiles
        int tail_div = e->beam_staged ? -1 : 0; // -1: balanced tiling
        if (const char *env = std::getenv("OK_BEAM_TAIL"))
            tail_div = std::atoi(env);
        int waves = 1; // balanced tiling: tiles per CTA (OK_BEAM_WAVES)
        if (const char *env = std::getenv("OK_BEAM_WAVES"))
            waves = std::max(1, std::atoi(env));
        e->auto_balance = 1; // OK_AUTO_BALANCE=0: keep the tiling by agent count
        if (const char *env = std::getenv("OK_AUTO_BALANCE"))
            e->auto_balance = std::atoi(env);
        if (tail_div < 0)
        { // the feedback tiling: its table is allocated once, with room for every re-cut (rebalance_beam_tiles)
            BeamFeedback      &fb = ag.feedback;
            ok::BalancedTiling bt = balanced(beam_ctas, waves, fb.runs);
            const size_t capacity = std::max<size_t>(bt.tiles.size(), static_cast<size_t>(bt.target));
            fb.tiles    = bt.tiles;
            fb.target   = static_cast<int32_t>(bt.target);
            fb.capacity = static_cast<int32_t>(capacity);
            if (int rc = upload_schedule(ag.beam, bt.tiles, capacity, beam_ctas))
                return rc;
            OK_CUDA(dev_alloc(fb.d_tile_ns, 2 * capacity));
            OK_CUDA(cudaMemset(fb.d_tile_ns.get(), 0, sizeof(uint32_t) * 2 * capacity));
        }
        else if (int rc = upload_schedule(ag.beam, ok::guided_tiles(track_id, n, e->batch_agents_beam, beam_ctas, tail_div), 0, beam_ctas))
            return rc;
    }
    if (e->beam_staged)
    { // the end-to-end tiling (see ok_step_host): OK_E2E_TILES tiles per CTA (default 4)
        int per_cta = 4;
        if (const char *env = std::getenv("OK_E2E_TILES"))
            per_cta = std::max(1, std::atoi(env));
        // OK_E2E_FLUSHERS = F > 0: F SMs are left to obs_flush_kernel, which moves finished tiles to the host while the
        // step kernel's CTAs carry on
        e->e2e_flushers = 0;
        if (const char *env = std::getenv("OK_E2E_FLUSHERS"))
            e->e2e_flushers = std::max(0, std::min(std::atoi(env), e->num_sms / 2));
        std::vector<ok::TileRun> runs;
        const int                e2e_ctas = (e->num_sms - e->e2e_flushers) * e->ctas_per_sm_beam;
        const ok::BalancedTiling e2e      = balanced(e2e_ctas, per_cta, runs);
        if (int rc = upload_schedule(ag.e2e, e2e.tiles, static_cast<size_t>(e2e.target), e2e_ctas))
            return rc;
        { // ok_step_host_q16: measured at the C3 shape 0.164 / 0.157 / 0.171 / 0.199 ms per tick with 2 / 3 / 4 / 6 tiles per CTA
            int per_cta_q16 = 3;
            if (const char *env = std::getenv("OK_E2E_TILES_Q16"))
                per_cta_q16 = std::max(1, std::atoi(env));
            else if (std::getenv("OK_E2E_TILES"))
                per_cta_q16 = per_cta;
            const int                q16_ctas = e->num_sms * e->ctas_per_sm_beam;
            const ok::BalancedTiling q16      = balanced(q16_ctas, per_cta_q16, runs);
            if (int rc = upload_schedule(ag.q16, q16.tiles, static_cast<size_t>(q16.target), q16_ctas))
                return rc;
        }
        OK_CUDA(dev_alloc(ag.act_stage, 2 * static_cast<size_t>(n)));
        OK_CUDA(dev_alloc(ag.act_ready, 1));
        OK_CUDA(cudaMemset(ag.act_ready.get(), 0, sizeof(uint32_t)));
        if (!e->act_stream)
        {
            OK_CUDA(make_stream(e->act_stream));
            OK_CUDA(make_event(e->ev_act));
        }
        if (const char *env = std::getenv("OK_ACT_STAGE"))
            e->act_stage_on = std::atoi(env) != 0;
        if (e->e2e_flushers > 0)
        {
            OK_CUDA(dev_alloc(ag.tile_flag, static_cast<size_t>(ag.e2e.n)));
            OK_CUDA(cudaMemset(ag.tile_flag.get(), 0, sizeof(uint32_t) * static_cast<size_t>(ag.e2e.n)));
            if (!e->flush_stream)
            {
                OK_CUDA(make_stream(e->flush_stream));
                OK_CUDA(make_event(e->ev_fork));
                OK_CUDA(make_event(e->ev_join));
            }
        }
    }

    // every agent starts where `Environment::resetAgent(agent, false)` puts it: RaceTrack::kStartingIdx
    std::vector<int32_t> pt(static_cast<size_t>(n));
    for (int64_t i = 0; i < n; ++i)
        pt[i] = e->tracks[e->h_track_id[i]].n_points() > 3 ? 3 : 0;
    return ok_reset_agents_host(e, nullptr, pt.data(), nullptr, nullptr, n, nullptr);
}
} // namespace

extern "C"
{
int64_t ok_num_agents(const OkEnv *e)
{
    return e ? e->n_agents : 0;
}

int32_t ok_num_rays(const OkEnv *e)
{
    return e ? e->rays : 0;
}

int ok_reset_agents(OkEnv *e, const int64_t *d_agent_idx, const int32_t *d_pt_idx, const float *d_lane_alpha,
                    const float *d_heading_off, int64_t n, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (n <= 0)
        return OK_SUCCESS;
    if (!d_pt_idx)
        return fail(OK_ERR_INVALID_ARG, "pt_idx is NULL");
    DeviceGuard g(e->cfg.device);
    rc = ensure_arena(e);
    if (rc)
        return rc;
    ok::StepParams  p = base_params(e);
    ok::ResetParams r{d_agent_idx, d_pt_idx, d_lane_alpha, d_heading_off, n, e->n_agents};
    const int       threads = 128;
    const int       blocks  = static_cast<int>((n + threads - 1) / threads);
    ok::reset_kernel<<<blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(p, r);
    OK_CUDA(cudaGetLastError());
    e->launches++;
    return OK_SUCCESS;
}

int ok_reset_agents_host(OkEnv *e, const int64_t *h_agent_idx, const int32_t *h_pt_idx, const float *h_lane_alpha,
                         const float *h_heading_off, int64_t n, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (n <= 0)
        return OK_SUCCESS;
    if (!h_pt_idx)
        return fail(OK_ERR_INVALID_ARG, "pt_idx is NULL");
    DeviceGuard  g(e->cfg.device);
    cudaStream_t s    = static_cast<cudaStream_t>(stream);
    const size_t need = static_cast<size_t>(n) * (8 + 4 + 4 + 4) + 64;
    if (need > e->stage_bytes)
    {
        e->stage_bytes = 0;
        OK_CUDA(dev_alloc(e->d_stage, need));
        e->stage_bytes = need;
    }
    int64_t *d_ai = reinterpret_cast<int64_t *>(e->d_stage.get());
    int32_t *d_pt = reinterpret_cast<int32_t *>(e->d_stage.get() + 8 * static_cast<size_t>(n));
    float   *d_la = reinterpret_cast<float *>(e->d_stage.get() + 12 * static_cast<size_t>(n));
    float   *d_ho = reinterpret_cast<float *>(e->d_stage.get() + 16 * static_cast<size_t>(n));
    if (h_agent_idx)
        OK_CUDA(cudaMemcpyAsync(d_ai, h_agent_idx, 8 * static_cast<size_t>(n), cudaMemcpyHostToDevice, s));
    OK_CUDA(cudaMemcpyAsync(d_pt, h_pt_idx, 4 * static_cast<size_t>(n), cudaMemcpyHostToDevice, s));
    if (h_lane_alpha)
        OK_CUDA(cudaMemcpyAsync(d_la, h_lane_alpha, 4 * static_cast<size_t>(n), cudaMemcpyHostToDevice, s));
    if (h_heading_off)
        OK_CUDA(cudaMemcpyAsync(d_ho, h_heading_off, 4 * static_cast<size_t>(n), cudaMemcpyHostToDevice, s));
    rc = ok_reset_agents(e, h_agent_idx ? d_ai : nullptr, d_pt, h_lane_alpha ? d_la : nullptr,
                         h_heading_off ? d_ho : nullptr, n, stream);
    if (rc)
        return rc;
    OK_CUDA(cudaStreamSynchronize(s));
    return OK_SUCCESS;
}

int ok_cast_rays(OkEnv *e, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    DeviceGuard    g(e->cfg.device);
    ok::StepParams p = base_params(e);
    p.do_move        = 0;
    return launch_step(e, p, static_cast<cudaStream_t>(stream));
}

int ok_launch_step(OkEnv *e, const float *d_thr, const float *d_steer, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if ((d_thr == nullptr) != (d_steer == nullptr))
        return fail(OK_ERR_INVALID_ARG, "pass both action arrays or neither");
    DeviceGuard    g(e->cfg.device);
    ok::StepParams p = base_params(e);
    p.do_move        = 1;
    p.ext_thr        = d_thr;
    p.ext_steer      = d_steer;
    return launch_step(e, p, static_cast<cudaStream_t>(stream));
}

int ok_launch_steps_random(OkEnv *e, uint64_t first_step, int32_t k, uint32_t seed, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    DeviceGuard    g(e->cfg.device);
    ok::StepParams p = base_params(e);
    p.do_move        = 1;
    p.action_source  = 1;
    p.seed           = seed;
    for (int32_t i = 0; i < k; ++i)
    {
        p.step = first_step + static_cast<uint64_t>(i);
        rc     = launch_step(e, p, static_cast<cudaStream_t>(stream));
        if (rc)
            return rc;
    }
    return OK_SUCCESS;
}

int ok_fill_random_actions(OkEnv *e, uint64_t step, uint32_t seed, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    DeviceGuard    g(e->cfg.device);
    ok::StepParams p = base_params(e);
    p.step           = step;
    p.seed           = seed;
    const int threads = 256;
    const int blocks  = static_cast<int>((e->n_agents + threads - 1) / threads);
    ok::fill_actions_kernel<<<blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(p, e->n_agents);
    OK_CUDA(cudaGetLastError());
    e->launches++;
    return OK_SUCCESS;
}

int ok_genetic_policy(OkEnv *e, const float *d_w1, const float *d_w2, int32_t hidden, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (!d_w1 || !d_w2 || hidden < 1 || hidden > 32)
        return fail(OK_ERR_INVALID_ARG, "weights must be given and 1 <= hidden <= 32");
    DeviceGuard    g(e->cfg.device);
    ok::StepParams p = base_params(e);
    const int      threads = 256;
    const int64_t  blocks  = (e->n_agents * 32 + threads - 1) / threads;
    ok::genetic_policy_kernel<<<static_cast<unsigned>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(
        p, d_w1, d_w2, hidden, e->n_agents);
    OK_CUDA(cudaGetLastError());
    e->launches++;
    return OK_SUCCESS;
}

int ok_cmaes_controller(OkEnv *e, const float *d_params, int32_t n_params, int32_t hidden, float throttle, float steer_scale,
                        void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (!d_params || hidden != 16)
        return fail(OK_ERR_INVALID_ARG, "parameters must be given and hidden must be 16 (CmaEsAgent::kHiddenSize)");
    if (n_params != 16 * e->rays + 16 + 8 * 16 + 8 + 8 + 1)
        return fail(OK_ERR_INVALID_ARG, "n_params must be 16 * rays + 169 (Controller::count_params)");
    DeviceGuard    g(e->cfg.device);
    ok::StepParams p = base_params(e);
    const int      threads = 256;
    const int64_t  blocks  = (e->n_agents * 32 + threads - 1) / threads;
    ok::cmaes_controller_kernel<<<static_cast<unsigned>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(
        p, d_params, n_params, throttle, steer_scale, e->n_agents);
    OK_CUDA(cudaGetLastError());
    e->launches++;
    return OK_SUCCESS;
}

} // extern "C"
namespace
{
// OkActorIO -> kernel parameters; *skip = nothing to do (no weights and nothing to record)
int actor_params(const OkActorIO *io, ok::ActorParams &q, bool *skip)
{
    *skip = false;
    if (!io)
        return fail(OK_ERR_INVALID_ARG, "io is NULL");
    q     = ok::ActorParams{};
    q.act = io->d_w1 != nullptr;
    if (q.act)
    {
        if (!io->d_b1 || !io->d_w2 || !io->d_b2 || !io->d_action_table)
            return fail(OK_ERR_INVALID_ARG, "weights, biases and the action table must all be given");
        if (io->hidden < 1 || io->hidden > 1024 || io->n_actions < 1 || io->n_actions > ok::kActorMaxActs)
            return fail(OK_ERR_INVALID_ARG, "1 <= hidden <= 1024 and 1 <= n_actions <= 8");
    }
    else if (!io->d_prev_reward && !io->d_prev_done)
        *skip = true;
    q.w1 = io->d_w1, q.b1 = io->d_b1, q.w2 = io->d_w2, q.b2 = io->d_b2;
    q.hidden = io->hidden, q.n_actions = io->n_actions;
    q.table = io->d_action_table, q.uniform = io->d_uniform, q.greedy = io->greedy;
    q.action_out = io->d_action, q.log_prob_out = io->d_log_prob, q.probs_out = io->d_probs, q.obs_out = io->d_obs;
    q.prev_reward_out = io->d_prev_reward, q.prev_done_out = io->d_prev_done;
    return OK_SUCCESS;
}

size_t actor_weight_bytes(const ok::ActorParams &q, int rays)
{
    // w1 | b1 | w2 | b2 | action table
    return q.act ? sizeof(float) * (static_cast<size_t>(q.hidden) * rays + q.hidden + static_cast<size_t>(q.n_actions) * q.hidden + 3 * static_cast<size_t>(q.n_actions)) : 0;
}
} // namespace
extern "C"
{
int ok_ppo_actor(OkEnv *e, const OkActorIO *io, uint64_t step, uint32_t seed, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    ok::ActorParams q;
    bool            skip = false;
    rc                   = actor_params(io, q, &skip);
    if (rc || skip)
        return rc;
    DeviceGuard    g(e->cfg.device);
    ok::StepParams p = base_params(e);
    p.step           = step;
    p.seed           = seed;
    const size_t smem = actor_weight_bytes(q, e->rays);
    if (smem > static_cast<size_t>(e->smem_optin))
        return fail(OK_ERR_CAPACITY, "the actor's weights do not fit in shared memory");
    if (smem > 48 * 1024)
        OK_CUDA(cudaFuncSetAttribute(ok::ppo_actor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    const int     threads = 256;
    const int64_t blocks  = (e->n_agents * ok::kActorLanes + threads - 1) / threads;
    ok::ppo_actor_kernel<<<static_cast<unsigned>(blocks), threads, smem, static_cast<cudaStream_t>(stream)>>>(p, q, e->n_agents);
    OK_CUDA(cudaGetLastError());
    e->launches++;
    return OK_SUCCESS;
}

int ok_ppo_actor_step(OkEnv *e, const OkActorIO *io, uint64_t step, uint32_t seed, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    ok::ActorParams q;
    bool            skip = false;
    rc                   = actor_params(io, q, &skip);
    if (rc)
        return rc;
    DeviceGuard  g(e->cfg.device);
    const size_t wbytes = actor_weight_bytes(q, e->rays) + sizeof(float) * 2 * static_cast<size_t>(e->batch_agents_beam); // + the tile's chosen actions
    // one launch when the env runs the unstaged beam kernel (the shape of small populations, where a tick is latency) and the
    // weights fit behind its shared memory; otherwise the same tick as two launches
    const bool fused = q.act && e->cfg.raycast_mode == OK_RAYCAST_BEAM && !e->beam_staged &&
                       ((e->smem_beam + 15) & ~static_cast<size_t>(15)) + wbytes <= static_cast<size_t>(std::max(0, e->actor_dyn_max));
    if (!fused)
    {
        if (!skip)
            if ((rc = ok_ppo_actor(e, io, step, seed, stream)) != OK_SUCCESS)
                return rc;
        return ok_launch_step(e, nullptr, nullptr, stream);
    }
    ok::StepParams p = base_params(e);
    p.do_move        = 1;
    p.step           = step; // (stored actions: the Philox counter and key are the actor's draw)
    p.seed           = seed;
    return launch_step(e, p, static_cast<cudaStream_t>(stream), &q, wbytes);
}

int ok_discounted_returns(OkEnv *e, const float *d_rewards, const uint8_t *d_done, float *d_out, int32_t steps, int64_t n,
                          float gamma, void *stream)
{
    if (!e)
        return fail(OK_ERR_INVALID_ARG, "env is NULL");
    if (!e->has_device)
        return fail(OK_ERR_NO_DEVICE, "this env was created without a CUDA device (device = -1)");
    if (!d_rewards || !d_out || steps < 0 || n < 0)
        return fail(OK_ERR_INVALID_ARG, "bad arguments");
    if (steps == 0 || n == 0)
        return OK_SUCCESS;
    DeviceGuard g(e->cfg.device);
    const int   threads = 128;
    ok::discounted_returns_kernel<<<static_cast<unsigned>((n + threads - 1) / threads), threads, 0, static_cast<cudaStream_t>(stream)>>>(
        d_rewards, d_done, d_out, steps, n, gamma);
    OK_CUDA(cudaGetLastError());
    e->launches++;
    return OK_SUCCESS;
}

int ok_track_query(OkEnv *e, const float *d_x, const float *d_y, const int32_t *d_track, int64_t n, int32_t *d_idx,
                   float *d_lane, float *d_bound, void *stream)
{
    if (!e)
        return fail(OK_ERR_INVALID_ARG, "env is NULL");
    if (!e->has_device)
        return fail(OK_ERR_NO_DEVICE, "this env was created without a CUDA device (device = -1)");
    if (e->tracks.empty())
        return fail(OK_ERR_STATE, "no track has been added");
    if (n <= 0)
        return OK_SUCCESS;
    if (!d_x || !d_y)
        return fail(OK_ERR_INVALID_ARG, "query coordinates are NULL");
    if (n > (int64_t{1} << 31) / 32 * 255)
        return fail(OK_ERR_INVALID_ARG, "too many queries for one launch");
    DeviceGuard g(e->cfg.device);
    int         rc = ensure_arena(e);
    if (rc)
        return rc;
    ok::StepParams  p{};
    p.arena  = e->d_arena.get();
    p.tracks = e->d_track_refs.get();
    ok::QueryParams q{d_x, d_y, d_track, n, static_cast<int32_t>(e->tracks.size()), d_idx, d_lane, d_bound};
    const int       threads = 256;
    const int64_t   blocks  = (n * 32 + threads - 1) / threads;
    ok::track_query_kernel<<<static_cast<unsigned>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(p, q);
    OK_CUDA(cudaGetLastError());
    e->launches++;
    return OK_SUCCESS;
}

int ok_track_query_host(OkEnv *e, const float *h_x, const float *h_y, const int32_t *h_track, int64_t n, int32_t *h_idx,
                        float *h_lane, float *h_bound, void *stream)
{
    if (!e)
        return fail(OK_ERR_INVALID_ARG, "env is NULL");
    if (!e->has_device)
        return fail(OK_ERR_NO_DEVICE, "this env was created without a CUDA device (device = -1)");
    if (n <= 0)
        return OK_SUCCESS;
    if (!h_x || !h_y)
        return fail(OK_ERR_INVALID_ARG, "query coordinates are NULL");
    DeviceGuard  g(e->cfg.device);
    cudaStream_t s     = static_cast<cudaStream_t>(stream);
    const size_t bytes = 4 * static_cast<size_t>(n);
    uint8_t     *d     = nullptr;
    OK_CUDA(cudaMalloc(&d, 6 * bytes));
    float   *d_x = reinterpret_cast<float *>(d), *d_y = reinterpret_cast<float *>(d + bytes);
    int32_t *d_t = reinterpret_cast<int32_t *>(d + 2 * bytes), *d_i = reinterpret_cast<int32_t *>(d + 3 * bytes);
    float   *d_l = reinterpret_cast<float *>(d + 4 * bytes), *d_b = reinterpret_cast<float *>(d + 5 * bytes);
    cudaError_t err = cudaMemcpyAsync(d_x, h_x, bytes, cudaMemcpyHostToDevice, s);
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(d_y, h_y, bytes, cudaMemcpyHostToDevice, s);
    if (err == cudaSuccess && h_track)
        err = cudaMemcpyAsync(d_t, h_track, bytes, cudaMemcpyHostToDevice, s);
    int rc = OK_SUCCESS;
    if (err == cudaSuccess)
        rc = ok_track_query(e, d_x, d_y, h_track ? d_t : nullptr, n, h_idx ? d_i : nullptr, h_lane ? d_l : nullptr,
                            h_bound ? d_b : nullptr, stream);
    if (err == cudaSuccess && rc == OK_SUCCESS && h_idx)
        err = cudaMemcpyAsync(h_idx, d_i, bytes, cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess && rc == OK_SUCCESS && h_lane)
        err = cudaMemcpyAsync(h_lane, d_l, bytes, cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess && rc == OK_SUCCESS && h_bound)
        err = cudaMemcpyAsync(h_bound, d_b, bytes, cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess)
        err = cudaStreamSynchronize(s);
    cudaFree(d);
    if (rc)
        return rc;
    if (err != cudaSuccess)
        return fail(OK_ERR_CUDA, std::string("ok_track_query_host: ") + cudaGetErrorString(err));
    return OK_SUCCESS;
}

} // extern "C"
namespace
{
// ok_step_host / ok_step_host_q16: `h_obs` is float[N][R], or uint16_t[N][R] when `q16`
int step_host_impl(OkEnv *e, const float *h_thr, const float *h_steer, void *h_obs_any, const bool q16, float *h_reward, uint8_t *h_done,
                   void *stream)
{
    NvtxRange range(q16 ? "ok_step_host_q16" : "ok_step_host");
    float *h_obs = q16 ? nullptr : static_cast<float *>(h_obs_any);
    int rc = check_ready(e);
    if (rc)
        return rc;
    if ((h_thr == nullptr) != (h_steer == nullptr))
        return fail(OK_ERR_INVALID_ARG, "pass both action arrays or neither");
    DeviceGuard  g(e->cfg.device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t n = static_cast<size_t>(e->n_agents);
    ok::StepParams p = base_params(e);
    p.do_move        = 1;
    // Pinned buffers are used in place: the kernel reads the actions and writes obs / reward / done straight
    // through the host mapping, so both transfers overlap the tick.  Pageable buffers fall back to staged copies.
    static const bool act_by_copy = [] { // OK_HOST_ACT=copy: DMA the two action arrays instead of reading them through the mapping
        const char *v = std::getenv("OK_HOST_ACT");
        return v && std::strcmp(v, "copy") == 0;
    }();
    const float *a_thr = pinned_alias(h_thr), *a_steer = pinned_alias(h_steer);
    if (h_thr)
    {
        if (a_thr && a_steer && !act_by_copy)
        {
            p.ext_thr   = a_thr;
            p.ext_steer = a_steer;
            p.ext_host  = 1;
        }
        else
        {
            OK_CUDA(cudaMemcpyAsync(e->d_buf[OK_BUF_ACT_THROTTLE], h_thr, 4 * n, cudaMemcpyHostToDevice, s));
            OK_CUDA(cudaMemcpyAsync(e->d_buf[OK_BUF_ACT_STEER], h_steer, 4 * n, cudaMemcpyHostToDevice, s));
        }
    }
    // OK_HOST_OBS=copy: DMA copies after the kernel instead of stores through the host mapping.
    // OK_HOST_SMALL=copy: only reward / done by DMA (round 1's choice: one element per agent makes small PCIe writes);
    // round 2 measures the mapped stores ahead: they cost 8,192 sector-sized writes per tick and save two copy
    // operations on the critical path after the kernel.
    static const bool obs_by_copy = [] {
        const char *v = std::getenv("OK_HOST_OBS");
        return v && std::strcmp(v, "copy") == 0;
    }();
    static const bool small_by_copy = [] {
        const char *v = std::getenv("OK_HOST_SMALL");
        return v && std::strcmp(v, "copy") == 0;
    }();
    p.host_obs    = obs_by_copy ? nullptr : pinned_alias(h_obs);
    if (reinterpret_cast<uintptr_t>(p.host_obs) & 15u)
        p.host_obs = nullptr; // the tile flush stores 16 bytes per lane: a buffer that is not 16-byte aligned takes the staged copy
    p.host_reward = (obs_by_copy || small_by_copy) ? nullptr : pinned_alias(h_reward);
    p.host_done   = (obs_by_copy || small_by_copy) ? nullptr : pinned_alias(h_done);
    if (q16 && h_obs_any)
    { // the fixed-point observations exist only as what the kernel stores through the mapping: no staged fallback
        p.host_obs_q16 = pinned_alias(static_cast<uint16_t *>(h_obs_any));
        if (!p.host_obs_q16)
            return fail(OK_ERR_INVALID_ARG, "ok_step_host_q16: h_obs_q16 must be pinned host memory (ok_host_alloc / cudaHostRegister)");
        if (reinterpret_cast<uintptr_t>(p.host_obs_q16) & 15u)
            return fail(OK_ERR_INVALID_ARG, "ok_step_host_q16: h_obs_q16 must be 16-byte aligned (the tile flush stores 16 bytes per lane)");
    }
    rc = launch_step(e, p, s);
    if (rc)
        return rc;
    if (h_obs && !p.host_obs)
        OK_CUDA(cudaMemcpyAsync(h_obs, e->d_buf[OK_BUF_OBS], buffer_bytes(e, OK_BUF_OBS), cudaMemcpyDeviceToHost, s));
    if (h_reward && !p.host_reward)
        OK_CUDA(cudaMemcpyAsync(h_reward, e->d_buf[OK_BUF_REWARD], 4 * n, cudaMemcpyDeviceToHost, s));
    if (h_done && !p.host_done)
        OK_CUDA(cudaMemcpyAsync(h_done, e->d_buf[OK_BUF_DONE], n, cudaMemcpyDeviceToHost, s));
    OK_CUDA(cudaStreamSynchronize(s));
    return OK_SUCCESS;
}
} // namespace
extern "C"
{
int ok_step_host(OkEnv *e, const float *h_thr, const float *h_steer, float *h_obs, float *h_reward, uint8_t *h_done, void *stream)
{
    return step_host_impl(e, h_thr, h_steer, h_obs, false, h_reward, h_done, stream);
}

int ok_step_host_q16(OkEnv *e, const float *h_thr, const float *h_steer, uint16_t *h_obs_q16, float *h_reward, uint8_t *h_done,
                     void *stream)
{
    return step_host_impl(e, h_thr, h_steer, h_obs_q16, true, h_reward, h_done, stream);
}

int ok_packed_layout(const OkEnv *e, OkPackedLayout *out)
{
    if (!e || !out)
        return fail(OK_ERR_INVALID_ARG, "NULL argument");
    if (e->n_agents <= 0)
        return fail(OK_ERR_STATE, "ok_alloc_agents has not been called");
    static_assert(OK_BUF_POS_X == 0 && OK_BUF_SS_Y == 12 && OK_BUF_HIT_REL == OK_BUF_HIT_ABS + 1, "packed blocks follow the enum order");
    for (int b = 0; b <= OK_BUF_SS_Y; ++b)
        out->state_offset[b] = e->buf_off[b] - e->buf_off[OK_BUF_POS_X];
    out->state_bytes    = e->buf_off[OK_BUF_SS_Y] + buffer_bytes(e, OK_BUF_SS_Y) - e->buf_off[OK_BUF_POS_X];
    out->hit_abs_offset = 0;
    out->hit_rel_offset = e->buf_off[OK_BUF_HIT_REL] - e->buf_off[OK_BUF_HIT_ABS];
    out->hits_bytes     = out->hit_rel_offset + buffer_bytes(e, OK_BUF_HIT_REL);
    return OK_SUCCESS;
}

int ok_step_packed(OkEnv *e, void *h_state, void *h_hits, int32_t move, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (!h_state)
        return fail(OK_ERR_INVALID_ARG, "h_state is NULL");
    OkPackedLayout lay;
    rc = ok_packed_layout(e, &lay);
    if (rc)
        return rc;
    DeviceGuard  g(e->cfg.device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OK_CUDA(cudaMemcpyAsync(e->d_buf[OK_BUF_POS_X], h_state, lay.state_bytes, cudaMemcpyHostToDevice, s));
    ok::StepParams p = base_params(e);
    p.do_move        = move ? 1 : 0;
    rc               = launch_step(e, p, s);
    if (rc)
        return rc;
    OK_CUDA(cudaMemcpyAsync(h_state, e->d_buf[OK_BUF_POS_X], lay.state_bytes, cudaMemcpyDeviceToHost, s));
    if (h_hits)
        OK_CUDA(cudaMemcpyAsync(h_hits, e->d_buf[OK_BUF_HIT_ABS], lay.hits_bytes, cudaMemcpyDeviceToHost, s));
    OK_CUDA(cudaStreamSynchronize(s));
    return OK_SUCCESS;
}

int ok_host_alloc(void **h_ptr, size_t bytes)
{
    if (!h_ptr)
        return fail(OK_ERR_INVALID_ARG, "h_ptr is NULL");
    OK_CUDA(cudaMallocHost(h_ptr, bytes));
    return OK_SUCCESS;
}

int ok_host_free(void *h_ptr)
{
    OK_CUDA(cudaFreeHost(h_ptr));
    return OK_SUCCESS;
}

int ok_get_buffer(OkEnv *e, int32_t which, void **d_ptr, int64_t shape[3], int32_t *dtype)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (which < 0 || which >= OK_BUF_COUNT)
        return fail(OK_ERR_INVALID_ARG, "unknown buffer id");
    const BufferDesc d = describe(which);
    if (d_ptr)
        *d_ptr = e->d_buf[which];
    if (shape)
    {
        shape[0] = e->n_agents;
        shape[1] = d.per_ray >= 1 ? e->rays : 0;
        shape[2] = d.per_ray == 2 ? 2 : 0;
    }
    if (dtype)
        *dtype = d.dtype;
    return OK_SUCCESS;
}

int ok_read_buffer(OkEnv *e, int32_t which, void *h_dst, size_t bytes, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (which < 0 || which >= OK_BUF_COUNT || !h_dst)
        return fail(OK_ERR_INVALID_ARG, "bad buffer id or NULL destination");
    if (bytes > buffer_bytes(e, which))
        return fail(OK_ERR_INVALID_ARG, "read larger than the buffer");
    DeviceGuard  g(e->cfg.device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OK_CUDA(cudaMemcpyAsync(h_dst, e->d_buf[which], bytes, cudaMemcpyDeviceToHost, s));
    OK_CUDA(cudaStreamSynchronize(s));
    return OK_SUCCESS;
}

int ok_write_buffer(OkEnv *e, int32_t which, const void *h_src, size_t bytes, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (which < 0 || which >= OK_BUF_COUNT || !h_src)
        return fail(OK_ERR_INVALID_ARG, "bad buffer id or NULL source");
    if (which == OK_BUF_TRACK_ID)
        return fail(OK_ERR_INVALID_ARG, "track ids are fixed by ok_alloc_agents (the tile table depends on them)");
    if (bytes > buffer_bytes(e, which))
        return fail(OK_ERR_INVALID_ARG, "write larger than the buffer");
    DeviceGuard  g(e->cfg.device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OK_CUDA(cudaMemcpyAsync(e->d_buf[which], h_src, bytes, cudaMemcpyHostToDevice, s));
    OK_CUDA(cudaStreamSynchronize(s));
    return OK_SUCCESS;
}

int ok_sync(OkEnv *e, void *stream)
{
    if (!e || !e->has_device)
        return fail(OK_ERR_NO_DEVICE, "no device");
    DeviceGuard g(e->cfg.device);
    OK_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    return OK_SUCCESS;
}

int ok_eval_sincosf(OkEnv *e, const float *h_in, float *h_sin, float *h_cos, int64_t n)
{
    if (!e || !e->has_device)
        return fail(OK_ERR_NO_DEVICE, "no device");
    if (!h_in || !h_sin || !h_cos || n <= 0)
        return fail(OK_ERR_INVALID_ARG, "bad arguments");
    DeviceGuard g(e->cfg.device);
    float      *d = nullptr;
    OK_CUDA(cudaMalloc(&d, sizeof(float) * 3 * static_cast<size_t>(n)));
    cudaError_t err = cudaMemcpy(d, h_in, sizeof(float) * n, cudaMemcpyHostToDevice);
    if (err == cudaSuccess)
    {
        ok::sincosf_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(d, d + n, d + 2 * n, n);
        e->launches++;
        err = cudaMemcpy(h_sin, d + n, sizeof(float) * n, cudaMemcpyDeviceToHost);
        if (err == cudaSuccess)
            err = cudaMemcpy(h_cos, d + 2 * n, sizeof(float) * n, cudaMemcpyDeviceToHost);
    }
    cudaFree(d);
    if (err != cudaSuccess)
        return fail(OK_ERR_CUDA, cudaGetErrorString(err));
    return OK_SUCCESS;
}

static int host_beam(OkEnv *e, int32_t id)
{
    if (!e || id < 0 || id >= static_cast<int32_t>(e->tracks.size()))
        return fail(OK_ERR_INVALID_ARG, "bad track id");
    e->beams.resize(e->tracks.size());
    if (e->beams[id])
        return OK_SUCCESS;
    std::string err;
    if (e->has_device)
    { // the table the kernels use, copied back
        auto dev = beam_device_table_for(e->tracks[id], beam_config(e), e->cfg.device, true, err);
        if (!dev)
            return fail(OK_ERR_INVALID_ARG, "beam table: " + err);
        auto        host = std::make_shared<std::vector<uint8_t>>(dev->bytes);
        DeviceGuard g(e->cfg.device);
        OK_CUDA(cudaMemcpy(host->data(), dev->ptr, dev->bytes, cudaMemcpyDeviceToHost));
        e->beams[id] = host;
        return OK_SUCCESS;
    }
    e->beams[id] = beam_table_for(e->tracks[id], beam_config(e), true, err);
    if (!e->beams[id])
        return fail(OK_ERR_INVALID_ARG, "beam table: " + err);
    return OK_SUCCESS;
}

int32_t ok_beam_lookup(OkEnv *e, int32_t id, float x, float y, float angle, uint16_t *h_items, int32_t capacity,
                       float *d_complete)
{
    return ok_beam_lookup_ex(e, id, x, y, angle, h_items, capacity, d_complete, nullptr, nullptr);
}

int32_t ok_beam_lookup_ex(OkEnv *e, int32_t id, float x, float y, float angle, uint16_t *h_items, int32_t capacity,
                          float *d_complete, float *d_inline, int32_t *n_inline)
{
    int rc = host_beam(e, id);
    if (rc)
        return rc;
    std::vector<uint16_t> items;
    float                 d = 0.0f;
    if (!ok::beam_lookup(*e->beams[id], x, y, angle, items, d, d_inline, n_inline))
        return OK_BEAM_NOT_COVERED;
    if (d_complete)
        *d_complete = d;
    if (h_items && capacity > 0)
        std::memcpy(h_items, items.data(), 2 * std::min<size_t>(items.size(), static_cast<size_t>(capacity)));
    return static_cast<int32_t>(items.size());
}

void ok_release_caches(void)
{
    std::lock_guard<std::mutex> lock(g_beam_mu);
    g_beam_cache.clear();
    g_beam_dev_cache.clear(); // tables still referenced by live envs stay alive until those envs are destroyed
    ok::beam_builder_release();
}

int64_t ok_beam_table_bytes(OkEnv *e, int32_t id)
{
    int rc = host_beam(e, id);
    if (rc)
        return rc;
    return static_cast<int64_t>(e->beams[id]->size());
}

int ok_pcie_probe(int32_t device, size_t bytes, int32_t iters, int32_t mode, double *gbps_out)
{
    if (!gbps_out || bytes < 16 || iters < 1 || mode < 0 || mode > 2)
        return fail(OK_ERR_INVALID_ARG, "ok_pcie_probe: bad arguments");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count)
        return fail(OK_ERR_NO_DEVICE, "ok_pcie_probe: no such CUDA device");
    DeviceGuard  g(device);
    bytes        = bytes / 16 * 16;
    void        *h = nullptr, *d = nullptr;
    cudaStream_t s = nullptr;
    cudaEvent_t  e0 = nullptr, e1 = nullptr;
    cudaError_t  err = cudaMallocHost(&h, bytes);
    if (err == cudaSuccess)
        err = cudaMalloc(&d, bytes);
    if (err == cudaSuccess)
        err = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    if (err == cudaSuccess)
        err = cudaEventCreate(&e0);
    if (err == cudaSuccess)
        err = cudaEventCreate(&e1);
    if (err == cudaSuccess)
    {
        std::memset(h, 0, bytes);
        cudaMemsetAsync(d, 1, bytes, s);
        int probe_grid = 296; // (OK_PROBE_GRID: how many CTAs it takes to fill the link with stores)
        if (const char *env = std::getenv("OK_PROBE_GRID"))
            probe_grid = std::max(1, std::atoi(env));
        auto once = [&]() {
            if (mode == 0)
                cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, s);
            else if (mode == 2)
                cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s);
            else
                ok::probe_store_kernel<<<probe_grid, 512, 0, s>>>(static_cast<const float4 *>(d), static_cast<float4 *>(h), bytes / 16);
        };
        for (int i = 0; i < 3; ++i)
            once();
        cudaEventRecord(e0, s);
        for (int i = 0; i < iters; ++i)
            once();
        cudaEventRecord(e1, s);
        err = cudaStreamSynchronize(s);
        float ms = 0.0f;
        if (err == cudaSuccess)
            err = cudaEventElapsedTime(&ms, e0, e1);
        if (err == cudaSuccess)
            *gbps_out = static_cast<double>(bytes) * iters / (static_cast<double>(ms) * 1e6);
    }
    if (e0)
        cudaEventDestroy(e0);
    if (e1)
        cudaEventDestroy(e1);
    if (s)
        cudaStreamDestroy(s);
    if (d)
        cudaFree(d);
    if (h)
        cudaFreeHost(h);
    if (err != cudaSuccess)
        return fail(OK_ERR_CUDA, std::string("ok_pcie_probe: ") + cudaGetErrorString(err));
    return OK_SUCCESS;
}

int ok_debug_stats(OkEnv *e, uint64_t out[4], int32_t enable)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    DeviceGuard g(e->cfg.device);
    if (out)
    {
        out[0] = out[1] = out[2] = out[3] = 0;
        if (e->ag.stats)
            OK_CUDA(cudaMemcpy(out, e->ag.stats.get(), 32, cudaMemcpyDeviceToHost));
    }
    if (enable && !e->ag.stats)
    {
        OK_CUDA(dev_alloc(e->ag.stats, 4));
    }
    if (e->ag.stats)
        OK_CUDA(cudaMemset(e->ag.stats.get(), 0, 32));
    if (!enable && e->ag.stats)
    {
        OK_CUDA(cudaDeviceSynchronize());
        e->ag.stats.reset();
    }
    return OK_SUCCESS;
}

int ok_debug_violations(OkEnv *e, uint64_t *count, int32_t *checks_compiled_in)
{
    if (!e || !e->has_device)
        return fail(OK_ERR_NO_DEVICE, "no device");
    DeviceGuard g(e->cfg.device);
    OK_CUDA(cudaDeviceSynchronize());
    unsigned long long staged = 0, unstaged = 0, actor = 0, grid = 0;
    OK_CUDA(ok::violations_step_staged(&staged));
    OK_CUDA(ok::violations_step_unstaged(&unstaged));
    OK_CUDA(ok::violations_step_actor(&actor));
    OK_CUDA(ok::violations_step_grid(&grid));
    if (count)
        *count = staged + unstaged + actor + grid;
    if (checks_compiled_in)
        *checks_compiled_in = OK_CHECKED;
    return OK_SUCCESS;
}

int ok_balance_schedule(OkEnv *e, void *stream, float out[2])
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    DeviceGuard g(e->cfg.device);
    if (e->cfg.raycast_mode == OK_RAYCAST_BEAM)
        if ((rc = rebalance_beam_tiles(e, static_cast<cudaStream_t>(stream))))
            return rc;
    if (out)
        out[0] = e->balance_before, out[1] = e->balance_after;
    return OK_SUCCESS;
}

int64_t ok_debug_tiles(OkEnv *e, int64_t *h_out, int64_t capacity)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    const Schedule &beam = e->ag.beam;
    if (e->cfg.raycast_mode != OK_RAYCAST_BEAM || !beam.d)
        return 0;
    DeviceGuard           g(e->cfg.device);
    std::vector<ok::Tile> tiles(static_cast<size_t>(beam.n));
    OK_CUDA(cudaMemcpy(tiles.data(), beam.d.get(), sizeof(ok::Tile) * tiles.size(), cudaMemcpyDeviceToHost));
    for (int64_t i = 0; h_out && i < std::min<int64_t>(capacity, beam.n); ++i)
        h_out[3 * i] = tiles[i].track, h_out[3 * i + 1] = tiles[i].count, h_out[3 * i + 2] = tiles[i].begin;
    return beam.n;
}

int64_t ok_debug_trace(OkEnv *e, uint64_t *h_out, int64_t capacity_words, int32_t tiles_per_cta)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    DeviceGuard  g(e->cfg.device);
    Agents      &ag    = e->ag;
    const size_t words = static_cast<size_t>(ag.beam.grid) * static_cast<size_t>(std::max(ag.trace_tiles, 0)) * 6;
    int64_t      got   = 0;
    OK_CUDA(cudaDeviceSynchronize());
    if (h_out && ag.trace && words)
    {
        got = static_cast<int64_t>(std::min<size_t>(words, static_cast<size_t>(std::max<int64_t>(capacity_words, 0))));
        OK_CUDA(cudaMemcpy(h_out, ag.trace.get(), 8 * static_cast<size_t>(got), cudaMemcpyDeviceToHost));
    }
    if (ag.trace && tiles_per_cta != ag.trace_tiles)
        ag.trace.reset(), ag.trace_tiles = 0;
    if (tiles_per_cta > 0)
    {
        const size_t words_new = static_cast<size_t>(ag.beam.grid) * tiles_per_cta * 6;
        if (!ag.trace)
            OK_CUDA(dev_alloc(ag.trace, words_new));
        OK_CUDA(cudaMemset(ag.trace.get(), 0, 8 * words_new));
        ag.trace_tiles = tiles_per_cta;
    }
    return got;
}

int ok_population_counters(OkEnv *e, OkPopulationCounters *out, void *stream)
{
    int rc = check_ready(e);
    if (rc)
        return rc;
    if (!out)
        return fail(OK_ERR_INVALID_ARG, "out is NULL");
    NvtxRange    range("ok_population_counters");
    DeviceGuard  g(e->cfg.device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!e->d_counters)
        OK_CUDA(dev_alloc(e->d_counters, 4));
    OK_CUDA(cudaMemsetAsync(e->d_counters.get(), 0, 4 * sizeof(unsigned long long), s));
    const int threads = 256;
    const int blocks  = static_cast<int>(std::min<int64_t>((e->n_agents + threads - 1) / threads, 4 * e->num_sms));
    ok::population_counters_kernel<<<blocks, threads, 0, s>>>(static_cast<const uint8_t *>(e->d_buf[OK_BUF_CRASHED]),
                                                               static_cast<const uint8_t *>(e->d_buf[OK_BUF_TIMED_OUT]),
                                                               static_cast<const uint8_t *>(e->d_buf[OK_BUF_DONE]), e->n_agents, e->d_counters.get());
    OK_CUDA(cudaGetLastError());
    e->launches++;
    unsigned long long h[4];
    OK_CUDA(cudaMemcpyAsync(h, e->d_counters.get(), sizeof h, cudaMemcpyDeviceToHost, s));
    OK_CUDA(cudaStreamSynchronize(s));
    out->agents = static_cast<uint64_t>(e->n_agents);
    out->alive = h[0], out->crashed = h[1], out->timed_out = h[2], out->done = h[3];
    return OK_SUCCESS;
}

int ok_launch_stats(const OkEnv *e, OkLaunchStats *out)
{
    if (!e || !out)
        return fail(OK_ERR_INVALID_ARG, "NULL argument");
    out->kernel_launches = e->launches;
    const Schedule &sch  = e->cfg.raycast_mode == OK_RAYCAST_BEAM ? e->ag.beam : e->ag.tiles;
    out->grid_blocks     = sch.grid;
    out->block_threads   = e->cfg.raycast_mode == OK_RAYCAST_BEAM ? e->beam_block : ok::kGridBlock;
    out->smem_bytes      = static_cast<int32_t>(e->cfg.raycast_mode == OK_RAYCAST_BEAM ? e->smem_beam : e->smem);
    out->tiles           = sch.n;
    return OK_SUCCESS;
}
}
