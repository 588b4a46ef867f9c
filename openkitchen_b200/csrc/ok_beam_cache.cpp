// ok_beam_cache.cpp -- the beam-table caches and the choice of builder (ok_beam_cache.hpp)
#include "ok_beam_cache.hpp"

#include "../../include/openkitchen_b200.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fcntl.h>
#include <map>
#include <mutex>
#include <sys/stat.h>
#include <thread>
#include <unistd.h>

namespace ok
{

DeviceBlob::~DeviceBlob()
{
    if (ptr)
    {
        DeviceGuard g(device);
        cudaFree(ptr); // an error after the runtime has shut down is harmless
    }
}

namespace
{
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

std::string beam_key(const Track &t, const BeamConfig &cfg)
{
    uint64_t h = fnv1a(t.segments.data(), t.segments.size() * sizeof(float));
    h          = fnv1a(t.x.data(), t.x.size() * sizeof(float), h);
    h          = fnv1a(t.y.data(), t.y.size() * sizeof(float), h);
    h          = fnv1a(t.w_left.data(), t.w_left.size() * sizeof(float), h);
    h          = fnv1a(t.w_right.data(), t.w_right.size() * sizeof(float), h);
    char key[128];
    std::snprintf(key, sizeof key, "v%d-%016llx-%zu-%g-%d-%g", kBeamBuildVersion, static_cast<unsigned long long>(h),
                  t.segments.size(), static_cast<double>(cfg.cell), cfg.bins, static_cast<double>(cfg.range));
    return key;
}

std::string device_key(const Track &t, const BeamConfig &cfg, int device)
{
    return beam_key(t, cfg) + "@" + std::to_string(device);
}

// OK_BEAM_BUILDER: cpu = host builder only; gpu = device builder only (its failure is an error); else the device builder,
// the host one where it fails
enum class Builder
{
    Automatic,
    Cpu,
    Gpu
};
Builder beam_builder()
{
    const char *force = std::getenv("OK_BEAM_BUILDER");
    if (force && std::strcmp(force, "cpu") == 0)
        return Builder::Cpu;
    if (force && std::strcmp(force, "gpu") == 0)
        return Builder::Gpu;
    return Builder::Automatic;
}

std::mutex                                                          g_beam_mu; // guards both caches
std::map<std::string, HostTable>                                    g_beam_cache;
// never destroyed: at process exit the CUDA runtime may already be gone when static destructors run
std::map<std::string, DeviceTable> &g_beam_dev_cache = *new std::map<std::string, DeviceTable>();

size_t table_bytes(const HostTable &t)
{
    return t->size();
}
size_t table_bytes(const DeviceTable &t)
{
    return t->bytes;
}

// inserts `table` into `cache`, emptied first when the two would hold more than `limit` bytes; g_beam_mu held.  Envs keep
// their own references: this only bounds what the cache itself pins.
template <typename T> T remember(std::map<std::string, T> &cache, const std::string &key, T table, size_t limit)
{
    size_t held = table_bytes(table);
    for (auto &kv : cache)
        held += table_bytes(kv.second);
    if (held > limit)
        cache.clear();
    cache[key] = table;
    return table;
}

HostTable beam_cached(const std::string &key)
{
    std::lock_guard<std::mutex> lock(g_beam_mu);
    auto                        it = g_beam_cache.find(key);
    return it == g_beam_cache.end() ? nullptr : it->second;
}

HostTable beam_remember(const std::string &key, std::shared_ptr<std::vector<uint8_t>> blob)
{
    std::lock_guard<std::mutex> lock(g_beam_mu);
    return remember<HostTable>(g_beam_cache, key, blob, size_t{12} << 30);
}

// The track's table built on the host.  `wait` = false: return nullptr (no error) when another process holds the
// track's build lock, so that the caller can build other tracks in the meantime; `wait` = true: wait for that process's
// file, or build after a timeout.
HostTable beam_table_for(const Track &t, const BeamConfig &cfg, bool wait, std::string &err)
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
    const bool built = build_beam_table(t, cfg, *blob, err);
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

// The track's table in the memory of `device`: built there by the device builder, or on the host and uploaded (see
// Builder).  `wait` as in beam_table_for.
DeviceTable beam_device_table_for(const Track &t, const BeamConfig &cfg, int device, Builder builder, bool wait, std::string &err)
{
    const std::string key = device_key(t, cfg, device);
    {
        std::lock_guard<std::mutex> lock(g_beam_mu);
        auto                        it = g_beam_dev_cache.find(key);
        if (it != g_beam_dev_cache.end())
            return it->second;
    }
    DeviceTable out;
    if (builder != Builder::Cpu)
    {
        uint8_t    *d = nullptr;
        size_t      bytes = 0;
        std::string gerr;
        if (build_beam_table_device(t, cfg, device, &d, &bytes, gerr))
            out = std::make_shared<DeviceBlob>(d, bytes, device);
        else if (builder == Builder::Gpu)
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
    return remember<DeviceTable>(g_beam_dev_cache, key, out, size_t{24} << 30);
}
} // namespace

BeamConfig beam_config(float cell, int32_t bins)
{
    BeamConfig c;
    c.cell  = cell;
    c.bins  = bins;
    c.range = 200.0f; // Agent::kSensorRange; a larger OkConfig::sensor_range stays exact through the grid walk
    if (const char *env = std::getenv("OK_BEAM_THREADS"))
        c.threads = std::atoi(env);
    else if (const char *lws = std::getenv("LOCAL_WORLD_SIZE")) // torchrun: the ranks of a box share its cores
        c.threads = std::max(1, static_cast<int>(std::thread::hardware_concurrency()) / std::max(1, std::atoi(lws)));
    return c;
}

int beam_device_tables(const std::vector<Track> &tracks, const BeamConfig &cfg, int device, std::vector<DeviceTable> &tables,
                       std::string &err)
{
    const Builder builder = beam_builder();
    const bool    verbose = std::getenv("OK_BEAM_VERBOSE") != nullptr;
    const auto    t_0     = std::chrono::steady_clock::now();
    tables.resize(tracks.size());
    if (builder != Builder::Cpu)
    { // the tables nobody has built yet in this process, all at once: the device builder pipelines them
        std::vector<const Track *> todo;
        std::vector<std::string>   keys;
        {
            std::lock_guard<std::mutex> lock(g_beam_mu);
            for (size_t i = 0; i < tracks.size(); ++i)
            {
                const std::string key = device_key(tracks[i], cfg, device);
                if (!tables[i] && !g_beam_dev_cache.count(key) && std::find(keys.begin(), keys.end(), key) == keys.end())
                    todo.push_back(&tracks[i]), keys.push_back(key);
            }
        }
        if (todo.size() > 1)
        {
            std::vector<uint8_t *> blobs;
            std::vector<size_t>    sizes;
            build_beam_tables_device(todo, cfg, device, blobs, sizes);
            std::lock_guard<std::mutex> lock(g_beam_mu);
            for (size_t k = 0; k < todo.size(); ++k)
                if (blobs[k])
                    g_beam_dev_cache[keys[k]] = std::make_shared<DeviceBlob>(blobs[k], sizes[k], device);
        }
    }
    // (host-built tables only) first every table nobody else is building, then the ones other ranks were busy with
    for (int pass = 0; pass < 2; ++pass)
        for (size_t i = 0; i < tracks.size(); ++i)
            if (!tables[i])
            {
                std::string why;
                tables[i] = beam_device_table_for(tracks[i], cfg, device, builder, pass == 1, why);
                if (!tables[i] && (pass == 1 || !why.empty()))
                {
                    err = "beam table: " + why;
                    return OK_ERR_INVALID_ARG;
                }
            }
    const auto t_1 = std::chrono::steady_clock::now();
    beam_builder_release(); // the device builder's scratch pool (kept from track to track) is no longer needed
    if (verbose)
        std::fprintf(stderr, "[ensure_arena] tables %.1f ms, pool release %.1f ms\n", std::chrono::duration<double, std::milli>(t_1 - t_0).count(),
                     std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_1).count());
    return OK_SUCCESS;
}

int beam_host_table(const Track &t, const BeamConfig &cfg, int device, HostTable &table, std::string &err)
{
    std::string why;
    if (device >= 0)
    { // the table the kernels use, copied back
        DeviceTable dev = beam_device_table_for(t, cfg, device, beam_builder(), true, why);
        if (!dev)
        {
            err = "beam table: " + why;
            return OK_ERR_INVALID_ARG;
        }
        auto        host = std::make_shared<std::vector<uint8_t>>(dev->bytes);
        DeviceGuard g(device);
        if (const cudaError_t rc = cudaMemcpy(host->data(), dev->ptr, dev->bytes, cudaMemcpyDeviceToHost); rc != cudaSuccess)
        {
            err = std::string("beam table copy: ") + cudaGetErrorString(rc);
            return OK_ERR_CUDA;
        }
        table = host;
        return OK_SUCCESS;
    }
    table = beam_table_for(t, cfg, true, why);
    if (!table)
    {
        err = "beam table: " + why;
        return OK_ERR_INVALID_ARG;
    }
    return OK_SUCCESS;
}

void beam_release_caches()
{
    std::lock_guard<std::mutex> lock(g_beam_mu);
    g_beam_cache.clear();
    g_beam_dev_cache.clear();
    beam_builder_release();
}

} // namespace ok
