// ok_beam_cache.hpp -- where a track's beam table comes from.
//
// Beam tables are pure functions of (segments, cell, bins, range) and take ~0.1-1 s of host time per track.  A table is
// built on the device (ok_beam_gpu.cu) or, with OK_BEAM_BUILDER=cpu, for host-only envs and when the device builder
// fails, on the host (ok_beam.cpp).  Three caches: one per process for device tables and one for host tables (envs over
// the same tracks share a table), and one on disk for host tables ($OK_BEAM_CACHE_DIR, default
// $TMPDIR/openkitchen_b200-cache-<uid>; OK_BEAM_CACHE=0 disables it) so that the ranks of one box -- which all need
// every table -- build each table once between them instead of once each.
#pragma once

#include "ok_beam.hpp"

#include <cuda_runtime.h>

#include <memory>
#include <string>
#include <vector>

namespace ok
{

// makes `dev` the current device for the guard's lifetime (dev < 0: does nothing)
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
    ~DeviceBlob();
};

using HostTable   = std::shared_ptr<const std::vector<uint8_t>>;
using DeviceTable = std::shared_ptr<const DeviceBlob>;

// the tables of an env of OkConfig::beam_cell / beam_bins; OK_BEAM_THREADS (or torchrun's LOCAL_WORLD_SIZE) sets the
// host builder's threads
BeamConfig beam_config(float cell, int32_t bins);

// The table of every track in the memory of `device`: tables[i] for tracks[i], entries already set are kept.  The tables
// no env of the process has built yet are built together, pipelined.  OK_SUCCESS, or an OK_ERR_* code with `err`.
int beam_device_tables(const std::vector<Track> &tracks, const BeamConfig &cfg, int device, std::vector<DeviceTable> &tables,
                       std::string &err);

// A host copy of one track's table: the device table copied back when device >= 0, the host-built one otherwise.
int beam_host_table(const Track &t, const BeamConfig &cfg, int device, HostTable &table, std::string &err);

// drops every table the caches hold (tables still referenced by live envs stay alive until those envs are destroyed)
void beam_release_caches();

} // namespace ok
