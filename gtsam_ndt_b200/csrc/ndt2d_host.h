// Host-side internals shared by the C-ABI translation units (ndt2d_capi.cu, ndt2d_pairs.cu, ndt2d_exchange.cu):
// the handle, its device buffers, error reporting and the helpers every entry point uses. Not part of the ABI.
#pragma once
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "ndt2d_internal.h"

namespace ndt2d {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

// A table every rank owns a copy of and every rank writes into, through CUDA IPC peer pointers, from inside a kernel:
// nslots rows of `world` blocks of block_bytes, block r of row (query % nslots) written by rank r. The first 32 bytes of a
// block are an ndt2d_best-shaped header whose epoch word (offset 16) = query + 1 is stored last, after a system-scope
// fence. Reading is a host-side poll of the OWN table (see peer_wait_row in ndt2d_exchange.cu).
struct PeerTable {
    int world = 0, rank = 0, slots = 0;
    size_t block_bytes = 0;
    unsigned char *table[NDT2D_MAX_RANKS] = {};
    bool opened[NDT2D_MAX_RANKS] = {};
    unsigned char *host = nullptr;      // pinned: the polled row, then a verified snapshot of the whole table
    std::vector<char> verified_ok;      // per row: the snapshot holds a verified, complete row
    size_t row_bytes() const { return (size_t)world * block_bytes; }
};

struct LevelMem {
    float4 *cells = nullptr;
    uint32_t *cnt = nullptr;
    unsigned long long *sums = nullptr;
    unsigned *dirty = nullptr; // incremental updates: one word per cell, zero between calls (allocated on the first ndt2d_add_target)
    int64_t cap = 0; // cells the allocations can hold (plus the zero records behind the table, see ZERO_PAD)
    // all-zero records behind a dense table: a point outside the lattice gathers records sentinel + {0, 1, njx, njx + 1}
    static int64_t zero_pad(int64_t njx) { return njx + 2; }
    unsigned char *base = nullptr; // ONE allocation: cells | sums | cnt, each sized for `cap` cells - a new target clears it with one memset
    size_t bytes = 0;
    void release()
    {
        if (base) cudaFree(base);
        if (dirty) cudaFree(dirty);
        base = nullptr; cells = nullptr; cnt = nullptr; sums = nullptr; dirty = nullptr;
        cap = 0; bytes = 0;
    }
    // Grow-only: scan-to-scan odometry sets a new target of about the same size for every scan, and a
    // cudaFree/cudaMalloc pair per level and call costs more than building the grid.
    cudaError_t ensure(int64_t nc, int64_t pad)
    {
        if (nc + pad <= cap) return cudaSuccess;
        release();
        const int64_t want = nc + pad + nc / 4 + 1024;
        cudaError_t e = cudaMalloc(&base, (size_t)want * 76);
        if (e != cudaSuccess) { release(); return e; }
        cells = reinterpret_cast<float4 *>(base);                                            // want * 32 bytes
        sums = reinterpret_cast<unsigned long long *>(base + (size_t)want * 32);              // want * 40
        cnt = reinterpret_cast<uint32_t *>(base + (size_t)want * 72);                         // want * 4
        cap = want;
        bytes = (size_t)want * 76;
        return cudaSuccess;
    }
};


} // namespace ndt2d

struct ndt2d_matcher {
    int device = 0;
    bool own_stream = false;
    ndt2d::LaunchCfg cfg{};
    ndt2d_params prm{};
    int nlevels = 1;
    float res[NDT2D_MAX_LEVELS] = {1.0f};
    bool explicit_grid = false;
    float gox = 0, goy = 0, gex = 0, gey = 0;
    bool has_target = false;
    bool sums_valid = false;
    ndt2d::LevelDev lv[NDT2D_MAX_LEVELS]{};
    ndt2d::LevelMem mem[NDT2D_MAX_LEVELS];
    ndt2d::DevBuf b_xy, b_off, b_init, b_res, b_pose, b_out, b_cnt, b_idx, b_terms, b_hyp, b_scores, b_tki, b_tkv, b_scratch,
        b_counter, b_beams, b_ranges, b_box, b_ptab, b_pcnt, b_psums, b_pgeo, b_ptargets, b_ppairs, b_perr, b_reloc,
        b_scand, b_sjobs, b_sinit,    // ndt2d_relocalize_pairs / _batch: per-chunk candidates, refinement jobs and their initial poses
        b_slevels,                    // ndt2d_relocalize_batch: the device copy of lv[] its sweep reads
        b_tpose,                      // targets from posed scans: per scan {cos, sin, p0, p1}
        b_sm_off, b_sm_start, b_sm_base, b_sm_pose, b_sm_tab;   // calls over submaps: their SubmapDev tables and member poses
    std::vector<int32_t> h_spairs;  // ndt2d_relocalize_pairs: the host copy its pairs are uploaded from
    std::vector<int64_t> h_sm_start, h_sm_base;   // calls over submaps: the host copies of SubmapDev::start and ::base
    int64_t reloc_off[2] = {0, 0}; // source of the asynchronous offsets upload of ndt2d_relocalize_device
    double beams_amin = 0, beams_ainc = 0;
    int beams_n = 0;
    // host-buffer batch calls are cut into chunks: chunk i+1 is copied on copy_stream while chunk i computes
    static constexpr int MAX_CHUNKS = 16;
    cudaStream_t copy_stream = nullptr;
    cudaStream_t work_stream[2] = {nullptr, nullptr}; // chunk kernels alternate so one chunk's tail overlaps the next
    cudaEvent_t ev_chunk[MAX_CHUNKS] = {};
    cudaEvent_t ev_begin = nullptr, ev_done[2] = {nullptr, nullptr};
    // multi-GPU exchanges over peer memory: the best hypothesis of a sharded sweep (ndt2d_exchange_*) and the refined
    // candidates of a sharded relocalisation (ndt2d_reloc_*)
    ndt2d::PeerTable ex, rx;
    int rx_k = 0;                   // candidates per rank and query in `rx`
    // upload relay (ndt2d_set_upload_relay): a share of the chunks of a host-buffer call travels host -> relay GPU over that
    // GPU's PCIe link, then relay GPU -> this GPU over NVLink
    int relay_dev = -1;
    double relay_frac = 0.0;
    cudaStream_t relay_stream = nullptr;       // on relay_dev: host -> relay buffer
    cudaStream_t relay_peer_stream = nullptr;  // on this device: relay buffer -> input buffer
    cudaEvent_t ev_relay[MAX_CHUNKS] = {};     // on relay_dev
    void *relay_buf = nullptr;                 // on relay_dev, relay_cap bytes
    size_t relay_cap = 0;
    // low-latency path of small host-buffer calls (a single align is 3 CUDA calls): pinned staging for one packed upload,
    // results written by the kernel straight into mapped pinned memory, work-queue counters from a pre-zeroed ring
    static constexpr size_t FAST_BYTES = 256 << 10;
    static constexpr int FAST_SCANS = 256, RING = 4096;
    bool fast_ready = false;                 // every allocation of the fast path exists and the ring is zeroed
    unsigned char *fast_host = nullptr;      // pinned + mapped, FAST_BYTES
    unsigned char *fast_host_dev = nullptr;  // its device address: small xy calls are staged by the kernel from there
    ndt2d_result *fast_res = nullptr;        // pinned + mapped, FAST_SCANS records
    ndt2d_result *fast_res_dev = nullptr;    // its device address
    ndt2d::DevBuf b_fast, b_ring;
    int ring_pos = 0;
    int64_t launches = 0;
    std::string err;
};

namespace ndt2d {

// records the message (ndt2d_last_error) and returns `code`
int fail(ndt2d_matcher *m, int code, const char *fmt, ...);

#define CK(m, call)                                                                                        \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return fail(m, e_ == cudaErrorMemoryAllocation ? NDT2D_ENOMEM : NDT2D_ECUDA, "%s: %s", #call, \
                        cudaGetErrorString(e_));                                                           \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev)
    {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int check_level(ndt2d_matcher *m, int level);
int upload(ndt2d_matcher *m, DevBuf &b, const void *src, size_t bytes);
// Launches one align. The caller sets the scans' input in `a` and leaves the fields it does not use zero: xy and offsets
// (points; also job_scan, or pairs and geo), or ranges, ranges_u16, nbeams and the range limits (LaserScan ranges, whose
// beam table is made from angle_min / angle_inc); then init, res and nscans, and its own work-queue counter and batch_scans
// where it has them. This fills in the target's levels, the parameters, the shared-memory capacity for scans of up to
// max_points points and, when counter is unset, the handle's work-queue counter.
int align_device(ndt2d_matcher *m, AlignArgs a, int max_points, double angle_min = 0.0, double angle_inc = 0.0);

} // namespace ndt2d
