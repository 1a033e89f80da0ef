// Internal (non-ABI) declarations shared by the kernels and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "ndt2d.h"

namespace ndt2d {

// One pyramid level as the kernels see it (SPEC 2). Passed by value in kernel parameters.
struct LevelDev {
    const float4 *cells;      // njx*njy records, two float4 each, followed by one all-zero sentinel record
    uint32_t *cnt;            // njx*njy
    unsigned long long *sums; // njx*njy*5, two's-complement i64
    float res, st, inv_st, ox, oy;
    int nhx, nhy, njx, njy, ov;
    double inv_std;           // SPEC 2: 1.0 / (double)st, the f64 scale of the lattice index
    double qs, qu;            // SPEC 3: fixed-point scale 2^22 / res and its unit res * 2^-22
    // 0: `cells` is the dense table indexed by jy*njx+jx. Otherwise `cells` is an open-addressing hash table of
    // hash_mask+1 records keyed by that index (the key sits in the record's `n` word, 0xffffffff = empty slot), with the
    // sentinel record at index hash_mask+1: the per-target tables of the batched scan-to-scan path (ndt2d_align_pairs).
    unsigned hash_mask;
    unsigned zero_rec;        // shared-memory tables of the fused pairs path only (TABLE_SHASH in ndt2d_device.cuh)
};

static constexpr unsigned kEmptyKey = 0xffffffffu;

// SPEC 2 and 3: the strides and fixed-point scales of a level of cell size res (ov: overlapping cells)
__host__ __device__ inline void level_strides(LevelDev &L, float res, int ov)
{
    L.res = res;
    L.ov = ov;
    L.st = ov ? res * 0.5f : res;
    L.inv_st = 1.0f / L.st;
    L.inv_std = 1.0 / (double)L.st;
    L.qs = 4194304.0 / (double)res;
    L.qu = (double)res * (1.0 / 4194304.0);
}

// SPEC 2 geometry of a level: its strides, and its lattice on the explicit grid (origin gox, goy; extent gex, gey) or
// auto-fitted to the bounding box {xmin, ymin, xmax, ymax} of the target's finite points. The host builds and the kernels
// that build a target scan's grid themselves (ndt2d_pairs.cu) share this one definition, so a pairs result equals
// set_target(scan) + align. The library is compiled with -fmad=false and -ffp-contract=off: every operation here is the
// IEEE one on both sides. Returns whether the lattice is usable: not empty, and fewer than 2^31 cells.
__host__ __device__ inline bool level_geometry(LevelDev &L, float res, int ov, bool explicit_grid, float gox, float goy, float gex,
                                               float gey, float xmin, float ymin, float xmax, float ymax)
{
    level_strides(L, res, ov);
    if (explicit_grid) {
        L.ox = gox; L.oy = goy;
        L.nhx = (int)ceilf(gex / L.st);
        L.nhy = (int)ceilf(gey / L.st);
    } else {
        if (!(xmin <= xmax)) { xmin = xmax = ymin = ymax = 0.0f; }
        L.ox = floorf(xmin / res) * res - res;
        L.oy = floorf(ymin / res) * res - res;
        L.nhx = (int)ceilf((xmax - L.ox) / L.st) + 2;
        L.nhy = (int)ceilf((ymax - L.oy) / L.st) + 2;
    }
    L.njx = L.nhx + ov;
    L.njy = L.nhy + ov;
    return L.nhx >= 1 && L.nhy >= 1 && (int64_t)L.njx * L.njy < ((int64_t)1 << 31);
}

// every level of a target's pyramid, for the build kernels (launch_build): blockIdx.y is the level
struct LevelSet {
    LevelDev lv[NDT2D_MAX_LEVELS];
    float4 *cells[NDT2D_MAX_LEVELS];   // the writable record tables (LevelDev::cells is the read-only view)
    // incremental update: per level one word per cell (zero between calls) and the list of the cells touched since the
    // last finalisation; nlist[l] is its length
    unsigned *dirty[NDT2D_MAX_LEVELS];
    unsigned *list[NDT2D_MAX_LEVELS];
    unsigned *nlist;
    int nlevels;
};

// The points a target is built from, as the build kernels read them (SPEC 3, 7.2): map-frame points (pose == nullptr), or
// scans with one pose each, as packed points (xy, offsets) or as LaserScan ranges (ranges, beams; SPEC 8).
struct TargetSrc {
    const float2 *xy;         // map-frame points, or the packed scan points
    int64_t n;                // points; nscans * nbeams beams for ranges
    const double *pose;       // per scan {cos, sin, p0, p1} (launch_pose_table); nullptr: xy are map-frame points
    const int64_t *offsets;   // packed scans: nscans + 1 entries
    int nscans;
    const void *ranges;       // LaserScan ranges: nscans rows of nbeams, f32 or u16
    const float2 *beams;      // (cb, sb) per beam
    int ranges_u16, nbeams;
    float range_scale, range_min, range_max;
};

struct AlignArgs {
    LevelDev lv[NDT2D_MAX_LEVELS];
    int nlevels;
    ndt2d_params prm;
    const float2 *xy;        // packed scans (xy mode)
    const int64_t *offsets;  // nscans+1 (xy mode)
    // ranges mode (SPEC 8): ranges != nullptr
    const void *ranges;
    const float2 *beams;     // (cb, sb) per beam
    int ranges_u16, nbeams;
    float range_scale, range_min, range_max;
    const double *init;
    ndt2d_result *res;
    // optional (xy mode): job j aligns scan job_scan[j] of the packed batch instead of scan j; a negative entry is an empty
    // scan (ndt2d_relocalize: k refinements of ONE scan from k initial poses)
    const int32_t *job_scan;
    // pairs mode (ndt2d_align_pairs): job p aligns scan pairs[2p+1] of the packed batch to the target whose per-level
    // geometry and hash tables are geo[pairs[2p] * nlevels + l]; lv[] is unused
    const int32_t *pairs;
    const LevelDev *geo;
    int nscans;              // jobs: scans, or pairs in pairs mode
    int batch_scans;         // scans of the whole API call when this launch is one chunk of it (0: nscans); kernel selection only
    int cap_points;          // shared-memory slot capacity in points (0: read scans from global memory)
    unsigned int *counter;   // work queue head, zeroed before launch
    int counter_is_zero;     // host side only: the caller guarantees *counter == 0 (no memset in launch_align)
};

struct LaunchCfg {
    int sm_count;
    int max_smem_optin;
    cudaStream_t stream;
    int block_align_max;     // calls with at most this many scans use the block-per-scan align kernel (-1: 8 x SMs)
    int align_help;          // helper warps in k_align (K = 1, staged scans): 0 never, 1 always, -1 up to HELP_MAX_SCANS scans
};

// all launchers return the cudaError_t of the launch; *launches is incremented per kernel launched
// SPEC 3: accumulate the source's points into every level of S and finalise, one accumulate launch (none without points)
// and one finalise launch whatever the number of levels. touch (incremental update): finalise only the cells the points
// touched; S.dirty are zero (and left zero), S.list[l] has room for src.n * (ov ? 4 : 1) cells, S.nlist is zeroed here.
cudaError_t launch_build(const LaunchCfg &c, const LevelSet &S, const ndt2d_params &p, const TargetSrc &src, bool touch, int64_t *launches);
// SPEC 7.2: table[4b..4b+3] = {cos_spec, sin_spec of poses[3b+2], poses[3b], poses[3b+1]} for the posed target sources
cudaError_t launch_pose_table(const LaunchCfg &c, const double *d_poses, int nscans, double *d_table, int64_t *launches);
cudaError_t launch_cell_index(const LaunchCfg &c, const LevelDev &L, const float2 *d_xy, int n, const double *d_pose,
                              int32_t *d_idx, int64_t *launches);
cudaError_t launch_point_terms(const LaunchCfg &c, const LevelDev &L, const float2 *d_xy, int n, const double *d_pose,
                               float *d_terms, int64_t *launches);
// poses: f64 x3 (poses_f32 == 0) or f32 x3 (sweep hypotheses). full: 10 sums, else score only.
cudaError_t launch_eval_poses(const LaunchCfg &c, const LevelDev &L, const float2 *d_xy, int n, const void *d_poses,
                              int poses_f32, int64_t npose, int full, double *d_out, int out_stride, int32_t *d_count,
                              int64_t *launches);
cudaError_t launch_align(const LaunchCfg &c, const AlignArgs &a, int64_t *launches);

// Batched scan-to-scan: one NDT grid per target scan, built by one warp per (target, level) into hash tables.
struct PairBuildArgs {
    const float2 *xy;
    const int64_t *offsets;
    const int32_t *targets;  // scan index of target slot t
    int ntargets, nlevels, ov, explicit_grid;
    float res[NDT2D_MAX_LEVELS];
    float gox, goy, gex, gey;
    int min_points;
    double eig_ratio;
    unsigned cap;            // slots per table (power of two); a table holds cap + 1 records (the last is the sentinel)
    float4 *tab;             // ntargets * nlevels tables
    uint32_t *cnt;           // ntargets * nlevels * cap
    unsigned long long *sums; // ... * 5
    LevelDev *geo;           // out: ntargets * nlevels
    int *error;              // out: set to 1 + slot when a target's lattice would exceed 2^31 cells
};
cudaError_t launch_pairs_build(const LaunchCfg &c, const PairBuildArgs &a, int64_t *launches);

// The submaps of a call over submaps (SPEC 7.3): submap g is members [offsets[g], offsets[g + 1]); member e is points
// [base[e], base[e] + start[e + 1] - start[e]) of the packed batch at pose table entry e. start numbers the points of all
// members in a row, so a submap's points are the flat indices [start[e0], start[e1]) of its members [e0, e1).
struct SubmapDev {
    const int64_t *offsets;  // nsubmaps + 1
    const int64_t *start;    // nmembers + 1
    const int64_t *base;     // nmembers
    const double *pose;      // nmembers * {cos, sin, p0, p1} (launch_pose_table)
};
// One BLOCK per (submap, level) builds the hash table k_pairs_build would build from the submap's posed points: the same
// tables and geometry (a.targets holds submap ids; a.offsets is not read), so k_align and k_search_sweep read them unchanged.
cudaError_t launch_submap_build(const LaunchCfg &c, const PairBuildArgs &a, const SubmapDev &s, int64_t *launches);

// Batched scan-to-scan, fused path (K = 1, scans small enough for shared memory): one warp per PAIR builds the target's
// grid for one pyramid level in its own shared-memory slice (radix sort of the cell keys, one lane per cell for the sums
// and the finalisation, compact record array behind a tagged u32 hash index), aligns the source on it, and goes on to the next
// level - no table ever touches global memory.
struct PairFusedArgs {
    const float2 *xy;
    const int64_t *offsets;
    const int32_t *pairs;    // (target scan, source scan) per pair
    const double *init;
    ndt2d_result *res;
    int npairs, nlevels, explicit_grid;
    float res_m[NDT2D_MAX_LEVELS];
    float gox, goy, gex, gey;
    ndt2d_params prm;
    unsigned cap_t;          // sort capacity in points (longest target, padded to 32)
    unsigned cap_s;          // source slot capacity in points (longest source, padded to 64)
    unsigned rmax;           // record capacity: longest target / min_points
    unsigned hslots;         // u32 entries of the hash index: four per bucket, a power of two of buckets >= 0.7 * rmax
    unsigned off_a, off_r, off_h, warp_bytes;   // byte offsets of the three areas in a warp's slice, and its size
    unsigned warps_per_block;
    unsigned int *counter;   // work queue head, zero on entry
    int *error;              // set to 1 + pair when a target's lattice would exceed 2^31 cells
};
// fills cap_*, rmax, hslots, off_*, warp_bytes; returns false when the fused path cannot be used (smem_optin too small)
bool pairs_fused_layout(PairFusedArgs &a, int64_t max_target_points, int64_t max_source_points, int smem_optin);
cudaError_t launch_pairs_fused(const LaunchCfg &c, const PairFusedArgs &a, int64_t *launches);
size_t align_smem_bytes(int cap_points, bool help = true); // dynamic shared memory per k_align block (help: with the helper-warp desks)
// Publication of a shard's best hypothesis into every rank's exchange table (peer pointers, NVLink stores).
struct PublishArgs {
    ndt2d_best *table[NDT2D_MAX_RANKS]; // table[r] = rank r's table as seen from this device (world entries used)
    int world, rank, row;               // row = query % nslots; world == 0: nothing to publish
    long long index_offset;
    unsigned long long epoch;           // query + 1
};

// Publication of a shard's k refined relocalisation candidates into every rank's table (ndt2d_relocalize_publish)
struct CandidatePublishArgs {
    ndt2d_candidate *table[NDT2D_MAX_RANKS]; // table[r] = this rank's block of the query's row in rank r's table
    int world, k;
    long long index_offset;
    unsigned long long epoch;           // query + 1
};
cudaError_t launch_publish_candidates(const LaunchCfg &c, const int64_t *d_best_idx, const double *d_best_score, const ndt2d_result *d_res,
                                      const CandidatePublishArgs &pub, int64_t *launches);

// top-k of scores by (-score, index); k small. d_work: nhyp bytes of scratch (mask). pub (optional, k == 1): the
// finishing block also stores the winner into the peers' exchange tables.
cudaError_t launch_topk(const LaunchCfg &c, const double *d_scores, int64_t nhyp, int k, int64_t *d_idx, double *d_val,
                        unsigned long long *d_scratch, int64_t *launches, const PublishArgs *pub = nullptr);
int topk_scratch_words(int sm_count);
// refinement jobs of a relocalisation: init[j] = hypothesis best_idx[j] widened to f64, job_scan[j] = 0 (or -1 when best_idx[j] < 0)
cudaError_t launch_topk_to_jobs(const LaunchCfg &c, const float *d_hyp, const int64_t *d_best_idx, int k, double *d_init, int32_t *d_job_scan,
                                int64_t *launches);
// finite bounding box of the target's points (SPEC 2, 7.2): d_box[4] = ordered-int encoded {xmin, ymin, xmax, ymax} (see bbox_decode)
cudaError_t launch_bbox(const LaunchCfg &c, const TargetSrc &src, int *d_box, int64_t *launches);
float bbox_decode(int v);

} // namespace ndt2d
