/*
 * ndt2d.h — C ABI of the B200-native 2D NDT scan matcher (libndt2d.so).
 *
 * Drop-in boundary for the matcher role in a GTSAM/iSAM 2D SLAM pipeline, as named by
 * BASELINE.json `north_star`: "set target map or scan, set cell resolution,
 * align(scan, initial pose) returning pose, score and Hessian".
 *
 * Reference interface replaced: NONE CITABLE. The reference mount holds a single file,
 * /root/reference/README.md:1 ("# GTSAM-NDT"); there is no matcher header, class or signature to
 * bind against (SURVEY.md section 8b). Each entry point below therefore cites the north_star
 * operation it serves and the SPEC.md section that fixes its arithmetic. INTEGRATION.md shows the
 * C++ binding a GTSAM-side maintainer would add.
 *
 * Conventions
 *  - plain pointers and sizes only; no C++ or torch types. All functions return 0 on success or an
 *    NDT2D_E* code; ndt2d_last_error() gives the text. No exceptions cross this boundary.
 *  - "host" pointers are ordinary (pageable or pinned) memory; functions with the _device suffix
 *    take CUDA device pointers on the handle's device and enqueue on the handle's stream without
 *    synchronising (call ndt2d_synchronize, or order your own work on ndt2d_stream()).
 *  - a point is two floats (x, y) in metres; a pose is three doubles (tx, ty, theta);
 *    x' = R(theta) x + t.
 *  - the caller owns every buffer it passes; the library owns all device memory behind the handle.
 *  - one handle = one CUDA device + one stream; a handle is not thread-safe, distinct handles are.
 *  - there is NO CPU fallback: without a CUDA device ndt2d_create fails with NDT2D_ECUDA.
 */
#ifndef NDT2D_H
#define NDT2D_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NDT2D_VERSION 200      /* 200: SPEC.md v4 (f64 point-to-cell geometry, cell-local records) */
#define NDT2D_MAX_LEVELS 8

enum {
    NDT2D_OK = 0,
    NDT2D_EINVAL = 1,   /* bad argument */
    NDT2D_ECUDA = 2,    /* CUDA runtime error (no device, launch failure, ...) */
    NDT2D_ENOTARGET = 3,/* align/evaluate/sweep before set_target */
    NDT2D_ENOMEM = 4,
    NDT2D_ETIMEOUT = 5  /* ndt2d_exchange_wait: a rank did not publish in time */
};

/* align status, SPEC.md section 5 */
enum {
    NDT2D_CONVERGED = 0,
    NDT2D_MAX_ITERATIONS = 1,
    NDT2D_STALLED = 2,
    NDT2D_NO_OVERLAP = 3
};

/* SPEC.md section 1 */
typedef struct ndt2d_params {
    double eig_ratio;       /* [0.01]  smaller covariance eigenvalue >= eig_ratio * larger */
    double eps_trans;       /* [1e-4]  m   */
    double eps_rot;         /* [1e-5]  rad */
    double max_step_trans;  /* [0.5]   m   */
    double max_step_rot;    /* [0.2]   rad */
    double lambda_init;     /* [1e-3] */
    double lambda_min;      /* [1e-9] */
    double lambda_max;      /* [1e7]  */
    double lambda_up;       /* [10]   */
    double lambda_down;     /* [5]    */
    double lambda_fail_up;  /* [3]    */
    int32_t min_points;     /* [3]  */
    int32_t max_iterations; /* [30] evaluations per pyramid level */
    int32_t overlap;        /* [0]  0: K = 1 cell per point; 1: four half-shifted grids, K = 4 */
    int32_t reserved;
} ndt2d_params;

/* what align returns: pose, score and Hessian (north_star), plus gradient and diagnostics */
typedef struct ndt2d_result {
    double pose[3];     /* tx, ty, theta in (-pi, pi] */
    double score;       /* S = sum of Gaussian likelihoods, higher is better */
    double grad[3];     /* gradient of f = -S at pose */
    double hessian[9];  /* Hessian of f = -S at pose, row-major 3x3, symmetric */
    int32_t iterations; /* evaluations used, all levels */
    int32_t status;     /* NDT2D_CONVERGED ... */
    int32_t count;      /* (point, cell) pairs that contributed at pose */
    int32_t reserved;
} ndt2d_result;

typedef struct ndt2d_matcher ndt2d_matcher;

/* ---- lifecycle ------------------------------------------------------------------------------ */
int ndt2d_version(void);
/* device: CUDA ordinal. The handle creates its own non-blocking stream. */
int ndt2d_create(int device, ndt2d_matcher **out);
/* same, but enqueue on the caller's cudaStream_t (passed as void*; NULL = default stream) */
int ndt2d_create_on_stream(int device, void *cuda_stream, ndt2d_matcher **out);
void ndt2d_destroy(ndt2d_matcher *m);
/* text of the last error on this handle (m == NULL: last ndt2d_create error in this thread) */
const char *ndt2d_last_error(const ndt2d_matcher *m);
void *ndt2d_stream(const ndt2d_matcher *m);
int ndt2d_synchronize(ndt2d_matcher *m);
/* number of this library's kernels launched through this handle so far */
int64_t ndt2d_kernel_launches(const ndt2d_matcher *m);

/* ---- configuration (north_star: "set cell resolution") -------------------------------------- */
void ndt2d_default_params(ndt2d_params *p);
int ndt2d_set_params(ndt2d_matcher *m, const ndt2d_params *p);
int ndt2d_get_params(const ndt2d_matcher *m, ndt2d_params *p);
/* one level of cell size `res` metres (SPEC 2). Drops the current target. */
int ndt2d_set_resolution(ndt2d_matcher *m, float res);
/* multi-resolution pyramid, coarse to fine (BASELINE.json configs[2]: 2.0/1.0/0.5 m) */
int ndt2d_set_resolutions(ndt2d_matcher *m, const float *res, int nlevels);
/* explicit lattice origin/extent in metres for every level; extent <= 0 restores auto-fit (SPEC 2) */
int ndt2d_set_grid(ndt2d_matcher *m, float ox, float oy, float extent_x, float extent_y);

/* ---- target (north_star: "set target map or scan"; kernel stage 1, SPEC 3) -------------------- */
int ndt2d_set_target(ndt2d_matcher *m, const float *xy, int64_t n);
int ndt2d_set_target_device(ndt2d_matcher *m, const float *d_xy, int64_t n);
/* incremental update (SPEC 7): same cells as a rebuild from the union. Needs an explicit grid
 * or points inside the current lattice; points outside are ignored. */
int ndt2d_add_target(ndt2d_matcher *m, const float *xy, int64_t n);
int ndt2d_add_target_device(ndt2d_matcher *m, const float *d_xy, int64_t n);
/* target from posed scans (SPEC 7.2): scan b, with pose poses[3b..3b+2] (f64 tx, ty, theta), is transformed into the map
 * frame in f64 inside the build, never rounded to f32. Packed points: offsets[0..nscans] index xy (offsets[0] = 0,
 * non-decreasing). LaserScan: nscans rows of nbeams ranges, beams kept as in ndt2d_align_batch_ranges (SPEC 8). With
 * identity poses the target equals ndt2d_set_target of the concatenated points bit for bit; add equals one set from all
 * the scans (SPEC 7). The host forms refuse (NDT2D_EINVAL, target untouched) a non-finite pose, nscans < 0, bad offsets
 * and nbeams < 1, and return after the build; the device forms check no array contents and are asynchronous on the
 * handle's stream, except that an auto-fitted set reads its bounding box back once. A device offsets table must also end
 * at npoints; a malformed one gives an unspecified target but no access outside the arrays. Add onto a target loaded
 * with ndt2d_set_cells is refused; add without a target is set. */
int ndt2d_set_target_scans(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const double *poses);
int ndt2d_add_target_scans(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const double *poses);
int ndt2d_set_target_scans_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, int nscans, int64_t npoints,
                                  const double *d_poses);
int ndt2d_add_target_scans_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, int nscans, int64_t npoints,
                                  const double *d_poses);
int ndt2d_set_target_ranges(ndt2d_matcher *m, const void *ranges, int ranges_are_u16, int nscans, int nbeams, double angle_min,
                            double angle_inc, float range_scale, float range_min, float range_max, const double *poses);
int ndt2d_add_target_ranges(ndt2d_matcher *m, const void *ranges, int ranges_are_u16, int nscans, int nbeams, double angle_min,
                            double angle_inc, float range_scale, float range_min, float range_max, const double *poses);
int ndt2d_set_target_ranges_device(ndt2d_matcher *m, const void *d_ranges, int ranges_are_u16, int nscans, int nbeams,
                                   double angle_min, double angle_inc, float range_scale, float range_min, float range_max,
                                   const double *d_poses);
int ndt2d_add_target_ranges_device(ndt2d_matcher *m, const void *d_ranges, int ranges_are_u16, int nscans, int nbeams,
                                   double angle_min, double angle_inc, float range_scale, float range_min, float range_max,
                                   const double *d_poses);
/* geom = {res, st, inv_st, ox, oy}; dims = {nhx, nhy, njx, njy} */
int ndt2d_level_geometry(const ndt2d_matcher *m, int level, float geom[5], int32_t dims[4]);
/* cell table: njx*njy records of 8 floats {mux, muy, B00, B01, B01, B11, n, valid}; (mux, muy) is the mean RELATIVE TO THE
 * CELL CENTRE ox + (jx - ov) * st + res / 2 (SPEC.md section 3, v4) */
int ndt2d_get_cells(ndt2d_matcher *m, int level, float *cells);
/* raw accumulators: n[njx*njy] and sums[njx*njy*5] = {sx, sy, sxx, sxy, syy} about the cell centre, in res * 2^-22 m units */
int ndt2d_get_sums(ndt2d_matcher *m, int level, uint32_t *n, int64_t *sums);
/* device pointer to the cell table of a level (valid until the target changes) */
const float *ndt2d_cells_device(const ndt2d_matcher *m, int level);
/* load a cell table computed elsewhere (e.g. saved by ndt2d_get_cells); geometry must be explicit (ndt2d_set_grid) or
 * already present; nrecords must equal the level's njx*njy. The target then has no sums (ndt2d_add_target is refused). */
int ndt2d_set_cells(ndt2d_matcher *m, int level, const float *cells, int64_t nrecords);
/* map files (SURVEY.md 8(f) rank 4): every level's lattice exactly as built (auto-fitted or explicit), the parameters that
 * shaped the cells (overlap, min_points, eig_ratio), the cell records and - with_sums != 0 - the integer sums, so that
 * ndt2d_add_target continues a loaded map bit for bit. Versioned binary file ("NDT2DMAP"); ndt2d_load_map replaces the
 * handle's resolutions, grid, those three parameters and the target. */
int ndt2d_save_map(ndt2d_matcher *m, const char *path, int with_sums);
int ndt2d_load_map(ndt2d_matcher *m, const char *path);

/* ---- evaluation (kernel stage 2, the Newton-step unit of work, SPEC 2 and 4) ------------------ */
/* lattice index hy*nhx+hx (or -1) of each point after the optional pose (NULL = none) */
int ndt2d_cell_index(ndt2d_matcher *m, int level, const float *xy, int n, const double *pose, int32_t *idx);
/* out[10*j..] = {S, g0,g1,g2, H00,H01,H02,H11,H12,H22} and count[j] for pose j of npose */
int ndt2d_evaluate(ndt2d_matcher *m, int level, const float *xy, int n, const double *poses, int npose,
                   double *out, int32_t *count);
int ndt2d_evaluate_device(ndt2d_matcher *m, int level, const float *d_xy, int n, const double *d_poses,
                          int npose, double *d_out, int32_t *d_count);
/* the ten f32 factors (e, c1..c9; SPEC 4) of every (point, cell) pair: terms[n*K*10], zeros where skipped (tests) */
int ndt2d_point_terms(ndt2d_matcher *m, int level, const float *xy, int n, const double *pose, float *terms);

/* ---- align (north_star: "align(scan, initial pose) returning pose, score and Hessian", SPEC 5) - */
int ndt2d_align(ndt2d_matcher *m, const float *xy, int n, const double init[3], ndt2d_result *res);
/* independent scans in one launch: scan b is points offsets[b] .. offsets[b+1]-1 of xy */
int ndt2d_align_batch(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans,
                      const double *init, ndt2d_result *res);
/* all-device variant; max_points >= longest scan (sizes the shared-memory staging) */
int ndt2d_align_batch_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, int nscans,
                             int max_points, const double *d_init, ndt2d_result *d_res);
/* LaserScan input (SPEC 8): ranges[nscans*nbeams], f32 metres or u16 * range_scale; beams outside
 * [range_min, range_max] (and u16 zeros) are dropped on the device */
int ndt2d_align_batch_ranges(ndt2d_matcher *m, const void *ranges, int ranges_are_u16, int nscans, int nbeams,
                             double angle_min, double angle_inc, float range_scale, float range_min,
                             float range_max, const double *init, ndt2d_result *res);
int ndt2d_align_batch_ranges_device(ndt2d_matcher *m, const void *d_ranges, int ranges_are_u16, int nscans,
                                    int nbeams, double angle_min, double angle_inc, float range_scale,
                                    float range_min, float range_max, const double *d_init,
                                    ndt2d_result *d_res);

/* ---- batched scan-to-scan (kernel stage 3, "batched multi-scan": odometry over a log, loop-closure candidates) ----
 * All scans are packed as for ndt2d_align_batch (xy + offsets[nscans+1]). Pair p aligns scan pairs[2p+1] (source) to
 * scan pairs[2p] (target) from init[3p..]: the result equals ndt2d_set_target(target scan) followed by
 * ndt2d_align(source scan, init) bit for bit (same lattice - auto-fitted per target, or the ndt2d_set_grid one - same
 * cells, same LM loop), but every target's grid is built once, by one warp, into a per-target hash table, and all pairs
 * are aligned by one launch. Needs ndt2d_set_resolution(s) only; the handle's own target is not touched.
 * Target scans are limited to 43 690 points (10 922 with overlapping grids). */
int ndt2d_align_pairs(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const int32_t *pairs,
                      int npairs, const double *init, ndt2d_result *res);
/* scans, initial poses and results on the device; offsets (also given on the host) and pairs on the host, because
 * the list of distinct targets and the chunking are host work. Asynchronous on the handle's stream. */
int ndt2d_align_pairs_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, const int64_t *offsets,
                             int nscans, const int32_t *pairs, int npairs, const double *d_init, ndt2d_result *d_res);

/* ---- windowed search over scan pairs (loop-closure candidates, SPEC 6.1) ----
 * A search window is H = (2nx+1)(2ny+1)(2nth+1) hypotheses around a centre pose c: hypothesis
 * j = ((ix+nx)(2ny+1) + (iy+ny))(2nth+1) + (it+nth) is ((float)(c0 + ix*step_x), (float)(c1 + iy*step_y),
 * (float)(c2 + it*step_th)) in f64 without contraction, theta not wrapped. nx, ny, nth >= 0, steps finite, reserved = 0,
 * H < 2^31. */
typedef struct ndt2d_window {
    int32_t nx, ny, nth, reserved;
    double step_x, step_y, step_th;
} ndt2d_window;
/* Scans packed as for ndt2d_align_pairs. Pair p = (target scan pairs[2p], source scan pairs[2p+1]) with centre
 * centres[3p..]: best_idx[p*k..], best_score[p*k..] and res[p*k..] equal, bit for bit, ndt2d_set_target(target scan) followed
 * by ndt2d_relocalize(level, source scan, the window's hypotheses around the centre, k) (best_score: ndt2d_sweep's top-k
 * scores). A slot without a candidate (H < k) has index -1, score 0 and an all-zero record with status NDT2D_NO_OVERLAP.
 * 1 <= k <= 32; best_score may be NULL. Needs ndt2d_set_resolution(s) only; the handle's own target is not touched. */
int ndt2d_relocalize_pairs(ndt2d_matcher *m, int level, const float *xy, const int64_t *offsets, int nscans,
                           const int32_t *pairs, int npairs, const double *centres, const ndt2d_window *win, int k,
                           int64_t *best_idx, double *best_score, ndt2d_result *res);
/* scans, centres and outputs on the device; offsets (also given on the host), pairs and the window on the host, as for
 * ndt2d_align_pairs_device. Asynchronous on the handle's stream. */
int ndt2d_relocalize_pairs_device(ndt2d_matcher *m, int level, const float *d_xy, const int64_t *d_offsets,
                                  const int64_t *offsets, int nscans, const int32_t *pairs, int npairs,
                                  const double *d_centres, const ndt2d_window *win, int k, int64_t *d_best_idx,
                                  double *d_best_score, ndt2d_result *d_res);

/* ---- pairs against submaps of posed scans (local submaps of keyframes for loop closure, SPEC 7.3) ----
 * Scans packed as for ndt2d_align_pairs. Submap g is members e in [submap_offsets[g], submap_offsets[g+1])
 * (submap_offsets[0] = 0, non-decreasing); member e is scan member_scans[e] at f64 pose member_poses[3e..3e+2]. Its target
 * is that of ndt2d_set_target_scans of the member scans at those poses (SPEC 7.2); a scan may be a member of several
 * submaps, at different poses, and a submap without members has an empty target. Pair p = (submap pairs[2p], source scan
 * pairs[2p+1]):
 *   ndt2d_align_submaps: res[p] equals ndt2d_set_target_scans(members) + ndt2d_align(source, init[3p..]) bit for bit;
 *   ndt2d_relocalize_submaps: best_idx / best_score / res[p*k..] equal ndt2d_set_target_scans(members) +
 *   ndt2d_relocalize(level, source, the window's hypotheses around centres[3p..], k), as for ndt2d_relocalize_pairs.
 * With the members expressed relative to an anchor keyframe, the result is the source's pose in the anchor's frame.
 * Submaps a pair names are limited to 43 690 points in all (10 922 with overlapping grids). Refused with NDT2D_EINVAL:
 * bad submap offsets, a member, source or submap index out of range, a non-finite member pose (host forms), an oversized
 * submap. A submap whose auto-fitted lattice exceeds 2^31 cells is reported after the call; its pairs end NO_OVERLAP.
 * The handle's own target is not touched. Device forms: scans, member poses, initial poses / centres and outputs on the
 * device; offsets (also given on the host), submap offsets, member scans, pairs and the window on the host, since the
 * target list and the chunking are host work. Asynchronous on the handle's stream. */
int ndt2d_align_submaps(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const int64_t *submap_offsets,
                        int nsubmaps, const int32_t *member_scans, const double *member_poses, const int32_t *pairs, int npairs,
                        const double *init, ndt2d_result *res);
int ndt2d_align_submaps_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, const int64_t *offsets, int nscans,
                               const int64_t *submap_offsets, int nsubmaps, const int32_t *member_scans, const double *d_member_poses,
                               const int32_t *pairs, int npairs, const double *d_init, ndt2d_result *d_res);
int ndt2d_relocalize_submaps(ndt2d_matcher *m, int level, const float *xy, const int64_t *offsets, int nscans,
                             const int64_t *submap_offsets, int nsubmaps, const int32_t *member_scans, const double *member_poses,
                             const int32_t *pairs, int npairs, const double *centres, const ndt2d_window *win, int k,
                             int64_t *best_idx, double *best_score, ndt2d_result *res);
int ndt2d_relocalize_submaps_device(ndt2d_matcher *m, int level, const float *d_xy, const int64_t *d_offsets,
                                    const int64_t *offsets, int nscans, const int64_t *submap_offsets, int nsubmaps,
                                    const int32_t *member_scans, const double *d_member_poses, const int32_t *pairs, int npairs,
                                    const double *d_centres, const ndt2d_window *win, int k, int64_t *d_best_idx,
                                    double *d_best_score, ndt2d_result *d_res);

/* ---- windowed search of a batch of scans against the handle's target (relocalisation in a known map, SPEC 6.2) ----
 * Scans packed as for ndt2d_align_batch. Scan b with centre centres[3b..]: best_idx[b*k..], best_score[b*k..] and
 * res[b*k..] equal, bit for bit, ndt2d_relocalize(level, scan b, the window's hypotheses around the centre, k) on this
 * handle (best_score: ndt2d_sweep's top-k scores). A slot without a candidate (H < k) has index -1, score 0 and an
 * all-zero record with status NDT2D_NO_OVERLAP. 1 <= k <= 32, nscans * k < 2^31; best_score may be NULL. Needs a
 * target; the target, the parameters and other results are not touched. One synchronisation. */
int ndt2d_relocalize_batch(ndt2d_matcher *m, int level, const float *xy, const int64_t *offsets, int nscans,
                           const double *centres, const ndt2d_window *win, int k, int64_t *best_idx,
                           double *best_score, ndt2d_result *res);
/* scans, offsets, centres and outputs on the device, the window on the host; max_points >= longest scan (sizes the
 * shared-memory staging, as for ndt2d_align_batch_device). Asynchronous on the handle's stream, reads nothing back. */
int ndt2d_relocalize_batch_device(ndt2d_matcher *m, int level, const float *d_xy, const int64_t *d_offsets, int nscans,
                                  int max_points, const double *d_centres, const ndt2d_window *win, int k,
                                  int64_t *d_best_idx, double *d_best_score, ndt2d_result *d_res);

/* ---- sweep (kernel stage 3: multi-hypothesis search for relocalisation / loop closure, SPEC 6) - */
/* hyp[3*j..] = (tx, ty, theta) f32. scores (optional, nhyp doubles). Top-k (k >= 1) by
 * (-score, index) into best_idx[k], best_score[k]. */
int ndt2d_sweep(ndt2d_matcher *m, int level, const float *xy, int n, const float *hyp, int64_t nhyp,
                double *scores, int k, int64_t *best_idx, double *best_score);
int ndt2d_sweep_device(ndt2d_matcher *m, int level, const float *d_xy, int n, const float *d_hyp,
                       int64_t nhyp, double *d_scores, int k, int64_t *d_best_idx, double *d_best_score);
/* sweep, then full align from each of the k best hypotheses; res[k] sorted like the top-k */
int ndt2d_relocalize(ndt2d_matcher *m, int level, const float *xy, int n, const float *hyp, int64_t nhyp,
                     int k, int64_t *best_idx, ndt2d_result *res);
/* the same with scan, hypotheses, indices and results on the device; asynchronous on the handle's stream (sweep, top-k and
 * the k refinements are queued back to back: the scan is not replicated and nothing returns to the host in between).
 * Entries with d_best_idx[j] < 0 (fewer than k hypotheses) hold an empty-scan result with status NDT2D_NO_OVERLAP. */
int ndt2d_relocalize_device(ndt2d_matcher *m, int level, const float *d_xy, int n, const float *d_hyp, int64_t nhyp,
                            int k, int64_t *d_best_idx, ndt2d_result *d_res);

/* ---- multi-GPU sweep: best-hypothesis exchange over peer memory (north_star: "independent ... pose
 *      hypotheses are split per GPU", only the best-hypothesis scores are combined) --------------
 * One process per GPU. Each rank owns a table of nslots x world records; the last block of the
 * arg-max kernel of a sharded sweep stores this rank's best {index, score, query + 1} straight into
 * row (query % nslots), column rank of EVERY rank's table (NVLink peer stores from inside the kernel:
 * the combine is part of the sweep launch, there is no separate collective). Reading the result is a
 * host-side poll of the caller's own table: nothing ever spins on the device.
 * Reference interface replaced: none citable (/root/reference/README.md:1 is the whole mount). */
#define NDT2D_IPC_HANDLE_BYTES 64
#define NDT2D_MAX_RANKS 16
typedef struct ndt2d_best {
    int64_t index;      /* global hypothesis index, -1 when the shard was empty */
    double score;
    uint64_t epoch;     /* query + 1; written last */
    uint64_t reserved;
} ndt2d_best;

/* allocate this rank's table and return its CUDA IPC handle (64 bytes) for the other ranks */
int ndt2d_exchange_create(ndt2d_matcher *m, int world, int rank, int nslots, unsigned char *handle);
/* handles = world x 64 bytes, entry r from rank r (the own entry is ignored); opens the peers' tables */
int ndt2d_exchange_open(ndt2d_matcher *m, const unsigned char *handles);
/* sweep of this rank's shard + top-1 + publication, asynchronous on the handle's stream. Hypothesis j of
 * the shard has global index index_offset + j. d_scores may be NULL. Slot discipline: row query % nslots is
 * overwritten by query + nslots, so a rank must have waited for query q - nslots/2 (or a later one) before it
 * publishes q; then no rank can overwrite a row another rank is still waiting on. */
int ndt2d_sweep_publish(ndt2d_matcher *m, int level, const float *d_xy, int n, const float *d_hyp,
                        int64_t nhyp, double *d_scores, int64_t index_offset, uint64_t query);
/* block until every rank has published `query` (or timeout_ms elapsed: NDT2D_ETIMEOUT), then return the
 * best hypothesis by (-score, index), as an unsharded ndt2d_sweep would (SPEC.md section 6) */
int ndt2d_exchange_wait(ndt2d_matcher *m, uint64_t query, int timeout_ms, int64_t *best_index, double *best_score);
/* frees the own table and closes the peers'. Synchronise the ranks first: a peer must not publish afterwards. */
int ndt2d_exchange_close(ndt2d_matcher *m);

/* ---- multi-GPU relocalisation end to end over peer memory ---------------------------------------------------------
 * Every rank sweeps its shard of the hypotheses, refines ITS OWN k best (sweep, top-k and the k aligns are queued on the
 * stream: ndt2d_relocalize_device) and stores the k candidates {global index, sweep score, refined record} into every
 * rank's table with one more small kernel. Every member of the global top-k is among its own shard's k best, so the
 * global answer - what ndt2d_relocalize returns on one GPU for the whole hypothesis set, bit for bit - is a local merge of
 * the world x k candidates: ONE exchange per query and no collective. Slots, handles and the wait follow the
 * best-hypothesis exchange above (same slot discipline). */
typedef struct ndt2d_candidate {
    int64_t index;          /* global hypothesis index, -1: the shard had fewer than k hypotheses */
    double sweep_score;
    uint64_t epoch;         /* of candidate 0 of a rank's block: query + 1, written last */
    uint64_t reserved;
    ndt2d_result refined;   /* the full align from that hypothesis */
} ndt2d_candidate;
int ndt2d_reloc_create(ndt2d_matcher *m, int world, int rank, int nslots, int kmax, unsigned char *handle);
int ndt2d_reloc_open(ndt2d_matcher *m, const unsigned char *handles);
/* asynchronous; hypothesis j of the shard has global index index_offset + j; 1 <= k <= kmax */
int ndt2d_relocalize_publish(ndt2d_matcher *m, int level, const float *d_xy, int n, const float *d_hyp, int64_t nhyp,
                             int64_t index_offset, int k, uint64_t query);
/* blocks until every rank has published `query`; best_idx[k], res[k] ordered like ndt2d_relocalize's */
int ndt2d_relocalize_wait(ndt2d_matcher *m, uint64_t query, int timeout_ms, int k, int64_t *best_idx, ndt2d_result *res);
int ndt2d_reloc_close(ndt2d_matcher *m);

/* ---- pinned host memory for callers that want full-speed copies ------------------------------ */
int ndt2d_host_alloc(void **p, size_t bytes);
/* flags: NDT2D_HOST_WRITE_COMBINED for buffers the CPU only writes (scan input): the copy engine reads them without
 * snooping the CPU caches; CPU reads from such memory are very slow */
#define NDT2D_HOST_WRITE_COMBINED 1
int ndt2d_host_alloc_flags(void **p, size_t bytes, int flags);
int ndt2d_host_free(void *p);

/* Upload relay for the host-buffer batch calls (ndt2d_align_batch, ndt2d_align_batch_ranges). On a multi-GPU box the host
 * side often cannot feed every GPU's PCIe link at once (measured on an 8 x B200 node: four GPUs get 23 GB/s each, the
 * other four 35 GB/s, one GPU alone 50-55 GB/s). With a relay, about `fraction` of a call's input chunks are copied
 * host -> relay_device (that GPU's link) and from there to this handle's device by a peer copy over NVLink, while the rest
 * takes the handle's own link; results are unchanged. relay_device must differ from the handle's device and be
 * peer-accessible; it needs no handle of its own and may serve a handle of another process at the same time. fraction
 * in (0, 1); relay_device < 0 switches the relay off. No reference counterpart (SURVEY.md 8b: none citable). */
int ndt2d_set_upload_relay(ndt2d_matcher *m, int relay_device, double fraction);

#ifdef __cplusplus
}
#endif
#endif /* NDT2D_H */
