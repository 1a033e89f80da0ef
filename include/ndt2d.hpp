// ndt2d.hpp — header-only C++ host mirror of the matcher interface, over the C ABI in ndt2d.h.
//
// This is the class a GTSAM-NDT style C++ front end holds in place of its CPU matcher: set the target map or
// scan, set the cell resolution, align(scan, initial pose) -> pose, score, Hessian (BASELINE.json north_star).
// Reference class/signature replaced: none citable — the reference mount is /root/reference/README.md:1 only
// (SURVEY.md 8b), so the method names follow the north_star's wording. INTEGRATION.md shows the GTSAM glue.
//
// Error behaviour: every failure of the C ABI becomes a std::runtime_error carrying ndt2d_last_error().
// There is no CPU fallback: constructing a Matcher without a B200-class CUDA device throws.
#ifndef NDT2D_HPP
#define NDT2D_HPP

#include <array>
#include <cmath>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "ndt2d.h"

namespace ndt2d {

struct Point2f {
    float x, y;
};

struct Pose2d {
    double x = 0, y = 0, theta = 0;
};

// A submap of posed scans (SPEC 7.3): member i is scan scans[i] of a packed batch at poses[i], e.g. a keyframe and its graph
// neighbours at their current estimates, relative to an anchor keyframe
struct Submap {
    std::vector<std::int32_t> scans;
    std::vector<Pose2d> poses;
};

using Result = ndt2d_result;   // pose[3], score, grad[3], hessian[9] (row-major), iterations, status, count
using Params = ndt2d_params;

// The Hessian align() returns is taken with respect to increments (dtx, dty, dtheta) of the pose IN THE TARGET FRAME
// (x' = R(theta) x + t). Pose-graph back ends (gtsam::BetweenFactor<Pose2>, g2o EDGE_SE2) express the translation error
// of a relative-pose measurement in the measurement's own (local) frame, dt_target = R(theta) dt_local, so the information
// matrix of such a factor is J^T H J with J = blockdiag(R(theta), 1). Writes the symmetrised 3x3 result, row-major.
// (For odometry theta is small and the two nearly coincide; for loop closures at large relative rotation they do not.)
inline void informationInLocalFrame(const ndt2d_result &r, double info[9])
{
    const double c = std::cos(r.pose[2]), s = std::sin(r.pose[2]);
    const double J[3][3] = {{c, -s, 0.0}, {s, c, 0.0}, {0.0, 0.0, 1.0}};
    double H[3][3], T[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) H[i][j] = 0.5 * (r.hessian[3 * i + j] + r.hessian[3 * j + i]);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) T[i][j] = H[i][0] * J[0][j] + H[i][1] * J[1][j] + H[i][2] * J[2][j];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) info[3 * i + j] = J[0][i] * T[0][j] + J[1][i] * T[1][j] + J[2][i] * T[2][j];
}

class Matcher {
  public:
    explicit Matcher(int device = 0, void *cuda_stream = reinterpret_cast<void *>(-1))
    {
        int rc = cuda_stream == reinterpret_cast<void *>(-1) ? ndt2d_create(device, &h_)
                                                             : ndt2d_create_on_stream(device, cuda_stream, &h_);
        if (rc != NDT2D_OK) throw std::runtime_error(std::string("ndt2d_create: ") + ndt2d_last_error(nullptr));
    }
    ~Matcher() { ndt2d_destroy(h_); }
    Matcher(const Matcher &) = delete;
    Matcher &operator=(const Matcher &) = delete;
    Matcher(Matcher &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    Matcher &operator=(Matcher &&o) noexcept
    {
        if (this != &o) {
            ndt2d_destroy(h_);
            h_ = o.h_;
            o.h_ = nullptr;
        }
        return *this;
    }

    // ---- configuration ------------------------------------------------------------------------
    Params params() const
    {
        Params p;
        ck(ndt2d_get_params(h_, &p));
        return p;
    }
    void setParams(const Params &p) { ck(ndt2d_set_params(h_, &p)); }
    void setResolution(float res) { ck(ndt2d_set_resolution(h_, res)); }
    void setResolutions(const std::vector<float> &coarse_to_fine)
    {
        ck(ndt2d_set_resolutions(h_, coarse_to_fine.data(), static_cast<int>(coarse_to_fine.size())));
    }
    void setGrid(float ox, float oy, float extent_x, float extent_y) { ck(ndt2d_set_grid(h_, ox, oy, extent_x, extent_y)); }

    // ---- target: a previous scan (scan-to-scan) or a map point cloud (scan-to-map) ---------------
    void setTarget(const Point2f *pts, std::int64_t n) { ck(ndt2d_set_target(h_, reinterpret_cast<const float *>(pts), n)); }
    void setTarget(const std::vector<Point2f> &pts) { setTarget(pts.data(), static_cast<std::int64_t>(pts.size())); }
    void addToTarget(const Point2f *pts, std::int64_t n) { ck(ndt2d_add_target(h_, reinterpret_cast<const float *>(pts), n)); }
    void addToTarget(const std::vector<Point2f> &pts) { addToTarget(pts.data(), static_cast<std::int64_t>(pts.size())); }

    // target from posed scans (keyframes at their optimised poses): scan b is points [offsets[b], offsets[b+1]) at poses[b],
    // transformed into the map frame in f64 inside the build; addScansToTarget equals one setTargetScans of all scans so far
    void setTargetScans(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets, const std::vector<Pose2d> &poses)
    {
        targetScans(points, offsets, poses, false);
    }
    void addScansToTarget(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets, const std::vector<Pose2d> &poses)
    {
        targetScans(points, offsets, poses, true);
    }
    // the same from LaserScan ranges[nscans * nbeams] in metres, beam i at angle_min + i * angle_inc, scan b at poses[b]
    void setTargetRanges(const std::vector<float> &ranges, int nbeams, double angle_min, double angle_inc, float range_min,
                         float range_max, const std::vector<Pose2d> &poses)
    {
        targetRanges(ranges, nbeams, angle_min, angle_inc, range_min, range_max, poses, false);
    }
    void addRangesToTarget(const std::vector<float> &ranges, int nbeams, double angle_min, double angle_inc, float range_min,
                           float range_max, const std::vector<Pose2d> &poses)
    {
        targetRanges(ranges, nbeams, angle_min, angle_inc, range_min, range_max, poses, true);
    }

    // map files: every level's lattice, the cell records and (withSums) the integer sums behind them, so that addToTarget
    // continues a loaded map bit for bit; loadMap replaces the resolutions, the grid and the target of this matcher
    void saveMap(const std::string &path, bool withSums = true) { ck(ndt2d_save_map(h_, path.c_str(), withSums ? 1 : 0)); }
    void loadMap(const std::string &path) { ck(ndt2d_load_map(h_, path.c_str())); }

    // ---- align(scan, initial pose) -> pose, score, Hessian -----------------------------------------
    Result align(const Point2f *scan, int n, const Pose2d &init)
    {
        const double p[3] = {init.x, init.y, init.theta};
        Result r;
        ck(ndt2d_align(h_, reinterpret_cast<const float *>(scan), n, p, &r));
        return r;
    }
    Result align(const std::vector<Point2f> &scan, const Pose2d &init) { return align(scan.data(), static_cast<int>(scan.size()), init); }

    // independent scans in one launch; scan b is points [offsets[b], offsets[b+1]) of `points`
    std::vector<Result> alignBatch(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets,
                                   const std::vector<Pose2d> &init)
    {
        const int nb = static_cast<int>(init.size());
        if (offsets.size() != init.size() + 1) throw std::invalid_argument("alignBatch: offsets.size() must be init.size() + 1");
        if (offsets.front() < 0 || static_cast<size_t>(offsets.back()) > points.size()) throw std::invalid_argument("alignBatch: offsets overrun points");
        std::vector<Result> out(init.size());
        static_assert(sizeof(Pose2d) == 3 * sizeof(double), "Pose2d must be three packed doubles");
        ck(ndt2d_align_batch(h_, reinterpret_cast<const float *>(points.data()), offsets.data(), nb,
                             reinterpret_cast<const double *>(init.data()), out.data()));
        return out;
    }

    // LaserScan input: ranges[nscans * nbeams] in metres, beam i at angle_min + i * angle_inc
    std::vector<Result> alignBatchRanges(const std::vector<float> &ranges, int nbeams, double angle_min, double angle_inc,
                                         float range_min, float range_max, const std::vector<Pose2d> &init)
    {
        if (nbeams < 1 || ranges.size() != init.size() * static_cast<size_t>(nbeams))
            throw std::invalid_argument("alignBatchRanges: ranges.size() must be init.size() * nbeams");
        std::vector<Result> out(init.size());
        ck(ndt2d_align_batch_ranges(h_, ranges.data(), 0, static_cast<int>(init.size()), nbeams, angle_min, angle_inc, 1.0f,
                                    range_min, range_max, reinterpret_cast<const double *>(init.data()), out.data()));
        return out;
    }

    // batched scan-to-scan: pair p aligns scan pairs[p].second (source) to scan pairs[p].first (target) of the packed batch;
    // equals setTarget(target) + align(source, init[p]) for every pair, with all grids built and all pairs aligned in one call
    std::vector<Result> alignPairs(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets,
                                   const std::vector<std::pair<std::int32_t, std::int32_t>> &pairs, const std::vector<Pose2d> &init)
    {
        if (pairs.size() != init.size()) throw std::invalid_argument("alignPairs: one initial pose per pair");
        if (offsets.empty()) throw std::invalid_argument("alignPairs: offsets must have nscans + 1 entries");
        if (offsets.front() < 0 || static_cast<size_t>(offsets.back()) > points.size()) throw std::invalid_argument("alignPairs: offsets overrun points");
        static_assert(sizeof(std::pair<std::int32_t, std::int32_t>) == 2 * sizeof(std::int32_t), "pairs must be packed int32 pairs");
        std::vector<Result> out(pairs.size());
        ck(ndt2d_align_pairs(h_, reinterpret_cast<const float *>(points.data()), offsets.data(), static_cast<int>(offsets.size() - 1),
                             reinterpret_cast<const std::int32_t *>(pairs.data()), static_cast<int>(pairs.size()),
                             reinterpret_cast<const double *>(init.data()), out.data()));
        return out;
    }

    // windowed search over scan pairs (loop-closure candidates): for every pair, the window's hypotheses around centres[p] are
    // swept on `level`, the k best refined; equals setTarget(target) + relocalize(source, window hypotheses, k, level) per pair.
    // Returns npairs * k records, pair-major; indices / scores (optional) receive the k sweep indices and scores per pair
    // (index -1: no candidate).
    std::vector<Result> relocalizePairs(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets,
                                        const std::vector<std::pair<std::int32_t, std::int32_t>> &pairs, const std::vector<Pose2d> &centres,
                                        const ndt2d_window &window, int k, int level = 0, std::vector<std::int64_t> *indices = nullptr,
                                        std::vector<double> *scores = nullptr)
    {
        if (pairs.size() != centres.size()) throw std::invalid_argument("relocalizePairs: one centre per pair");
        if (offsets.empty()) throw std::invalid_argument("relocalizePairs: offsets must have nscans + 1 entries");
        if (offsets.front() < 0 || static_cast<size_t>(offsets.back()) > points.size()) throw std::invalid_argument("relocalizePairs: offsets overrun points");
        if (k < 1) throw std::invalid_argument("relocalizePairs: k >= 1");
        const size_t n = pairs.size() * static_cast<size_t>(k);
        std::vector<Result> out(n);
        std::vector<std::int64_t> idx(n, -1);
        std::vector<double> val(n, 0.0);
        ck(ndt2d_relocalize_pairs(h_, level, reinterpret_cast<const float *>(points.data()), offsets.data(), static_cast<int>(offsets.size() - 1),
                                  reinterpret_cast<const std::int32_t *>(pairs.data()), static_cast<int>(pairs.size()),
                                  reinterpret_cast<const double *>(centres.data()), &window, k, idx.data(), val.data(), out.data()));
        if (indices) *indices = std::move(idx);
        if (scores) *scores = std::move(val);
        return out;
    }

    // pairs against submaps of posed scans (SPEC 7.3): pair p = (submap pairs[p].first, source scan pairs[p].second); submap g
    // is the scans submaps[g].scans of the packed batch at submaps[g].poses. alignSubmaps equals setTargetScans(members) +
    // align(source, init[p]) per pair; relocalizeSubmaps equals setTargetScans(members) + relocalize(source, window
    // hypotheses around centres[p], k, level), returned as relocalizePairs returns them.
    std::vector<Result> alignSubmaps(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets,
                                     const std::vector<Submap> &submaps, const std::vector<std::pair<std::int32_t, std::int32_t>> &pairs,
                                     const std::vector<Pose2d> &init)
    {
        if (pairs.size() != init.size()) throw std::invalid_argument("alignSubmaps: one initial pose per pair");
        checkPacked(points, offsets, "alignSubmaps");
        PackedSubmaps s(submaps);
        std::vector<Result> out(pairs.size());
        ck(ndt2d_align_submaps(h_, reinterpret_cast<const float *>(points.data()), offsets.data(), static_cast<int>(offsets.size() - 1),
                               s.offsets.data(), static_cast<int>(submaps.size()), s.scans.data(), s.poses.data(),
                               reinterpret_cast<const std::int32_t *>(pairs.data()), static_cast<int>(pairs.size()),
                               reinterpret_cast<const double *>(init.data()), out.data()));
        return out;
    }
    std::vector<Result> relocalizeSubmaps(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets,
                                          const std::vector<Submap> &submaps, const std::vector<std::pair<std::int32_t, std::int32_t>> &pairs,
                                          const std::vector<Pose2d> &centres, const ndt2d_window &window, int k, int level = 0,
                                          std::vector<std::int64_t> *indices = nullptr, std::vector<double> *scores = nullptr)
    {
        if (pairs.size() != centres.size()) throw std::invalid_argument("relocalizeSubmaps: one centre per pair");
        checkPacked(points, offsets, "relocalizeSubmaps");
        if (k < 1) throw std::invalid_argument("relocalizeSubmaps: k >= 1");
        PackedSubmaps s(submaps);
        const size_t n = pairs.size() * static_cast<size_t>(k);
        std::vector<Result> out(n);
        std::vector<std::int64_t> idx(n, -1);
        std::vector<double> val(n, 0.0);
        ck(ndt2d_relocalize_submaps(h_, level, reinterpret_cast<const float *>(points.data()), offsets.data(),
                                    static_cast<int>(offsets.size() - 1), s.offsets.data(), static_cast<int>(submaps.size()), s.scans.data(),
                                    s.poses.data(), reinterpret_cast<const std::int32_t *>(pairs.data()), static_cast<int>(pairs.size()),
                                    reinterpret_cast<const double *>(centres.data()), &window, k, idx.data(), val.data(), out.data()));
        if (indices) *indices = std::move(idx);
        if (scores) *scores = std::move(val);
        return out;
    }

    // windowed relocalisation of a batch of scans in this handle's map: for scan b, the window's hypotheses around centres[b]
    // are swept on `level` and the k best refined; equals relocalize(scan b, window hypotheses, k, level) per scan.
    // Returns nscans * k records, scan-major; indices / scores (optional) receive the k sweep indices and scores per scan
    // (index -1: no candidate).
    std::vector<Result> relocalizeBatch(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets,
                                        const std::vector<Pose2d> &centres, const ndt2d_window &window, int k, int level = 0,
                                        std::vector<std::int64_t> *indices = nullptr, std::vector<double> *scores = nullptr)
    {
        if (offsets.empty()) throw std::invalid_argument("relocalizeBatch: offsets must have nscans + 1 entries");
        if (centres.size() != offsets.size() - 1) throw std::invalid_argument("relocalizeBatch: one centre per scan");
        if (offsets.front() < 0 || static_cast<size_t>(offsets.back()) > points.size()) throw std::invalid_argument("relocalizeBatch: offsets overrun points");
        if (k < 1) throw std::invalid_argument("relocalizeBatch: k >= 1");
        const size_t n = centres.size() * static_cast<size_t>(k);
        std::vector<Result> out(n);
        std::vector<std::int64_t> idx(n, -1);
        std::vector<double> val(n, 0.0);
        ck(ndt2d_relocalize_batch(h_, level, reinterpret_cast<const float *>(points.data()), offsets.data(), static_cast<int>(centres.size()),
                                  reinterpret_cast<const double *>(centres.data()), &window, k, idx.data(), val.data(), out.data()));
        if (indices) *indices = std::move(idx);
        if (scores) *scores = std::move(val);
        return out;
    }

    // ---- multi-hypothesis search (relocalisation, loop-closure candidates) --------------------------
    // hypotheses: (x, y, theta) float triples. Returns the k best (index, score), best first.
    std::vector<std::pair<std::int64_t, double>> sweep(const std::vector<Point2f> &scan, const std::vector<float> &hyp_xyt, int k,
                                                       int level = 0, std::vector<double> *scores = nullptr)
    {
        const std::int64_t m = static_cast<std::int64_t>(hyp_xyt.size() / 3);
        std::vector<std::int64_t> idx(static_cast<size_t>(k), -1);
        std::vector<double> val(static_cast<size_t>(k), 0.0);
        if (scores) scores->assign(static_cast<size_t>(m), 0.0);
        ck(ndt2d_sweep(h_, level, reinterpret_cast<const float *>(scan.data()), static_cast<int>(scan.size()), hyp_xyt.data(), m,
                       scores ? scores->data() : nullptr, k, idx.data(), val.data()));
        std::vector<std::pair<std::int64_t, double>> out;
        for (int i = 0; i < k && idx[static_cast<size_t>(i)] >= 0; ++i) out.emplace_back(idx[static_cast<size_t>(i)], val[static_cast<size_t>(i)]);
        return out;
    }
    // sweep, then a full align from each of the k best
    std::vector<Result> relocalize(const std::vector<Point2f> &scan, const std::vector<float> &hyp_xyt, int k, int level = 0)
    {
        std::vector<std::int64_t> idx(static_cast<size_t>(k), -1);
        std::vector<Result> res(static_cast<size_t>(k));
        ck(ndt2d_relocalize(h_, level, reinterpret_cast<const float *>(scan.data()), static_cast<int>(scan.size()), hyp_xyt.data(),
                            static_cast<std::int64_t>(hyp_xyt.size() / 3), k, idx.data(), res.data()));
        return res;
    }

    // ---- evaluation at fixed poses: {S, g0,g1,g2, H00,H01,H02,H11,H12,H22} ---------------------------
    std::array<double, 10> evaluate(const std::vector<Point2f> &scan, const Pose2d &pose, int level = 0, int *count = nullptr)
    {
        const double p[3] = {pose.x, pose.y, pose.theta};
        std::array<double, 10> out{};
        std::int32_t c = 0;
        ck(ndt2d_evaluate(h_, level, reinterpret_cast<const float *>(scan.data()), static_cast<int>(scan.size()), p, 1, out.data(), &c));
        if (count) *count = c;
        return out;
    }

    // ---- several GPUs, one process each: best-hypothesis exchange of a sharded sweep over peer memory ------
    // exchangeCreate() returns this rank's 64-byte IPC handle; all-gather the handles with the host code's own
    // transport (MPI, sockets, ...) and pass them, ordered by rank, to exchangeOpen().
    std::array<unsigned char, NDT2D_IPC_HANDLE_BYTES> exchangeCreate(int world, int rank, int nslots = 64)
    {
        std::array<unsigned char, NDT2D_IPC_HANDLE_BYTES> h{};
        ck(ndt2d_exchange_create(h_, world, rank, nslots, h.data()));
        return h;
    }
    void exchangeOpen(const std::vector<unsigned char> &handles_by_rank) { ck(ndt2d_exchange_open(h_, handles_by_rank.data())); }
    // device pointers; hypothesis j of the shard has global index index_offset + j; asynchronous
    void sweepPublish(int level, const float *d_scan_xy, int n, const float *d_hyp_xyt, std::int64_t nhyp, std::int64_t index_offset,
                      std::uint64_t query, double *d_scores = nullptr)
    {
        ck(ndt2d_sweep_publish(h_, level, d_scan_xy, n, d_hyp_xyt, nhyp, d_scores, index_offset, query));
    }
    std::pair<std::int64_t, double> exchangeWait(std::uint64_t query, int timeout_ms = 10000)
    {
        std::int64_t idx = -1;
        double score = 0.0;
        ck(ndt2d_exchange_wait(h_, query, timeout_ms, &idx, &score));
        return {idx, score};
    }
    void exchangeClose() { ck(ndt2d_exchange_close(h_)); }

    // multi-GPU relocalisation end to end over peer memory (ndt2d_reloc_* / ndt2d_relocalize_* in ndt2d.h): every rank
    // sweeps its shard, refines its own k best and stores the candidates into every rank's table; relocalizeWait merges them
    std::array<unsigned char, NDT2D_IPC_HANDLE_BYTES> relocCreate(int world, int rank, int nslots = 16, int kmax = 8)
    {
        std::array<unsigned char, NDT2D_IPC_HANDLE_BYTES> h{};
        ck(ndt2d_reloc_create(h_, world, rank, nslots, kmax, h.data()));
        return h;
    }
    void relocOpen(const std::vector<unsigned char> &handles_by_rank) { ck(ndt2d_reloc_open(h_, handles_by_rank.data())); }
    void relocalizePublish(int level, const float *d_scan_xy, int n, const float *d_hyp_xyt, std::int64_t nhyp, std::int64_t index_offset, int k,
                           std::uint64_t query)
    {
        ck(ndt2d_relocalize_publish(h_, level, d_scan_xy, n, d_hyp_xyt, nhyp, index_offset, k, query));
    }
    std::vector<Result> relocalizeWait(std::uint64_t query, int k, std::vector<std::int64_t> *indices = nullptr, int timeout_ms = 10000)
    {
        std::vector<std::int64_t> idx(static_cast<size_t>(k), -1);
        std::vector<Result> res(static_cast<size_t>(k));
        ck(ndt2d_relocalize_wait(h_, query, timeout_ms, k, idx.data(), res.data()));
        if (indices) *indices = idx;
        return res;
    }
    void relocClose() { ck(ndt2d_reloc_close(h_)); }

    ndt2d_matcher *handle() const { return h_; }
    void synchronize() { ck(ndt2d_synchronize(h_)); }
    // a share of the input of the host-buffer batch calls travels over another GPU's PCIe link and NVLink (ndt2d_set_upload_relay)
    void setUploadRelay(int relayDevice, double fraction = 0.5) { ck(ndt2d_set_upload_relay(h_, relayDevice, fraction)); }

  private:
    void ck(int rc) const
    {
        if (rc != NDT2D_OK) throw std::runtime_error(std::string("libndt2d (") + std::to_string(rc) + "): " + ndt2d_last_error(h_));
    }
    void targetScans(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets, const std::vector<Pose2d> &poses,
                     bool add)
    {
        if (offsets.size() != poses.size() + 1) throw std::invalid_argument("setTargetScans: offsets.size() must be poses.size() + 1");
        if (offsets.back() < 0 || static_cast<size_t>(offsets.back()) > points.size())
            throw std::invalid_argument("setTargetScans: offsets overrun points");
        const float *xy = reinterpret_cast<const float *>(points.data());
        const double *p = reinterpret_cast<const double *>(poses.data());
        const int nb = static_cast<int>(poses.size());
        ck(add ? ndt2d_add_target_scans(h_, xy, offsets.data(), nb, p) : ndt2d_set_target_scans(h_, xy, offsets.data(), nb, p));
    }
    static void checkPacked(const std::vector<Point2f> &points, const std::vector<std::int64_t> &offsets, const char *name)
    {
        if (offsets.empty()) throw std::invalid_argument(std::string(name) + ": offsets must have nscans + 1 entries");
        if (offsets.front() < 0 || static_cast<size_t>(offsets.back()) > points.size())
            throw std::invalid_argument(std::string(name) + ": offsets overrun points");
    }
    // the C ABI's three submap arrays
    struct PackedSubmaps {
        std::vector<std::int64_t> offsets{0};
        std::vector<std::int32_t> scans;
        std::vector<double> poses;
        explicit PackedSubmaps(const std::vector<Submap> &submaps)
        {
            for (const Submap &s : submaps) {
                if (s.scans.size() != s.poses.size()) throw std::invalid_argument("Submap: one pose per member scan");
                scans.insert(scans.end(), s.scans.begin(), s.scans.end());
                for (const Pose2d &p : s.poses) poses.insert(poses.end(), {p.x, p.y, p.theta});
                offsets.push_back(static_cast<std::int64_t>(scans.size()));
            }
        }
    };
    void targetRanges(const std::vector<float> &ranges, int nbeams, double angle_min, double angle_inc, float range_min,
                      float range_max, const std::vector<Pose2d> &poses, bool add)
    {
        if (nbeams < 1 || ranges.size() != poses.size() * static_cast<size_t>(nbeams))
            throw std::invalid_argument("setTargetRanges: ranges.size() must be poses.size() * nbeams");
        const double *p = reinterpret_cast<const double *>(poses.data());
        const int nb = static_cast<int>(poses.size());
        ck(add ? ndt2d_add_target_ranges(h_, ranges.data(), 0, nb, nbeams, angle_min, angle_inc, 1.0f, range_min, range_max, p)
               : ndt2d_set_target_ranges(h_, ranges.data(), 0, nb, nbeams, angle_min, angle_inc, 1.0f, range_min, range_max, p));
    }
    ndt2d_matcher *h_ = nullptr;
};

} // namespace ndt2d

#endif // NDT2D_HPP
