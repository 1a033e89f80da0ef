// Hand-written sm_100a kernels of the 2D NDT hot path (BASELINE.json north_star items 1-3):
//   (1) grid build: integer accumulation with warp-level segmented reduction + finalise (SPEC 3)
//   (2) Newton-step evaluation and the whole Levenberg-Marquardt loop on the device (SPEC 4, 5)
//   (3) batched multi-hypothesis scoring and top-k (SPEC 6)
// These are gather-bound kernels over an L2-resident cell table: no tensor cores (north_star).
// Reference file:line: none (the mount is /root/reference/README.md:1 only); arithmetic follows SPEC.md.
#include "ndt2d_align.cuh"

#include <math.h>
#include <string.h>

#include <type_traits>

namespace ndt2d {

static constexpr unsigned FULL_MASK = 0xffffffffu;

// ------------------------------------------------------------------------------------------------
// (1) grid build
// ------------------------------------------------------------------------------------------------

// Target point sources (TargetSrc): map-frame points, or posed scans as packed points or as LaserScan ranges.
enum { SRC_POINTS = 0, SRC_SCANS = 1, SRC_RANGES = 2 };

// Point i of the source in f64 map coordinates; false when there is no such point (i >= n, a dropped beam, a non-finite
// scan coordinate). Map-frame points are widened (SPEC 3); a scan point is transformed by its scan's pose and not rounded
// (SPEC 7.2). A packed point finds its scan by binary search over offsets[1 .. nscans-1]: whatever the offsets hold, the
// scan index stays in [0, nscans) and only points below n are read.
template <int SRC>
__device__ __forceinline__ bool target_point(const TargetSrc &s, int64_t i, double &X, double &Y)
{
    X = Y = 0.0;
    if (i >= s.n) return false;
    if (SRC == SRC_POINTS) {
        const float2 p = __ldg(s.xy + i);
        X = (double)p.x;
        Y = (double)p.y;
        return true;
    }
    float x, y;
    int b;
    bool ok = true;
    if (SRC == SRC_SCANS) {
        const float2 p = __ldg(s.xy + i);
        x = p.x; y = p.y;
        int lo = 0, hi = s.nscans - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__ldg(s.offsets + mid) <= i) lo = mid;
            else hi = mid - 1;
        }
        b = lo;
    } else {
        b = (int)(i / s.nbeams);
        const int beam = (int)(i - (int64_t)b * s.nbeams);
        float rho;
        if (s.ranges_u16) {
            const unsigned short u = __ldg(reinterpret_cast<const unsigned short *>(s.ranges) + i);
            rho = __fmul_rn((float)u, s.range_scale);
            ok = (u != 0);
        } else {
            rho = __ldg(reinterpret_cast<const float *>(s.ranges) + i);
        }
        ok = ok && (rho >= s.range_min) && (rho <= s.range_max);   // SPEC 8
        const float2 bt = __ldg(s.beams + beam);
        x = __fmul_rn(rho, bt.x);
        y = __fmul_rn(rho, bt.y);
    }
    if (!ok || !isfinite(x) || !isfinite(y)) return false;
    posed_point(s.pose + 4 * (size_t)b, x, y, X, Y);
    return true;
}

// the posed sources' per-scan {cos, sin, p0, p1}, sin and cos by SPEC 4.2
__global__ void k_pose_table(const double *__restrict__ poses, int nscans, double *__restrict__ tab)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nscans) return;
    double sn, cs;
    sincos_spec(poses[3 * (size_t)b + 2], sn, cs);
    tab[4 * (size_t)b] = cs;
    tab[4 * (size_t)b + 1] = sn;
    tab[4 * (size_t)b + 2] = poses[3 * (size_t)b];
    tab[4 * (size_t)b + 3] = poses[3 * (size_t)b + 1];
}

// SPEC 3 accumulation into level blockIdx.y of S: every level of a pyramid from the same points in one launch (a target
// SCAN's grids are so small that the launches, not the work, were the cost of building them; sequential scan-to-scan
// odometry builds three levels per step). One point per lane; for each of the K cells of the point, lanes holding the
// same cell in consecutive positions (laser scans are spatially coherent) are combined with a segmented shuffle reduction
// and only the head of each run issues the integer atomics. Integer sums are associative, so the result is independent
// of the order of points, warps and atomics (a window of packed scan points may straddle two scans).
// TOUCH (incremental update): the first run head to reach a cell since the last finalisation (an exchange on the cell's
// dirty word) appends it to the level's list, so that the finalisation can visit the touched cells only.
template <int OV, bool TOUCH, int SRC>
__global__ void __launch_bounds__(256) k_accumulate(const __grid_constant__ LevelSet S, const TargetSrc src)
{
    const int l = blockIdx.y;
    const LevelDev &L = S.lv[l];
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t warp_id = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (int64_t base = warp_id * 32; base < src.n; base += warps_total * 32) {
        double X, Y;
        const bool valid = target_point<SRC>(src, base + lane, X, Y);
        accumulate_window<OV>(L, valid, X, Y, lane, [&](int key, unsigned c, long long sx, long long sy, long long sxx, long long sxy, long long syy) {
            if (TOUCH && atomicExch(S.dirty[l] + key, 1u) == 0u) S.list[l][atomicAdd(S.nlist + l, 1u)] = (unsigned)key;
            atomicAdd(L.cnt + key, c);
            unsigned long long *s = L.sums + 5 * (size_t)key;
            atomicAdd(s + 0, (unsigned long long)sx);
            atomicAdd(s + 1, (unsigned long long)sy);
            atomicAdd(s + 2, (unsigned long long)sxx);
            atomicAdd(s + 3, (unsigned long long)sxy);
            atomicAdd(s + 4, (unsigned long long)syy);
        });
    }
}

// SPEC 3 finalisation of level blockIdx.y of S, one thread per cell (the arithmetic is finalize_record() in
// ndt2d_device.cuh): every cell, or with LIST the cells of the level's touched list, whose dirty words are cleared.
template <bool LIST>
__global__ void __launch_bounds__(256) k_finalize(const __grid_constant__ LevelSet S, int min_points, double eig_ratio)
{
    const int l = blockIdx.y;
    const LevelDev &L = S.lv[l];
    float4 *__restrict__ cells = S.cells[l];
    const int64_t n = LIST ? (int64_t)S.nlist[l] : (int64_t)L.njx * L.njy;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = LIST ? (int64_t)S.list[l][e] : e;
        const long long *s = reinterpret_cast<const long long *>(L.sums) + 5 * c;
        float4 ra, rb;
        finalize_record(L.cnt[c], s[0], s[1], s[2], s[3], s[4], L.qu, min_points, eig_ratio, ra, rb);
        cells[2 * c] = ra;
        cells[2 * c + 1] = rb;
        if (LIST) S.dirty[l][c] = 0u;
    }
}

// ------------------------------------------------------------------------------------------------
// (2a) small per-point kernels used by the API's diagnostic entry points
// ------------------------------------------------------------------------------------------------

__global__ void k_cell_index(const LevelDev L, const float2 *__restrict__ xy, int n, const double *__restrict__ pose,
                             int32_t *__restrict__ idx)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float2 p = xy[i];
    int hx, hy;
    bool in;
    if (pose) {
        const PosePk P = pose_pack(pose_for_level(pose[0], pose[1], pose[2], L));
        float2 ps = sanitize(p);
        unsigned ux, uy;
        u64 df;
        in = locate_point(P, ps.x, ps.y, (unsigned)L.nhx, (unsigned)L.nhy, ux, uy, df);
        hx = (int)ux;
        hy = (int)uy;
    } else {
        in = lattice_of_point(L, p.x, p.y, hx, hy);
    }
    idx[i] = in ? hy * L.nhx + hx : -1;
}

template <int OV>
__global__ void k_point_terms(const LevelDev L, const float2 *__restrict__ xy, int n, const double *__restrict__ pose,
                              float *__restrict__ terms)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    constexpr int K = OV ? 4 : 1;
    const PosePk P = pose_pack(pose_for_level(pose[0], pose[1], pose[2], L));
    const LatticePk G = lattice_pack<OV>(L, TABLE_DENSE);
    float2 p = sanitize(xy[i]);
    PointPk pt;
    rotate_point(P, p.x, p.y, pt);
    float *out = terms + (size_t)i * K * 10;
    for (int t = 0; t < K * 10; ++t) out[t] = 0.0f;
    unsigned hx, hy;
    if (!locate_point(P, p.x, p.y, G.nhx, G.nhy, hx, hy, pt.df)) return;
    for (int k = 0; k < K; ++k) {
        unsigned cidx = (hy + (k >> 1)) * (unsigned)L.njx + (hx + (k & 1));
        Cell4 rec = load_cell(L.cells, cidx);
        pt.XY = local_xy(G, pt.df, k);
        float T[10];
        if (pair_terms_scalar(rec, pt, T))
            for (int t = 0; t < 10; ++t) out[k * 10 + t] = T[t];
    }
}

// ------------------------------------------------------------------------------------------------
// (2b)/(3) one scan against many poses: the Newton-step evaluation and the sweep
// ------------------------------------------------------------------------------------------------

static constexpr int EVAL_THREADS = 256;
// resident k_eval_poses blocks per SM for the score-only sweep: 4 (32 warps, 56 registers) and 5 (40 warps, 48 registers) both
// reach 446.8 M hypotheses/s, 6 (48 warps, 40 registers: constants re-materialised in the loop) 434 M
static constexpr int EVAL_BLOCKS = 4;
static constexpr int EVAL_BLOCKS_FULL = 3; // the full evaluation needs the align kernel's 80 registers: 24 warps per SM

// Block stages the scan in shared memory once (coalesced float2 loads), then each warp takes poses
// from a grid-stride loop. FULL: ten f64 sums per pose; otherwise the score only (sweep).
template <int OV, bool FULL, bool F32POSE, bool STAGED>
__global__ void __launch_bounds__(EVAL_THREADS, FULL ? EVAL_BLOCKS_FULL : EVAL_BLOCKS) k_eval_poses(const LevelDev L, const float2 *__restrict__ xy, int n,
                                                               const void *__restrict__ poses, int64_t npose,
                                                               double *__restrict__ out, int out_stride,
                                                               int32_t *__restrict__ count)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int npad = (n + 63) & ~63;
    float2 *sp = reinterpret_cast<float2 *>(smem_raw);
    constexpr bool P64 = STAGED && !FULL;   // the score-only sweep needs the points in f64 only: widen them once, here
    if (STAGED) {
        // sanitised points, padded with the far-away point to a multiple of 64 (SPEC 4)
        for (int i = threadIdx.x; i < npad; i += blockDim.x) {
            const float2 p = i < n ? sanitize(__ldg(xy + i)) : make_float2(1e18f, 1e18f);
            if (P64) reinterpret_cast<double2 *>(smem_raw)[i] = make_double2((double)p.x, (double)p.y);
            else sp[i] = p;
        }
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * (EVAL_THREADS / 32);
    for (int64_t j = (int64_t)blockIdx.x * (EVAL_THREADS / 32) + (threadIdx.x >> 5); j < npose; j += warps_total) {
        double tx, ty, th;
        if (F32POSE) {
            const float *h = reinterpret_cast<const float *>(poses) + 3 * j;
            tx = (double)__ldg(h); ty = (double)__ldg(h + 1); th = (double)__ldg(h + 2);
        } else {
            const double *h = reinterpret_cast<const double *>(poses) + 3 * j;
            tx = __ldg(h); ty = __ldg(h + 1); th = __ldg(h + 2);
        }
        Pose32 q = pose_for_level<!FULL>(tx, ty, th, L);   // the score-only sweep takes the sin/cos coefficients from constant memory
        Eval E;
        // FULL: the transposed reduction leaves sum number E.slot in every lane (lanes with the same slot hold the same bits)
        if (STAGED) eval_warp<OV, FULL, true, FULL, TABLE_DENSE, P64>(L, sp, n, q, lane, E);
        else eval_warp<OV, FULL, false, FULL>(L, xy, n, q, lane, E);
        if (FULL) out[(size_t)j * out_stride + E.slot] = E.v[0];
        else if (lane == 0) out[(size_t)j * out_stride] = E.v[0];
        if (count && lane == 0) count[j] = E.count;
    }
}

// ------------------------------------------------------------------------------------------------
// (2c) batched align: one warp per scan, the whole LM loop on the device
// ------------------------------------------------------------------------------------------------

// 24 warps per SM at 80 registers, as six blocks of four warps. Measured operating points (gpurun_out/x10_variants.jsonl, M matches/s
// on configs[1], all bit-identical): 128 x 6: 20.46, 256 x 3: 20.32, 384 x 2: 20.22 (the same 24 warps in larger blocks: a block
// holds its shared memory until its last warp has drained the queue), 160 x 4 (20 warps, 96 registers): 19.53, 320 x 2 (20
// warps): 19.43, 256 x 2 (16 warps, 104 registers, the only point whose loop has no register copies): 19.17.
// ALIGN_THREADS (k_align's block size) lives in ndt2d_align.cuh with the helper-warp machinery
static constexpr int ALIGN_MIN_BLOCKS = 6;
// batches of at most this many scans run k_align with helper warps, when the handle leaves the choice open
// (tools/midsize_probe.py: -12 % at 1250-2500 scans, -5 % at 5000, +-0 at 10 000, +2 % at 20 000,
// +8 % at 65 536 - the helper form's point loop is 134 instructions against 129)
static constexpr int HELP_MAX_SCANS = 8192;

// ------------------------------------------------------------------------------------------------
// (2d) low-latency align: one BLOCK per scan, for calls with few scans (a single align above all)
// ------------------------------------------------------------------------------------------------
// With one warp per scan an evaluation is 17 dependent (gather, compute) steps, ~9 us; a lone align is latency, not
// throughput. Here the eight warps of a block compute the SPEC 4 factors (e, c1..c9) of different 64-point steps at
// the same time and park them in shared memory; they are then applied to the 64 partial sums in the order SPEC 4
// prescribes (increasing point index, cell order within a point) - by five warps, each owning whole accumulators - so the
// sums, and everything after, are the bits of the one-warp kernel. The LM logic is executed by every thread on the same
// shared-memory state (uniform).

static constexpr int BLOCK_ALIGN_THREADS = 256; // at least 5 warps (the second half of eval_block)
static_assert(BLOCK_ALIGN_THREADS >= 160 && BLOCK_ALIGN_THREADS % 32 == 0, "eval_block applies the factors with five warps");

template <int OV>
__device__ __forceinline__ void eval_block(const LevelDev *L, const float2 *pts, int n, WarpState *ws, u64 *fac)
{
    constexpr int NC = OV ? 4 : 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double *pose = ws->pn;
    const PosePk P = pose_pack(pose_for_level(pose[0], pose[1], pose[2], *L));
    const LatticePk G = lattice_pack<OV>(*L, TABLE_DENSE);
    const float4 *__restrict__ cells = L->cells;
    const int nsteps = (n + 63) >> 6;
    for (int step = warp; step < nsteps; step += BLOCK_ALIGN_THREADS / 32) {
        Fetched<OV> F;
        fetch<OV, true, TABLE_DENSE>(cells, G, P, pts, n, (step << 6) + lane, F);
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            Factors X;
            int c = 0;
            F.A.XY = local_xy(G, F.A.df, k);
            F.B.XY = local_xy(G, F.B.df, k);
            cell_factors<true>(F.cA[k], F.cB[k], F.A, F.B, X, c);
            park_factors(X, fac + ((size_t)(step * NC + k) * FACTOR_WORDS) * 32 + lane);
        }
    }
    __syncthreads();
    // Second half: the parked factors are applied in SPEC order - but SPEC 4 orders the updates of ONE accumulator; the ten
    // accumulators of a partial are independent chains. Five warps each take the accumulators that end in the same sums
    // (warp 0: T0 T3 T9 and the count; warps 1-3: the per-point pairs (T1,T2) (T4,T5) (T6,T8); warp 4: T7), widen to f64
    // and run SPEC 4's butterfly for their sums: the serial tail of an evaluation is a fifth of what one warp would need.
    if (warp < 5) {
        const int ne = nsteps * NC;
        const u64 *o = fac + lane;
        if (warp == 0) {
            u64 s0 = 0ull, s3 = 0ull, s9 = 0ull;
            int cnt = 0;
            for (int e = 0; e < ne; ++e, o += FACTOR_WORDS * 32) {
                const u64 ee = o[0 * 32];
                // a contributing pair has e = exp(-h) with h < 30, never zero; a skipped pair has e = 0 exactly
                cnt += (lo32(ee) != 0.0f ? 1 : 0) + (hi32(ee) != 0.0f ? 1 : 0);
                add2_acc(s0, ee);
                fma2_acc(s3, ee, o[7 * 32]);
                fma2_acc(s9, ee, o[8 * 32]);
            }
            const double t0 = warp_sum((double)lo32(s0) + (double)hi32(s0));
            const double t3 = warp_sum((double)lo32(s3) + (double)hi32(s3));
            const double t9 = warp_sum((double)lo32(s9) + (double)hi32(s9));
            cnt = __reduce_add_sync(FULL_MASK, cnt);
            if (lane == 0) { ws->t[0] = t0; ws->t[3] = t3; ws->t[9] = t9; ws->tcount = cnt; }
        } else if (warp < 4) {
            const int w0 = 2 * warp - 1;                      // words (1,2) (3,4) (5,6): the pair of point A, of point B
            u64 a = 0ull, b = 0ull;
            for (int e = 0; e < ne; ++e, o += FACTOR_WORDS * 32) {
                const u64 ee = o[0 * 32];
                fma2_acc(a, o[w0 * 32], bc(lo32(ee)));
                fma2_acc(b, o[(w0 + 1) * 32], bc(hi32(ee)));
            }
            const double tl = warp_sum((double)lo32(a) + (double)lo32(b));
            const double th = warp_sum((double)hi32(a) + (double)hi32(b));
            const int il = warp == 1 ? 1 : warp == 2 ? 4 : 6, ih = warp == 1 ? 2 : warp == 2 ? 5 : 8;
            if (lane == 0) { ws->t[il] = tl; ws->t[ih] = th; }
        } else {
            float a = 0.0f, b = 0.0f;
            for (int e = 0; e < ne; ++e, o += FACTOR_WORDS * 32) {
                const u64 ee = o[0 * 32];
                float cA, cB;
                upk(o[9 * 32], cA, cB);
                a = __fmaf_rn(lo32(ee), cA, a);
                b = __fmaf_rn(hi32(ee), cB, b);
            }
            const double t7 = warp_sum((double)a + (double)b);
            if (lane == 0) ws->t[7] = t7;
        }
    }
    __syncthreads();
}

template <int OV>
__device__ __forceinline__ int align_level_block(const LevelDev *L, const ndt2d_params &P, const float2 *pts, int n, WarpState *ws,
                                                 u64 *fac, int &evals_total)
{
    // eval_block begins its second half with __syncthreads() and ends with one
    return lm_level<BlockScope>(P, n, ws, evals_total, [&]() { eval_block<OV>(L, pts, n, ws, fac); });
}

// SPEC 8 for one warp: the beams of LaserScan `job` with range_min <= rho <= range_max, converted to points and written to
// `slot` in beam order; returns how many were kept. (k_align's staging step in ranges mode, and k_align_block's, done by warp 0.)
__device__ __forceinline__ int stage_ranges(const AlignArgs &a, unsigned job, float2 *slot, int lane)
{
    int kept = 0;
    for (int b0 = 0; b0 < a.nbeams; b0 += 32) {
        int b = b0 + lane;
        float rho = 0.0f;
        bool ok = false;
        if (b < a.nbeams) {
            if (a.ranges_u16) {
                unsigned short u = __ldg(reinterpret_cast<const unsigned short *>(a.ranges) + (size_t)job * a.nbeams + b);
                rho = __fmul_rn((float)u, a.range_scale);
                ok = (u != 0);
            } else {
                rho = __ldg(reinterpret_cast<const float *>(a.ranges) + (size_t)job * a.nbeams + b);
                ok = true;
            }
            ok = ok && (rho >= a.range_min) && (rho <= a.range_max);
        }
        unsigned m = __ballot_sync(FULL_MASK, ok);
        if (ok) {
            float2 bt = __ldg(a.beams + b);
            int dst = kept + __popc(m & ((1u << lane) - 1u));
            slot[dst] = sanitize(make_float2(__fmul_rn(rho, bt.x), __fmul_rn(rho, bt.y)));
        }
        kept += __popc(m);
    }
    return kept;
}

// RANGES: LaserScan input (a.ranges != nullptr); warp 0 converts and compacts the beams, the other warps wait at the barrier
template <int OV, bool RANGES = false>
__global__ void __launch_bounds__(BLOCK_ALIGN_THREADS) k_align_block(const __grid_constant__ AlignArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_n;
    WarpState *ws = reinterpret_cast<WarpState *>(smem_raw);
    float2 *pts = reinterpret_cast<float2 *>(smem_raw + sizeof(WarpState));
    u64 *fac = reinterpret_cast<u64 *>(smem_raw + sizeof(WarpState) + (size_t)a.cap_points * sizeof(float2));
    const int job = blockIdx.x, tid = threadIdx.x;
    int n;
    if (RANGES) {
        if (tid < 32) {
            const int kept = stage_ranges(a, (unsigned)job, pts, tid);
            for (int i = kept + tid; i < ((kept + 63) & ~63); i += 32) pts[i] = make_float2(1e18f, 1e18f);
            if (tid == 0) s_n = kept;
        }
        if (tid < 3) ws->p[tid] = __ldg(a.init + 3 * (size_t)job + tid);
        __syncthreads();
        n = s_n;
    } else {
        const int scan = a.job_scan ? __ldg(a.job_scan + job) : job;
        const int64_t o0 = scan >= 0 ? __ldg(a.offsets + scan) : 0, o1 = scan >= 0 ? __ldg(a.offsets + scan + 1) : 0;
        n = (int)(o1 - o0);
        const int npad = (n + 63) & ~63;
        const float2 *src = a.xy + o0;
        for (int i = tid; i < npad; i += BLOCK_ALIGN_THREADS) pts[i] = i < n ? sanitize(__ldg(src + i)) : make_float2(1e18f, 1e18f);
        if (tid < 3) ws->p[tid] = __ldg(a.init + 3 * (size_t)job + tid);
        __syncthreads();
    }
    int evals = 0, status = NDT2D_NO_OVERLAP;
    for (int l = 0; l < a.nlevels; ++l) status = align_level_block<OV>(&a.lv[l], a.prm, pts, n, ws, fac, evals);
    if (tid == 0) write_result(*ws, evals, status, a.res + job);
}

// Persistent kernel: warps pull scan indices from a global counter until the batch is drained.
// STAGED: the scan is copied once into this warp's shared-memory slot and re-read from there on
// every iteration (an align touches its points 10-30 times, its HBM bytes once).
// RANGES: the scan arrives as LaserScan ranges and is converted in the staging step (SPEC 8).
// PAIRS (ndt2d_align_pairs): job p aligns scan a.pairs[2p+1] to target slot a.pairs[2p]; the target's levels are
// a.geo[slot * nlevels + l], whose cell tables are hash tables built by k_pairs_build.
// HELP (K = 1, scans staged in shared memory, dense table): warps that find the queue empty help the warps of their block that
// still hold a scan (ndt2d_align.cuh); the launch's tail and batches that do not fill the GPU finish sooner, same bits.
template <int OV, bool STAGED, bool RANGES, bool PAIRS = false, bool HELP = false>
__global__ void __launch_bounds__(ALIGN_THREADS, (STAGED || RANGES) ? ALIGN_MIN_BLOCKS : 1) k_align(const __grid_constant__ AlignArgs a)
{
    static_assert(!HELP || (OV == 0 && (STAGED || RANGES) && !PAIRS), "helpers park one cell's factors per step and read the owner's staged scan");
    unsigned char *smem_raw = align_smem();
    constexpr bool SM = STAGED || RANGES;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // per-warp slot of cap points (a multiple of 64), after the warp states (and the help desks)
    WarpState *ws = reinterpret_cast<WarpState *>(smem_raw) + warp;
    float2 *slot = reinterpret_cast<float2 *>(HELP ? help_slots() : smem_raw + kAlignWarps * sizeof(WarpState)) + (size_t)warp * a.cap_points;
    const float2 far = make_float2(1e18f, 1e18f);
    if (HELP) {
        HelpDesk *d = help_desk(warp);
        if (lane == 0) {
            d->post = d->cur = 0u;
            d->active = 1u;          // every warp may own scans until it has seen the queue empty itself
            d->slot_bytes = (unsigned)a.cap_points * (unsigned)sizeof(float2);
            d->level = d->n = 0;
        }
        if (lane < 7) { d->helper[lane] = kNoHelper; d->done[lane] = 0u; }
        __syncthreads();
    }

    bool first_job = true;
    for (;;) {
        unsigned job = 0;
        if (HELP && first_job) {
            // a warp's first scan is assigned statically, warp w of every block before warp w + 1 of any: a batch that does
            // not fill the GPU is spread over the blocks, and the warps left without a scan are helpers next to an owner
            job = (unsigned)warp * gridDim.x + blockIdx.x;
            first_job = false;
        } else {
            if (lane == 0) job = atomicAdd(a.counter, 1u);
            job = __shfl_sync(FULL_MASK, job, 0);
            if (HELP) job += gridDim.x * (unsigned)kAlignWarps;
        }
        const bool drained = job >= (unsigned)a.nscans;
        if (drained) {
            if (HELP) {
                if (lane == 0) sts_volatile(&help_desk(warp)->active, 0u);   // releases this warp's helpers
                help_others<OV>(a.lv);
            }
            break;
        }
        ScanView v;
        v.pts = slot; v.n = 0;
        if (RANGES) {
            v.n = stage_ranges(a, job, slot, lane);   // SPEC 8: keep beams with range_min <= rho <= range_max, in beam order
        } else {
            const int src_scan = PAIRS ? __ldg(a.pairs + 2 * (size_t)job + 1) : a.job_scan ? __ldg(a.job_scan + job) : (int)job;
            int64_t o0 = src_scan >= 0 ? __ldg(a.offsets + src_scan) : 0, o1 = src_scan >= 0 ? __ldg(a.offsets + src_scan + 1) : 0;
            v.n = (int)(o1 - o0);
            const float2 *src = a.xy + o0;
            if (STAGED) {
                for (int i = lane; i < v.n; i += 32) slot[i] = sanitize(__ldg(src + i));
            } else {
                v.pts = src;
            }
        }
        if (SM) {
            const int npad = (v.n + 63) & ~63;
            for (int i = v.n + lane; i < npad; i += 32) slot[i] = far;
            __syncwarp();
        }
        if (lane < 3) ws->p[lane] = __ldg(a.init + 3 * (size_t)job + lane);
        __syncwarp();
        int evals = 0, status = NDT2D_NO_OVERLAP;
        const LevelDev *levels = PAIRS ? a.geo + (size_t)__ldg(a.pairs + 2 * (size_t)job) * a.nlevels : a.lv;
        for (int l = 0; l < a.nlevels; ++l) status = align_level<OV, SM, PAIRS ? TABLE_GHASH : TABLE_DENSE, HELP>(levels + l, a.prm, v, ws, evals, l);
        if (lane == 0) write_result(*ws, evals, status, a.res + job);
        __syncwarp(); // the slot is rewritten by the next job
    }
}

// ------------------------------------------------------------------------------------------------
// (3) top-k of the sweep scores: k passes of a grid-wide arg-max (ties to the smaller index)
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ bool better(double s1, long long i1, double s2, long long i2)
{
    // order by (-score, index); an empty candidate has index -1
    if (i2 < 0) return i1 >= 0;
    if (i1 < 0) return false;
    return (s1 > s2) || (s1 == s2 && i1 < i2);
}

// scratch layout: [0] ticket counter, then per block {score bits, index}
// pub.world > 0 (multi-GPU sweep): the finishing warp also stores the winner into row pub.row, column pub.rank of
// every rank's exchange table - lane r writes to rank r over NVLink (or locally for r == rank) - record first, a
// system-scope fence, then the epoch that tells the reader the record is complete.
__global__ void __launch_bounds__(256) k_argmax_pass(const double *__restrict__ scores, int64_t n, int pass,
                                                     int64_t *__restrict__ best_idx, double *__restrict__ best_val,
                                                     unsigned long long *__restrict__ scratch, const PublishArgs pub)
{
    __shared__ double s_val[8];
    __shared__ long long s_idx[8];
    __shared__ bool s_last;
    double bv = 0.0;
    long long bi = -1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        bool taken = false;
        for (int t = 0; t < pass; ++t) taken |= (best_idx[t] == i);
        double v = scores[i];
        if (!taken && !(v != v) && better(v, i, bv, bi)) { bv = v; bi = i; }
    }
    auto warp_best = [&]() {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double v2 = __shfl_xor_sync(FULL_MASK, bv, o);
            long long i2 = __shfl_xor_sync(FULL_MASK, bi, o);
            if (better(v2, i2, bv, bi)) { bv = v2; bi = i2; }
        }
    };
    warp_best();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_val[warp] = bv; s_idx[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        bv = lane < 8 ? s_val[lane] : 0.0;
        bi = lane < 8 ? s_idx[lane] : -1;
        warp_best();
        if (lane == 0) {
            scratch[1 + 2 * blockIdx.x] = (unsigned long long)__double_as_longlong(bv);
            scratch[2 + 2 * blockIdx.x] = (unsigned long long)bi;
            __threadfence();
            unsigned long long ticket = atomicAdd(scratch, 1ull);
            s_last = (ticket == (unsigned long long)gridDim.x - 1ull);
        }
    }
    __syncthreads();
    if (s_last && warp == 0) {
        __threadfence();
        bv = 0.0;
        bi = -1;
        for (int b = lane; b < (int)gridDim.x; b += 32) {
            double v = __longlong_as_double((long long)scratch[1 + 2 * b]);
            long long i = (long long)scratch[2 + 2 * b];
            if (better(v, i, bv, bi)) { bv = v; bi = i; }
        }
        warp_best();
        if (lane == 0) {
            best_idx[pass] = bi;
            best_val[pass] = bi >= 0 ? bv : 0.0;
            scratch[0] = 0ull; // ready for the next pass
        }
        if (lane < pub.world) {
            ndt2d_best *dst = pub.table[lane] + (size_t)pub.row * pub.world + pub.rank;
            dst->index = bi >= 0 ? bi + pub.index_offset : -1;
            dst->score = bi >= 0 ? bv : 0.0;
            __threadfence_system();
            *reinterpret_cast<volatile unsigned long long *>(&dst->epoch) = pub.epoch;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------

static inline int grid_for(int64_t items, int per_block, int sm_count, int blocks_per_sm)
{
    int64_t need = (items + per_block - 1) / per_block;
    int64_t cap = (int64_t)sm_count * blocks_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

// calls f(std::integral_constant<int, SRC>()) for the kind of target source
template <class F>
static cudaError_t with_src(const TargetSrc &s, F f)
{
    if (!s.pose) return f(std::integral_constant<int, SRC_POINTS>());
    if (s.ranges) return f(std::integral_constant<int, SRC_RANGES>());
    return f(std::integral_constant<int, SRC_SCANS>());
}

cudaError_t launch_pose_table(const LaunchCfg &c, const double *d_poses, int nscans, double *d_table, int64_t *launches)
{
    if (nscans <= 0) return cudaSuccess;
    k_pose_table<<<(nscans + 127) / 128, 128, 0, c.stream>>>(d_poses, nscans, d_table);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_build(const LaunchCfg &c, const LevelSet &S, const ndt2d_params &p, const TargetSrc &src, bool touch, int64_t *launches)
{
    if (touch) {
        cudaError_t e = cudaMemsetAsync(S.nlist, 0, (size_t)S.nlevels * sizeof(unsigned), c.stream);
        if (e != cudaSuccess) return e;
    }
    if (src.n > 0) {
        const dim3 grid(grid_for(src.n, 256, c.sm_count, 8), S.nlevels);
        cudaError_t e = with_src(src, [&](auto mode) {
            constexpr int SRC = decltype(mode)::value;
            auto kern = S.lv[0].ov ? (touch ? k_accumulate<1, true, SRC> : k_accumulate<1, false, SRC>)
                                   : (touch ? k_accumulate<0, true, SRC> : k_accumulate<0, false, SRC>);
            kern<<<grid, 256, 0, c.stream>>>(S, src);
            return cudaGetLastError();
        });
        if (e != cudaSuccess) return e;
        ++*launches;
    }
    // as many threads as touched cells at most (K per point), or as cells in the largest level
    int64_t items = 1;
    if (touch) items = src.n * (S.lv[0].ov ? 4 : 1);
    else for (int l = 0; l < S.nlevels; ++l) items = std::max<int64_t>(items, (int64_t)S.lv[l].njx * S.lv[l].njy);
    auto fin = touch ? k_finalize<true> : k_finalize<false>;
    fin<<<dim3(grid_for(items, 256, c.sm_count, 8), S.nlevels), 256, 0, c.stream>>>(S, p.min_points, p.eig_ratio);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_cell_index(const LaunchCfg &c, const LevelDev &L, const float2 *d_xy, int n, const double *d_pose,
                              int32_t *d_idx, int64_t *launches)
{
    if (n <= 0) return cudaSuccess;
    k_cell_index<<<(n + 255) / 256, 256, 0, c.stream>>>(L, d_xy, n, d_pose, d_idx);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_point_terms(const LaunchCfg &c, const LevelDev &L, const float2 *d_xy, int n, const double *d_pose,
                               float *d_terms, int64_t *launches)
{
    if (n <= 0) return cudaSuccess;
    if (L.ov) k_point_terms<1><<<(n + 127) / 128, 128, 0, c.stream>>>(L, d_xy, n, d_pose, d_terms);
    else k_point_terms<0><<<(n + 127) / 128, 128, 0, c.stream>>>(L, d_xy, n, d_pose, d_terms);
    ++*launches;
    return cudaGetLastError();
}

template <int OV, bool FULL, bool F32POSE>
static cudaError_t launch_eval_t(const LaunchCfg &c, const LevelDev &L, const float2 *d_xy, int n, const void *d_poses,
                                 int64_t npose, double *d_out, int out_stride, int32_t *d_count)
{
    size_t smem = (size_t)((n + 63) & ~63) * (FULL ? sizeof(float2) : sizeof(double2));   // score only: points staged as f64
    int grid = grid_for(npose, EVAL_THREADS / 32, c.sm_count, FULL ? EVAL_BLOCKS_FULL : EVAL_BLOCKS);
    if (smem <= (size_t)c.max_smem_optin - 1024) {
        auto kern = k_eval_poses<OV, FULL, F32POSE, true>;
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<grid, EVAL_THREADS, smem, c.stream>>>(L, d_xy, n, d_poses, npose, d_out, out_stride, d_count);
    } else {
        k_eval_poses<OV, FULL, F32POSE, false><<<grid, EVAL_THREADS, 0, c.stream>>>(L, d_xy, n, d_poses, npose, d_out,
                                                                                   out_stride, d_count);
    }
    return cudaGetLastError();
}

cudaError_t launch_eval_poses(const LaunchCfg &c, const LevelDev &L, const float2 *d_xy, int n, const void *d_poses,
                              int poses_f32, int64_t npose, int full, double *d_out, int out_stride, int32_t *d_count,
                              int64_t *launches)
{
    if (npose <= 0) return cudaSuccess;
    ++*launches;
    if (L.ov) {
        if (full) return poses_f32 ? launch_eval_t<1, true, true>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count)
                                   : launch_eval_t<1, true, false>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count);
        return poses_f32 ? launch_eval_t<1, false, true>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count)
                         : launch_eval_t<1, false, false>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count);
    }
    if (full) return poses_f32 ? launch_eval_t<0, true, true>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count)
                               : launch_eval_t<0, true, false>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count);
    return poses_f32 ? launch_eval_t<0, false, true>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count)
                     : launch_eval_t<0, false, false>(c, L, d_xy, n, d_poses, npose, d_out, out_stride, d_count);
}

// dynamic shared memory of one k_align block whose warps stage scans of up to cap_points points (0: no staging)
size_t align_smem_bytes(int cap_points, bool help)
{
    return (cap_points > 0 ? (size_t)cap_points * sizeof(float2) : 0) * (ALIGN_THREADS / 32) +
           (ALIGN_THREADS / 32) * (sizeof(WarpState) + (help ? sizeof(HelpDesk) : 0));
}

template <int OV, bool STAGED, bool RANGES, bool PAIRS = false, bool HELP = false>
static cudaError_t launch_align_t(const LaunchCfg &c, const AlignArgs &a)
{
    auto kern = k_align<OV, STAGED, RANGES, PAIRS, HELP>;
    size_t smem = align_smem_bytes((STAGED || RANGES) ? a.cap_points : 0, HELP);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    if (smem > 4096) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
    }
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, ALIGN_THREADS, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    // HELP: one block per scan while blocks are free (its other warps start as helpers); the first scans are dealt out
    // warp 0 of every block first
    int grid = grid_for(a.nscans, HELP ? 1 : ALIGN_THREADS / 32, c.sm_count, per_sm);
    kern<<<grid, ALIGN_THREADS, smem, c.stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_align(const LaunchCfg &c, const AlignArgs &a, int64_t *launches)
{
    if (a.nscans <= 0) return cudaSuccess;
    if (!a.counter_is_zero) {
        cudaError_t e = cudaMemsetAsync(a.counter, 0, sizeof(unsigned int), c.stream);
        if (e != cudaSuccess) return e;
    }
    ++*launches;
    const bool ranges = (a.ranges != nullptr);
    const bool staged = a.cap_points > 0;
    // few scans: latency matters, not throughput - one block per scan (k_align_block) if its factor buffer fits
    // (tools/midsize_probe.py: the block form wins up to ~1250 scans on a 148-SM part, four resident blocks per SM)
    if (staged && !a.pairs && a.nscans <= (c.block_align_max >= 0 ? c.block_align_max : 8 * c.sm_count)) {
        const int NC = a.prm.overlap ? 4 : 1;
        const size_t smem = sizeof(WarpState) + (size_t)a.cap_points * sizeof(float2) +
                            (size_t)(a.cap_points / 64) * NC * FACTOR_WORDS * 32 * sizeof(u64);
        if (smem <= (size_t)c.max_smem_optin) {
            cudaError_t e2 = cudaSuccess;
            auto kern = a.prm.overlap ? (ranges ? k_align_block<1, true> : k_align_block<1, false>)
                                      : (ranges ? k_align_block<0, true> : k_align_block<0, false>);
            if (smem > 48 * 1024) e2 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e2 != cudaSuccess) return e2;
            kern<<<a.nscans, BLOCK_ALIGN_THREADS, smem, c.stream>>>(a);
            return cudaGetLastError();
        }
    }
    if (a.pairs) {
        if (a.prm.overlap) return staged ? launch_align_t<1, true, false, true>(c, a) : launch_align_t<1, false, false, true>(c, a);
        return staged ? launch_align_t<0, true, false, true>(c, a) : launch_align_t<0, false, false, true>(c, a);
    }
    if (a.prm.overlap) {
        if (ranges) return launch_align_t<1, true, true>(c, a);
        return staged ? launch_align_t<1, true, false>(c, a) : launch_align_t<1, false, false>(c, a);
    }
    // K = 1, scans in shared memory: the helper-warp form (c.align_help: 0 never, 1 always, -1 = batches whose tail matters)
    const bool help = c.align_help > 0 || (c.align_help < 0 && (a.batch_scans > 0 ? a.batch_scans : a.nscans) <= HELP_MAX_SCANS);
    if (ranges) return help ? launch_align_t<0, true, true, false, true>(c, a) : launch_align_t<0, true, true>(c, a);
    if (staged) return help ? launch_align_t<0, true, false, false, true>(c, a) : launch_align_t<0, true, false>(c, a);
    return launch_align_t<0, false, false>(c, a);
}

cudaError_t launch_topk(const LaunchCfg &c, const double *d_scores, int64_t nhyp, int k, int64_t *d_idx, double *d_val,
                        unsigned long long *d_scratch, int64_t *launches, const PublishArgs *pub)
{
    int grid = grid_for(nhyp, 256 * 4, c.sm_count, 4);
    cudaError_t e = cudaMemsetAsync(d_scratch, 0, sizeof(unsigned long long), c.stream);
    if (e != cudaSuccess) return e;
    PublishArgs none;
    memset(&none, 0, sizeof(none));
    for (int pass = 0; pass < k; ++pass) {
        k_argmax_pass<<<grid, 256, 0, c.stream>>>(d_scores, nhyp, pass, d_idx, d_val, d_scratch, (pub && pass == 0) ? *pub : none);
        ++*launches;
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

int topk_scratch_words(int sm_count) { return 1 + 2 * sm_count * 4; }

// One block: thread (r, j) builds candidate j - global index, sweep score, refined record - and stores it into rank r's table
// (NVLink peer stores, or local for the own rank); after every thread's system-scope fence and a block barrier, thread r
// stores the epoch of its rank's block: a reader that sees the epoch sees the k candidates.
__global__ void __launch_bounds__(256) k_publish_candidates(const int64_t *__restrict__ best_idx, const double *__restrict__ best_score,
                                                            const ndt2d_result *__restrict__ res, const CandidatePublishArgs pub)
{
    for (int t = threadIdx.x; t < pub.world * pub.k; t += blockDim.x) {
        const int r = t / pub.k, j = t % pub.k;
        ndt2d_candidate *dst = pub.table[r] + j;
        const long long i = best_idx[j];
        dst->index = i >= 0 ? i + pub.index_offset : -1;
        dst->sweep_score = i >= 0 ? best_score[j] : 0.0;
        dst->reserved = 0ull;
        dst->refined = res[j];
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < pub.world) {
        __threadfence_system();
        *reinterpret_cast<volatile unsigned long long *>(&pub.table[threadIdx.x]->epoch) = pub.epoch;
    }
}

cudaError_t launch_publish_candidates(const LaunchCfg &c, const int64_t *d_best_idx, const double *d_best_score, const ndt2d_result *d_res,
                                      const CandidatePublishArgs &pub, int64_t *launches)
{
    k_publish_candidates<<<1, 256, 0, c.stream>>>(d_best_idx, d_best_score, d_res, pub);
    ++*launches;
    return cudaGetLastError();
}

__global__ void k_topk_to_jobs(const float *__restrict__ hyp, const int64_t *__restrict__ best_idx, int k, double *__restrict__ init,
                               int32_t *__restrict__ job_scan)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const int64_t i = best_idx[j];
    job_scan[j] = i >= 0 ? 0 : -1;
#pragma unroll
    for (int t = 0; t < 3; ++t) init[3 * j + t] = i >= 0 ? (double)__ldg(hyp + 3 * i + t) : 0.0;
}

cudaError_t launch_topk_to_jobs(const LaunchCfg &c, const float *d_hyp, const int64_t *d_best_idx, int k, double *d_init, int32_t *d_job_scan,
                                int64_t *launches)
{
    if (k <= 0) return cudaSuccess;
    k_topk_to_jobs<<<(k + 127) / 128, 128, 0, c.stream>>>(d_hyp, d_best_idx, k, d_init, d_job_scan);
    ++*launches;
    return cudaGetLastError();
}

// order-preserving float <-> int map so that integer atomicMin/atomicMax order floats
__host__ __device__ static inline int float_to_ordered(float f)
{
    int i;
#ifdef __CUDA_ARCH__
    i = __float_as_int(f);
#else
    memcpy(&i, &f, 4);
#endif
    return i >= 0 ? i : i ^ 0x7fffffff;
}

float bbox_decode(int v)
{
    int i = v >= 0 ? v : v ^ 0x7fffffff;
    float f;
    memcpy(&f, &i, 4);
    return f;
}

// auto-fit (SPEC 2, 7.2): bounding box of the finite points - of the f32 roundings of a posed scan point's map coordinates;
// min/max are order-independent
template <int SRC>
__global__ void __launch_bounds__(256) k_bbox(const TargetSrc src, int *__restrict__ box)
{
    float xmin = INFINITY, ymin = INFINITY, xmax = -INFINITY, ymax = -INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < src.n; i += (int64_t)gridDim.x * blockDim.x) {
        double X, Y;
        if (!target_point<SRC>(src, i, X, Y)) continue;
        const float x = (float)X, y = (float)Y;
        if (!isfinite(x) || !isfinite(y)) continue;
        xmin = fminf(xmin, x); xmax = fmaxf(xmax, x);
        ymin = fminf(ymin, y); ymax = fmaxf(ymax, y);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        xmin = fminf(xmin, __shfl_xor_sync(FULL_MASK, xmin, o));
        ymin = fminf(ymin, __shfl_xor_sync(FULL_MASK, ymin, o));
        xmax = fmaxf(xmax, __shfl_xor_sync(FULL_MASK, xmax, o));
        ymax = fmaxf(ymax, __shfl_xor_sync(FULL_MASK, ymax, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(box + 0, float_to_ordered(xmin));
        atomicMin(box + 1, float_to_ordered(ymin));
        atomicMax(box + 2, float_to_ordered(xmax));
        atomicMax(box + 3, float_to_ordered(ymax));
    }
}

cudaError_t launch_bbox(const LaunchCfg &c, const TargetSrc &src, int *d_box, int64_t *launches)
{
    int init[4] = {float_to_ordered(INFINITY), float_to_ordered(INFINITY), float_to_ordered(-INFINITY),
                   float_to_ordered(-INFINITY)};
    cudaError_t e = cudaMemcpyAsync(d_box, init, sizeof(init), cudaMemcpyHostToDevice, c.stream);
    if (e != cudaSuccess || src.n <= 0) return e;
    ++*launches;
    return with_src(src, [&](auto mode) {
        k_bbox<decltype(mode)::value><<<grid_for(src.n, 256 * 4, c.sm_count, 4), 256, 0, c.stream>>>(src, d_box);
        return cudaGetLastError();
    });
}

} // namespace ndt2d
