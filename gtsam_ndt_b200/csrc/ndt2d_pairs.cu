// ndt2d_align_pairs: batched scan-to-scan. One grid per target scan, built by one warp per (target, level) into a hash
// table (k_pairs_build, below); the pairs are then aligned by k_align in pairs mode (ndt2d_kernels.cu). The host side
// finds the distinct targets, sizes the tables and cuts the call into chunks that fit the table budget.
// Reference interface: none citable (/root/reference/README.md:1 is the whole mount).
#include "ndt2d_align.cuh"
#include "ndt2d_host.h"

namespace ndt2d {

static constexpr unsigned FULL_MASK = 0xffffffffu;

// Same arithmetic as the dense build (SPEC 2 auto-fit lattice, SPEC 3 integer sums and finalisation), so every record
// equals the one ndt2d_set_target(scan) would produce; only the container differs: a scan touches a few hundred of
// the cells of its bounding box, so the cells live in an open-addressing hash table keyed by the dense cell index.
static constexpr int PAIRS_LIST_CAP = 2304; // claimed-slot list per warp (u16 entries, 36 KB per block); longer: full-table scan

template <int OV>
__global__ void __launch_bounds__(256) k_pairs_build(const PairBuildArgs a)
{
    const int lane = threadIdx.x & 31;
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (wid >= (int64_t)a.ntargets * a.nlevels) return;
    const int t = (int)(wid / a.nlevels), l = (int)(wid % a.nlevels);
    // slots this warp claimed, so that the finalisation visits the few hundred occupied slots instead of the whole table
    __shared__ unsigned short s_list[8][PAIRS_LIST_CAP];
    __shared__ int s_nlist[8];
    const int w = threadIdx.x >> 5;
    if (lane == 0) s_nlist[w] = 0;
    const int scan = __ldg(a.targets + t);
    const int64_t o0 = __ldg(a.offsets + scan), o1 = __ldg(a.offsets + scan + 1);
    const int n = (int)(o1 - o0);
    const float2 *__restrict__ src = a.xy + o0;

    // SPEC 2 auto-fit: bounding box of the finite points (min and max are order independent)
    float xmin = INFINITY, ymin = INFINITY, xmax = -INFINITY, ymax = -INFINITY;
    if (!a.explicit_grid) {
        for (int i = lane; i < n; i += 32) {
            float2 p = __ldg(src + i);
            if (!isfinite(p.x) || !isfinite(p.y)) continue;
            xmin = fminf(xmin, p.x); xmax = fmaxf(xmax, p.x);
            ymin = fminf(ymin, p.y); ymax = fmaxf(ymax, p.y);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            xmin = fminf(xmin, __shfl_xor_sync(FULL_MASK, xmin, o));
            ymin = fminf(ymin, __shfl_xor_sync(FULL_MASK, ymin, o));
            xmax = fmaxf(xmax, __shfl_xor_sync(FULL_MASK, xmax, o));
            ymax = fmaxf(ymax, __shfl_xor_sync(FULL_MASK, ymax, o));
        }
    }
    // geometry, the f32 expressions of setup_level() in ndt2d_capi.cu (every lane computes the same values)
    LevelDev L;
    L.res = a.res[l];
    L.ov = a.ov;
    L.st = L.ov ? __fmul_rn(L.res, 0.5f) : L.res;
    L.inv_st = __fdiv_rn(1.0f, L.st);
    if (a.explicit_grid) {
        L.ox = a.gox; L.oy = a.goy;
        L.nhx = (int)ceilf(__fdiv_rn(a.gex, L.st));
        L.nhy = (int)ceilf(__fdiv_rn(a.gey, L.st));
    } else {
        if (!(xmin <= xmax)) { xmin = xmax = ymin = ymax = 0.0f; }
        L.ox = __fsub_rn(__fmul_rn(floorf(__fdiv_rn(xmin, L.res)), L.res), L.res);
        L.oy = __fsub_rn(__fmul_rn(floorf(__fdiv_rn(ymin, L.res)), L.res), L.res);
        L.nhx = (int)ceilf(__fdiv_rn(__fsub_rn(xmax, L.ox), L.st)) + 2;
        L.nhy = (int)ceilf(__fdiv_rn(__fsub_rn(ymax, L.oy), L.st)) + 2;
    }
    bool too_big = L.nhx < 1 || L.nhy < 1 || (int64_t)(L.nhx + L.ov) * (int64_t)(L.nhy + L.ov) >= ((int64_t)1 << 31);
    if (too_big) { L.nhx = L.nhy = 0; }      // nothing is inside: every align against this target ends NO_OVERLAP
    L.njx = L.nhx + L.ov;
    L.njy = L.nhy + L.ov;
    L.inv_std = __ddiv_rn(1.0, (double)L.st);
    L.qs = __ddiv_rn(4194304.0, (double)L.res);
    L.qu = __dmul_rn((double)L.res, 1.0 / 4194304.0);
    L.hash_mask = a.cap - 1u;
    float4 *rec = a.tab + (size_t)wid * ((size_t)a.cap + 1) * 2;
    uint32_t *cnt = a.cnt + (size_t)wid * a.cap;
    unsigned long long *sums = a.sums + (size_t)wid * a.cap * 5;
    L.cells = rec;
    L.cnt = cnt;
    L.sums = sums;
    if (lane == 0) {
        a.geo[wid] = L;
        if (too_big) atomicMax(a.error, t + 1);
    }

    // clear the records: empty key in every slot's `n` word; the sentinel record after the last slot
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 empty = make_float4(0.f, 0.f, __int_as_float((int)kEmptyKey), 0.f);
    for (unsigned s = lane; s <= a.cap; s += 32) {
        rec[2 * (size_t)s] = zero;
        rec[2 * (size_t)s + 1] = s < a.cap ? empty : zero;
    }
    // (cnt and sums are zero on entry: they are zeroed when allocated and every finalisation zeroes what it consumed)
    __syncwarp();

    // SPEC 3 accumulation, as k_accumulate: runs of equal cells are combined in the warp, run heads find or claim the
    // cell's slot (compare-and-swap on the key word) and add into its integer sums
    unsigned *keyword = reinterpret_cast<unsigned *>(rec);   // key of slot s = word 8 s + 6
    float2 pnext = lane < n ? __ldg(src + lane) : make_float2(0.f, 0.f);   // the next window's point is requested one window ahead
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const float2 p = pnext;
        if (i + 32 < n) pnext = __ldg(src + i + 32);
        accumulate_window<OV>(L, i < n, p.x, p.y, lane, [&](int key, unsigned c, long long sx, long long sy, long long sxx, long long sxy, long long syy) {
            unsigned s = hash_slot((unsigned)key, L.hash_mask);
            bool placed = false;
            // the table is at most 2/3 full by construction; the probe count is bounded all the same, so that
            // inconsistent arguments (offsets on the device that differ from the host copy) cannot hang the GPU
            for (unsigned probes = 0; probes <= L.hash_mask; ++probes) {
                unsigned was = atomicCAS(keyword + 8 * (size_t)s + 6, kEmptyKey, (unsigned)key);
                if (was == kEmptyKey) {
                    const int pos = atomicAdd(&s_nlist[w], 1);
                    if (pos < PAIRS_LIST_CAP) s_list[w][pos] = (unsigned short)s;
                    placed = true;
                    break;
                }
                if (was == (unsigned)key) { placed = true; break; }
                s = (s + 1u) & L.hash_mask;
            }
            if (!placed) { atomicMax(a.error, t + 1); return; }
            atomicAdd(cnt + s, c);
            unsigned long long *q = sums + 5 * (size_t)s;
            atomicAdd(q + 0, (unsigned long long)sx);
            atomicAdd(q + 1, (unsigned long long)sy);
            atomicAdd(q + 2, (unsigned long long)sxx);
            atomicAdd(q + 3, (unsigned long long)sxy);
            atomicAdd(q + 4, (unsigned long long)syy);
        });
    }
    __threadfence();
    __syncwarp();

    // SPEC 3 finalisation of the occupied slots; the key stays in the record's `n` word for the probing reader, and the
    // slot's sums go back to zero for the next build that uses this memory
    auto finish = [&](unsigned s) {
        const unsigned key = *(volatile unsigned *)(keyword + 8 * (size_t)s + 6);
        if (key == kEmptyKey) return;
        const unsigned nn = *(volatile uint32_t *)(cnt + s);
        volatile long long *q = reinterpret_cast<volatile long long *>(sums + 5 * (size_t)s);
        const long long q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3], q4 = q[4];
        float4 ra, rb;
        finalize_record(nn, q0, q1, q2, q3, q4, L.qu, a.min_points, a.eig_ratio, ra, rb);
        rb.z = __int_as_float((int)key);
        rec[2 * (size_t)s] = ra;
        rec[2 * (size_t)s + 1] = rb;
        cnt[s] = 0u;
        q[0] = 0; q[1] = 0; q[2] = 0; q[3] = 0; q[4] = 0;
    };
    const int nlist = s_nlist[w];
    if (nlist <= PAIRS_LIST_CAP) {
        for (int e = lane; e < nlist; e += 32) finish(s_list[w][e]);
    } else {
        for (unsigned s = lane; s < a.cap; s += 32) finish(s);
    }
}

// ------------------------------------------------------------------------------------------------
// fused path: one warp per pair, the target's grid in shared memory
// ------------------------------------------------------------------------------------------------

static constexpr int FUSED_WARPS_MAX = 8;        // warps per block: as many as let two blocks share an SM, at most this (5 at 1080-point scans)
static constexpr unsigned FUSED_WS_BYTES = 224;    // room for the WarpState (216 B)
static constexpr unsigned FUSED_STATE_BYTES = 352; // WarpState + LevelDev (112 B), rounded up to 16

// SPEC 2 geometry of one level of a target's grid from its bounding box: the f32 expressions of setup_level() in
// ndt2d_capi.cu (every lane computes the same values). Returns false when the lattice is unusable (empty or >= 2^31
// cells): nothing is inside then and every align against this target ends NO_OVERLAP.
__device__ __forceinline__ bool pair_level_geometry(LevelDev &L, float res, int ov, bool explicit_grid, float gox, float goy, float gex,
                                                    float gey, float xmin, float ymin, float xmax, float ymax)
{
    L.res = res;
    L.ov = ov;
    L.st = L.ov ? __fmul_rn(L.res, 0.5f) : L.res;
    L.inv_st = __fdiv_rn(1.0f, L.st);
    if (explicit_grid) {
        L.ox = gox; L.oy = goy;
        L.nhx = (int)ceilf(__fdiv_rn(gex, L.st));
        L.nhy = (int)ceilf(__fdiv_rn(gey, L.st));
    } else {
        if (!(xmin <= xmax)) { xmin = xmax = ymin = ymax = 0.0f; }
        L.ox = __fsub_rn(__fmul_rn(floorf(__fdiv_rn(xmin, L.res)), L.res), L.res);
        L.oy = __fsub_rn(__fmul_rn(floorf(__fdiv_rn(ymin, L.res)), L.res), L.res);
        L.nhx = (int)ceilf(__fdiv_rn(__fsub_rn(xmax, L.ox), L.st)) + 2;
        L.nhy = (int)ceilf(__fdiv_rn(__fsub_rn(ymax, L.oy), L.st)) + 2;
    }
    const bool bad = L.nhx < 1 || L.nhy < 1 || (int64_t)(L.nhx + L.ov) * (int64_t)(L.nhy + L.ov) >= ((int64_t)1 << 31);
    if (bad) { L.nhx = L.nhy = 0; }
    L.njx = L.nhx + L.ov;
    L.njy = L.nhy + L.ov;
    L.inv_std = __ddiv_rn(1.0, (double)L.st);
    L.qs = __ddiv_rn(4194304.0, (double)L.res);
    L.qu = __dmul_rn((double)L.res, 1.0 / 4194304.0);
    return !bad;
}

// SPEC 3 for one (target scan, level) by ONE warp, entirely in its shared-memory slice. The integer sums are order
// independent, so grouping the points by cell with a sort and summing each group in one lane gives the sums - and
// therefore the records - of the dense build bit for bit. Steps: (1) cell key of every point (one past the last cell
// for a point outside the lattice); (2) LSD radix sort of the point indices by key, 8 bits per pass, only as many passes
// as the lattice has key bits; (3) run heads = the cells; (4) one lane per cell with at least min_points points: integer
// sums over its points, finalisation, 24-byte record appended to the compact array (so the records are in key order),
// and (key tag, record id) entered into the bucket index: first bucket from hash_slot(key) with a free entry, conflicts
// between the lanes of a round resolved inside the warp, no atomics. Returns the number of records.
// Shared memory: keyof[cap_t] u32, two index buffers of cap_t + 2 u16 (ping-pong; the idle one holds the run heads
// afterwards), the record area (the radix histogram lives there during the sort) and the slot index.
__device__ __noinline__ int build_table_shared(const LevelDev *Lp, const float2 *__restrict__ src, int n, int min_points, double eig_ratio,
                                               unsigned *keyof, unsigned cap_t, float *rec, unsigned *hidx, unsigned hslots)
{
    const LevelDev &L = *Lp;
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    // the two index buffers, selected by pointer arithmetic: as an array of two pointers indexed by `cur` the compiler kept them in
    // local memory and went through generic loads and stores in the sort loops (r2z profile: 14 % of the kernel's samples there)
    unsigned short *const perm0 = reinterpret_cast<unsigned short *>(keyof + cap_t);
    const unsigned perm_stride = cap_t + 2;
    auto perm_of = [&](int which) { return perm0 + (which ? perm_stride : 0u); };
    unsigned *hist = reinterpret_cast<unsigned *>(rec);     // 256 counters; the record area is not in use during the sort
    const unsigned ncells = (unsigned)L.njx * (unsigned)L.njy;
    // (1) keys; four windows of points are requested at a time (a warp has no other latency hiding here)
    int m = 0;
#pragma unroll 1
    for (int base = 0; base < n; base += 128) {
        float2 pw[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + 32 * u + lane;
            pw[u] = i < n ? __ldg(src + i) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + 32 * u + lane;
            int hx = 0, hy = 0;
            const bool in = i < n && lattice_of_point(L, pw[u].x, pw[u].y, hx, hy);
            if (i < n) {
                keyof[i] = in ? (unsigned)(hy * L.njx + hx) : ncells;
                perm0[i] = (unsigned short)i;
            }
            m += __popc(__ballot_sync(FULL_MASK, in));
        }
    }
    __syncwarp();
    if (m == 0) {
        for (unsigned s = lane; s < hslots; s += 32) hidx[s] = 0xffffffffu;
        if (lane < 6) rec[lane] = lane == 5 ? __int_as_float(-1) : 0.0f;      // no records: an empty index and the zero record
        __syncwarp();
        return 0;
    }
    // (2) radix sort of the indices by key (keys 0 .. ncells)
    const int nbits = 32 - __clz(ncells);
    int cur = 0;
#pragma unroll 1
    for (int shift = 0; shift < nbits; shift += 8) {
        const unsigned short *const pin = perm_of(cur);
        unsigned short *const pout = perm_of(cur ^ 1);
        for (int b = lane; b < 256; b += 32) hist[b] = 0u;
        __syncwarp();
#pragma unroll 2
        for (int i = lane; i < n; i += 32) atomicAdd(&hist[(keyof[pin[i]] >> shift) & 255u], 1u);
        __syncwarp();
        unsigned c[8], sum = 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j) { c[j] = hist[8 * lane + j]; sum += c[j]; }
        unsigned incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(FULL_MASK, incl, o);
            if (lane >= o) incl += v;
        }
        unsigned run = incl - sum;
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; ++j) { hist[8 * lane + j] = run; run += c[j]; }
        __syncwarp();
#pragma unroll 1
        for (int base = 0; base < n; base += 32) {      // windows in order: the scatter is stable
            const int i = base + lane;
            const bool valid = i < n;
            const unsigned short ix = valid ? pin[i] : (unsigned short)0;
            const unsigned d = valid ? (keyof[ix] >> shift) & 255u : 256u + (unsigned)lane;
            const unsigned peers = __match_any_sync(FULL_MASK, d);
            const unsigned rank = __popc(peers & lt);
            const unsigned off = valid ? hist[d] : 0u;
            __syncwarp();
            if (valid && rank == 0u) hist[d] = off + __popc(peers);
            __syncwarp();
            if (valid) pout[off + rank] = ix;
        }
        __syncwarp();
        cur ^= 1;
    }
    // (3) run heads among the m points inside the lattice (they come first: the outside key is the largest)
    const unsigned short *order = perm_of(cur);
    unsigned short *hpos = perm_of(cur ^ 1);
    int nruns = 0;
#pragma unroll 1
    for (int base = 0; base < m; base += 32) {
        const int i = base + lane;
        const bool head = i < m && (i == 0 || keyof[order[i]] != keyof[order[i - 1]]);
        const unsigned mask = __ballot_sync(FULL_MASK, head);
        if (head) hpos[nruns + __popc(mask & lt)] = (unsigned short)i;
        nruns += __popc(mask);
    }
    if (lane == 0) hpos[nruns] = (unsigned short)m;
    __syncwarp();
    // the cells with at least min_points points, compacted (start | length << 16): the index area is free until (4b)
    int nvalid = 0;
#pragma unroll 1
    for (int base = 0; base < nruns; base += 32) {
        const int r = base + lane;
        const int start = r < nruns ? (int)hpos[r] : 0;
        const int len = r < nruns ? (int)hpos[r + 1] - start : 0;
        const bool ok = len >= min_points;
        const unsigned mask = __ballot_sync(FULL_MASK, ok);
        if (ok) hidx[nvalid + __popc(mask & lt)] = (unsigned)start | ((unsigned)len << 16);
        nvalid += __popc(mask);
    }
    __syncwarp();
    // (4a) one lane per cell: integer sums over its points, finalisation, record
    int nrec = 0;
#pragma unroll 1
    for (int base = 0; base < nvalid; base += 32) {
        const int v = base + lane;
        const bool ok = v < nvalid;
        const unsigned sl = ok ? hidx[v] : 0u;
        const int start = (int)(sl & 0xffffu), len = (int)(sl >> 16);
        unsigned kr = 0u;
        float4 ra = make_float4(0.f, 0.f, 0.f, 0.f), rb = ra;
        if (ok) {
            kr = keyof[order[start]];
            const int jx = (int)(kr % (unsigned)L.njx), jy = (int)(kr / (unsigned)L.njx);
            const double cx = (double)L.ox + ((double)(jx - L.ov)) * (double)L.st + 0.5 * (double)L.res;
            const double cy = (double)L.oy + ((double)(jy - L.ov)) * (double)L.st + 0.5 * (double)L.res;
            long long s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0;
#pragma unroll 1
            for (int p = start; p < start + len; p += 4) {      // four independent loads per trip (L2 round trips overlap)
                float2 pt[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) pt[u] = __ldg(src + order[min(p + u, start + len - 1)]);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (p + u < start + len) {
                        const double dx = (double)pt[u].x - cx, dy = (double)pt[u].y - cy;
                        const long long qx = __double2ll_rn(dx * L.qs), qy = __double2ll_rn(dy * L.qs);
                        s0 += qx; s1 += qy; s2 += qx * qx; s3 += qx * qy; s4 += qy * qy;
                    }
                }
            }
            finalize_record((unsigned)len, s0, s1, s2, s3, s4, L.qu, min_points, eig_ratio, ra, rb);
        }
        const bool keep = ok && rb.w != 0.0f;               // a degenerate cell (SPEC 3: l1 <= 1e-10) stays invalid: no record
        const unsigned mask = __ballot_sync(FULL_MASK, keep);
        const unsigned id = (unsigned)nrec + __popc(mask & lt);
        if (keep) {
            float *o = rec + 6 * (size_t)id;                 // {mux, muy, B00, B01, B11, key}
            o[0] = ra.x; o[1] = ra.y; o[2] = ra.z; o[3] = ra.w; o[4] = rb.y; o[5] = __int_as_float((int)kr);
        }
        nrec += __popc(mask);
    }
    __syncwarp();
    // (4b) the bucket index (lookup_shared in ndt2d_device.cuh): every pending lane counts the used entries of its bucket; the
    // lanes of a round that want the same bucket take its free entries in lane order, the rest move on by one bucket
    for (unsigned s = lane; s < hslots; s += 32) hidx[s] = 0xffffffffu;
    __syncwarp();
    const unsigned bmask = hslots / 4u - 1u;
#pragma unroll 1
    for (int base = 0; base < nrec; base += 32) {
        const unsigned id = (unsigned)(base + lane);
        bool pending = id < (unsigned)nrec;
        const unsigned kr = pending ? (unsigned)__float_as_int(rec[6 * (size_t)id + 5]) : 0u;
        unsigned b = hash_slot(kr, bmask);
        while (__any_sync(FULL_MASK, pending)) {
            unsigned used = 0u;
            if (pending) {
#pragma unroll
                for (int j = 0; j < 4; ++j) used += hidx[4u * b + j] != 0xffffffffu ? 1u : 0u;
            }
            const unsigned peers = __match_any_sync(FULL_MASK, pending ? b : 0x100000u + (unsigned)lane);
            const unsigned pos = used + __popc(peers & lt);
            const bool win = pending && pos < 4u;
            __syncwarp();
            if (win) hidx[4u * b + pos] = ((kr & 0x7fffu) << 16) | id;
            __syncwarp();
            if (win) pending = false;
            else if (pending) b = (b + 1u) & bmask;
        }
    }
    // the all-zero record behind the compact array: what a failed lookup loads (finite factors, valid = 0)
    if (lane < 6) rec[6 * (size_t)nrec + lane] = lane == 5 ? __int_as_float(-1) : 0.0f;
    __syncwarp();
    return nrec;
}

__global__ void __launch_bounds__(FUSED_WARPS_MAX * 32) k_pairs_fused(const __grid_constant__ PairFusedArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char *slice = smem_raw + (size_t)warp * a.warp_bytes;
    WarpState *ws = reinterpret_cast<WarpState *>(slice);
    LevelDev *Ls = reinterpret_cast<LevelDev *>(slice + FUSED_WS_BYTES);
    unsigned *area_a = reinterpret_cast<unsigned *>(slice + a.off_a);
    float2 *slot = reinterpret_cast<float2 *>(slice + a.off_a);
    float *rec = reinterpret_cast<float *>(slice + a.off_r);
    unsigned *hidx = reinterpret_cast<unsigned *>(slice + a.off_h);
    const float2 far = make_float2(1e18f, 1e18f);
    for (;;) {
        unsigned job = 0;
        if (lane == 0) job = atomicAdd(a.counter, 1u);
        job = __shfl_sync(FULL_MASK, job, 0);
        if (job >= (unsigned)a.npairs) break;
        const int tscan = __ldg(a.pairs + 2 * (size_t)job), sscan = __ldg(a.pairs + 2 * (size_t)job + 1);
        const int64_t t0 = __ldg(a.offsets + tscan), t1 = __ldg(a.offsets + tscan + 1);
        const int64_t s0 = __ldg(a.offsets + sscan), s1 = __ldg(a.offsets + sscan + 1);
        const int tn = (int)(t1 - t0), sn = (int)(s1 - s0);
        const float2 *__restrict__ tsrc = a.xy + t0;
        const float2 *__restrict__ ssrc = a.xy + s0;
        // SPEC 2 auto-fit: bounding box of the target's finite points
        float xmin = INFINITY, ymin = INFINITY, xmax = -INFINITY, ymax = -INFINITY;
        if (!a.explicit_grid) {
            for (int base = 0; base < tn; base += 128) {
                float2 pw[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int i = base + 32 * u + lane;
                    pw[u] = i < tn ? __ldg(tsrc + i) : make_float2(NAN, NAN);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (!isfinite(pw[u].x) || !isfinite(pw[u].y)) continue;
                    xmin = fminf(xmin, pw[u].x); xmax = fmaxf(xmax, pw[u].x);
                    ymin = fminf(ymin, pw[u].y); ymax = fmaxf(ymax, pw[u].y);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                xmin = fminf(xmin, __shfl_xor_sync(FULL_MASK, xmin, o));
                ymin = fminf(ymin, __shfl_xor_sync(FULL_MASK, ymin, o));
                xmax = fmaxf(xmax, __shfl_xor_sync(FULL_MASK, xmax, o));
                ymax = fmaxf(ymax, __shfl_xor_sync(FULL_MASK, ymax, o));
            }
        }
        if (lane < 3) ws->p[lane] = __ldg(a.init + 3 * (size_t)job + lane);
        __syncwarp();
        int evals = 0, status = NDT2D_NO_OVERLAP;
        for (int l = 0; l < a.nlevels; ++l) {
            LevelDev L;
            const bool usable = pair_level_geometry(L, a.res_m[l], 0, a.explicit_grid != 0, a.gox, a.goy, a.gex, a.gey, xmin, ymin, xmax, ymax);
            L.cells = reinterpret_cast<const float4 *>(rec); // TABLE_SHASH: the compact array of 24-byte records
            L.cnt = hidx;                                    //              and the bucket index
            L.sums = nullptr;
            L.hash_mask = a.hslots / 4u - 1u;
            L.zero_rec = 0u;
            if (!usable && lane == 0) atomicMax(a.error, (int)job + 1);
            __syncwarp();                                    // the previous level's evaluation has finished with *Ls
            if (lane == 0) *Ls = L;
            __syncwarp();
            const int nrec = build_table_shared(Ls, tsrc, tn, a.prm.min_points, a.prm.eig_ratio, area_a, a.cap_t, rec, hidx, a.hslots);
            if (lane == 0) Ls->zero_rec = (unsigned)nrec;
            // the sort buffers are dead: the same area takes the source scan (sanitised, padded with the far-away point)
            const int npad = (sn + 63) & ~63;
#pragma unroll 4
            for (int i = lane; i < npad; i += 32) slot[i] = i < sn ? sanitize(__ldg(ssrc + i)) : far;
            __syncwarp();
            status = lm_level<WarpScope>(a.prm, sn, ws, evals, [&]() { eval_to_smem<0, true, TABLE_SHASH>(Ls, slot, sn, ws); });
        }
        if (lane == 0) write_result(*ws, evals, status, a.res + job);
        __syncwarp();
    }
}

bool pairs_fused_layout(PairFusedArgs &a, int64_t max_target_points, int64_t max_source_points, int smem_optin)
{
    if (max_target_points > 65533 || max_source_points > (1 << 20)) return false;
    a.cap_t = (unsigned)((std::max<int64_t>(max_target_points, 1) + 31) & ~(int64_t)31);
    a.cap_s = (unsigned)((std::max<int64_t>(max_source_points, 1) + 63) & ~(int64_t)63);
    a.rmax = (unsigned)(a.cap_t / (unsigned)std::max(a.prm.min_points, 2)) + 1u;
    a.hslots = 64;                                                  // four entries per bucket; buckets >= 0.7 * rmax
    while (a.hslots < 4u * ((7u * a.rmax + 9u) / 10u)) a.hslots <<= 1;
    if (a.rmax > 65534u || a.hslots > 4u * 65536u) return false;  // record ids are 16 bits; hash_slot() yields 17 bits
    auto up16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    const size_t size_a = up16(std::max<size_t>((size_t)a.cap_s * 8, (size_t)a.cap_t * 4 + 2 * ((size_t)a.cap_t + 2) * 2));
    const size_t size_r = up16(std::max<size_t>(((size_t)a.rmax + 1) * 24, 1024));      // records + the zero record; the radix histogram
    a.off_a = FUSED_STATE_BYTES;
    a.off_r = (unsigned)(a.off_a + size_a);
    a.off_h = (unsigned)(a.off_r + size_r);
    a.warp_bytes = (unsigned)up16(a.off_h + (size_t)a.hslots * 4);
    static_assert(sizeof(WarpState) <= FUSED_WS_BYTES && sizeof(LevelDev) <= FUSED_STATE_BYTES - FUSED_WS_BYTES, "per-warp state area");
    // two blocks per SM (each gets half of the opt-in limit minus the 1 KB the driver reserves per block)
    a.warps_per_block = (unsigned)std::min<size_t>(FUSED_WARPS_MAX, ((size_t)smem_optin / 2 - 1024) / a.warp_bytes);
    return a.warps_per_block >= 2;
}

cudaError_t launch_pairs_fused(const LaunchCfg &c, const PairFusedArgs &a, int64_t *launches)
{
    if (a.npairs <= 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(a.counter, 0, sizeof(unsigned int), c.stream);
    if (e != cudaSuccess) return e;
    const int wpb = (int)a.warps_per_block;
    const size_t smem = (size_t)a.warp_bytes * wpb;
    if (smem > 48 * 1024) {
        e = cudaFuncSetAttribute(k_pairs_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    e = cudaFuncSetAttribute(k_pairs_fused, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pairs_fused, wpb * 32, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    const int64_t need = ((int64_t)a.npairs + wpb - 1) / wpb;
    const int64_t cap = (int64_t)c.sm_count * per_sm;
    k_pairs_fused<<<(int)std::min(need, cap), wpb * 32, smem, c.stream>>>(a);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_pairs_build(const LaunchCfg &c, const PairBuildArgs &a, int64_t *launches)
{
    const int64_t warps = (int64_t)a.ntargets * a.nlevels;
    if (warps <= 0) return cudaSuccess;
    const int grid = (int)((warps + 7) / 8);
    if (a.ov) k_pairs_build<1><<<grid, 256, 0, c.stream>>>(a);
    else k_pairs_build<0><<<grid, 256, 0, c.stream>>>(a);
    ++*launches;
    return cudaGetLastError();
}

} // namespace ndt2d

using namespace ndt2d;

extern "C" {

// ---- batched scan-to-scan (north_star stage 3, "batched multi-scan"): many (target scan, source scan) pairs per call ----

static unsigned next_pow2(unsigned v)
{
    unsigned p = 1;
    while (p < v) p <<= 1;
    return p;
}

// d_xy / d_offsets / d_init / d_res: device; h_offsets / pairs: host (the chunking and the target list are host work).
// One chunk = as many pairs as fit the table budget. Asynchronous on the handle's stream apart from the uploads of the
// small per-chunk index lists; *err_out (optional) receives the device error flag after a synchronisation.
static int align_pairs_impl(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, const int64_t *h_offsets, int nscans,
                            const int32_t *pairs, int npairs, const double *d_init, ndt2d_result *d_res)
{
    int64_t max_src = 0, max_tgt = 0;
    for (int p = 0; p < npairs; ++p) {
        const int t = pairs[2 * p], s = pairs[2 * p + 1];
        if (t < 0 || t >= nscans || s < 0 || s >= nscans) return fail(m, NDT2D_EINVAL, "pair %d: scan index out of range", p);
        max_tgt = std::max(max_tgt, h_offsets[t + 1] - h_offsets[t]);
        max_src = std::max(max_src, h_offsets[s + 1] - h_offsets[s]);
    }
    const int K = m->prm.overlap ? 4 : 1, L = m->nlevels;
    CK(m, m->b_perr.ensure(4));
    CK(m, cudaMemsetAsync(m->b_perr.p, 0, 4, m->cfg.stream));
    // fused path: K = 1 and scans that fit a warp's shared-memory slice (1080-beam scans: 27 KB per warp, 8 warps per SM)
    {
        PairFusedArgs f;
        memset(&f, 0, sizeof(f));
        f.prm = m->prm;
        const char *env = getenv("NDT2D_PAIRS_FUSED");
        if (K == 1 && !(env && atoi(env) == 0) && pairs_fused_layout(f, max_tgt, max_src, m->cfg.max_smem_optin)) {
            int rcu;
            if ((rcu = upload(m, m->b_ppairs, pairs, (size_t)npairs * 8))) return rcu;
            CK(m, cudaStreamSynchronize(m->cfg.stream));     // `pairs` is the caller's buffer
            f.xy = reinterpret_cast<const float2 *>(d_xy);
            f.offsets = d_offsets;
            f.pairs = m->b_ppairs.as<int32_t>();
            f.init = d_init;
            f.res = d_res;
            f.npairs = npairs; f.nlevels = L; f.explicit_grid = m->explicit_grid ? 1 : 0;
            for (int l = 0; l < L; ++l) f.res_m[l] = m->res[l];
            f.gox = m->gox; f.goy = m->goy; f.gex = m->gex; f.gey = m->gey;
            f.counter = m->b_counter.as<unsigned int>();
            f.error = m->b_perr.as<int>();
            CK(m, launch_pairs_fused(m->cfg, f, &m->launches));
            return NDT2D_OK;
        }
    }
    // general path (overlapping grids, long scans): slots per table: 1.5 x the most cells a target can occupy (every point in cells of its own), rounded up to a power
    // of two: at most 2/3 full in that worst case, typically a quarter (a 1080-beam scan occupies ~500 cells)
    const uint64_t want = 3ull * (uint64_t)std::max<int64_t>(max_tgt, 16) * K / 2;
    if (want > 65536) return fail(m, NDT2D_EINVAL, "align_pairs: target scans of %lld points need more than 65536 table slots",
                                  (long long)max_tgt);
    const unsigned cap = next_pow2((unsigned)want);
    const size_t per_target = (size_t)L * (((size_t)cap + 1) * 32 + (size_t)cap * 44 + sizeof(LevelDev));
    size_t budget = (size_t)8 << 30;
    if (const char *e = getenv("NDT2D_PAIRS_BYTES")) budget = (size_t)strtoull(e, nullptr, 10);
    const int tmax = (int)std::max<size_t>(1, std::min<size_t>(budget / per_target, (size_t)nscans));
    int rc;
    std::vector<int32_t> slot((size_t)nscans, -1), targets, resolved;
    int p0 = 0;
    while (p0 < npairs) {
        // the next chunk: pairs in order until the chunk's distinct targets would exceed the budget
        targets.clear();
        resolved.clear();
        int p1 = p0;
        for (; p1 < npairs; ++p1) {
            const int t = pairs[2 * p1];
            if (slot[t] < 0) {
                if ((int)targets.size() == tmax) break;
                slot[t] = (int32_t)targets.size();
                targets.push_back(t);
            }
            resolved.push_back(slot[t]);
            resolved.push_back(pairs[2 * p1 + 1]);
        }
        const size_t T = targets.size(), TL = T * (size_t)L;
        CK(m, m->b_ptab.ensure(TL * ((size_t)cap + 1) * 32));
        // the accumulators are zero between builds (every finalisation zeroes what it consumed): clear them when they are (re)allocated
        if (m->b_pcnt.cap < TL * cap * 4 || m->b_psums.cap < TL * cap * 40) {
            CK(m, cudaStreamSynchronize(m->cfg.stream));
            CK(m, m->b_pcnt.ensure(TL * cap * 4));
            CK(m, m->b_psums.ensure(TL * cap * 40));
            CK(m, cudaMemsetAsync(m->b_pcnt.p, 0, m->b_pcnt.cap, m->cfg.stream));
            CK(m, cudaMemsetAsync(m->b_psums.p, 0, m->b_psums.cap, m->cfg.stream));
        }
        CK(m, m->b_pgeo.ensure(TL * sizeof(LevelDev)));
        if ((rc = upload(m, m->b_ptargets, targets.data(), T * 4))) return rc;
        if ((rc = upload(m, m->b_ppairs, resolved.data(), resolved.size() * 4))) return rc;
        CK(m, cudaStreamSynchronize(m->cfg.stream)); // the vectors are reused by the next chunk
        PairBuildArgs b;
        memset(&b, 0, sizeof(b));
        b.xy = reinterpret_cast<const float2 *>(d_xy);
        b.offsets = d_offsets;
        b.targets = m->b_ptargets.as<int32_t>();
        b.ntargets = (int)T; b.nlevels = L; b.ov = m->prm.overlap; b.explicit_grid = m->explicit_grid ? 1 : 0;
        for (int l = 0; l < L; ++l) b.res[l] = m->res[l];
        b.gox = m->gox; b.goy = m->goy; b.gex = m->gex; b.gey = m->gey;
        b.min_points = m->prm.min_points; b.eig_ratio = m->prm.eig_ratio;
        b.cap = cap;
        b.tab = m->b_ptab.as<float4>(); b.cnt = m->b_pcnt.as<uint32_t>(); b.sums = m->b_psums.as<unsigned long long>();
        b.geo = m->b_pgeo.as<LevelDev>();
        b.error = m->b_perr.as<int>();
        CK(m, launch_pairs_build(m->cfg, b, &m->launches));
        AlignArgs a{};
        a.xy = reinterpret_cast<const float2 *>(d_xy);
        a.offsets = d_offsets;
        a.pairs = m->b_ppairs.as<int32_t>();
        a.geo = m->b_pgeo.as<LevelDev>();
        a.init = d_init + 3 * (size_t)p0;
        a.res = d_res + p0;
        a.nscans = p1 - p0;
        if ((rc = align_device(m, a, (int)max_src))) return rc;
        for (int32_t t : targets) slot[t] = -1;
        p0 = p1;
    }
    return NDT2D_OK;
}

static int align_pairs_check(ndt2d_matcher *m)
{
    int err = 0;
    CK(m, cudaMemcpyAsync(&err, m->b_perr.p, 4, cudaMemcpyDeviceToHost, m->cfg.stream));
    int rc = ndt2d_synchronize(m);
    if (rc) return rc;
    if (err) return fail(m, NDT2D_EINVAL, "align_pairs: the auto-fitted lattice of a target scan exceeds 2^31 cells "
                                          "(a point far from the rest?); its pairs were returned with status NO_OVERLAP");
    return NDT2D_OK;
}

static int align_pairs_validate(ndt2d_matcher *m, const int64_t *offsets, int nscans, const int32_t *pairs, int npairs)
{
    if (nscans < 0 || npairs < 0 || (nscans > 0 && !offsets) || (npairs > 0 && !pairs)) return fail(m, NDT2D_EINVAL, "bad arguments");
    if (m->nlevels < 1) return fail(m, NDT2D_EINVAL, "no resolution set");
    for (int b = 0; b < nscans; ++b) {
        int64_t nb = offsets[b + 1] - offsets[b];
        if (nb < 0 || nb > 0x7fffffff) return fail(m, NDT2D_EINVAL, "offsets not monotone at scan %d", b);
    }
    if (nscans > 0 && offsets[0] < 0) return fail(m, NDT2D_EINVAL, "bad offsets");
    return NDT2D_OK;
}

int ndt2d_align_pairs_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, const int64_t *offsets, int nscans,
                             const int32_t *pairs, int npairs, const double *d_init, ndt2d_result *d_res)
{
    if (!m) return NDT2D_EINVAL;
    int rc = align_pairs_validate(m, offsets, nscans, pairs, npairs);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!d_offsets || !d_init || !d_res) return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    return align_pairs_impl(m, d_xy, d_offsets, offsets, nscans, pairs, npairs, d_init, d_res);
}

int ndt2d_align_pairs(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const int32_t *pairs, int npairs,
                      const double *init, ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    int rc = align_pairs_validate(m, offsets, nscans, pairs, npairs);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!init || !res) return fail(m, NDT2D_EINVAL, "bad arguments");
    const int64_t total = offsets[nscans];
    if (total > 0 && !xy) return fail(m, NDT2D_EINVAL, "bad offsets / xy");
    DeviceGuard g(m->device);
    if ((rc = upload(m, m->b_xy, xy, (size_t)total * 8))) return rc;
    if ((rc = upload(m, m->b_off, offsets, (size_t)(nscans + 1) * 8))) return rc;
    if ((rc = upload(m, m->b_init, init, (size_t)npairs * 24))) return rc;
    CK(m, m->b_res.ensure((size_t)npairs * sizeof(ndt2d_result)));
    rc = align_pairs_impl(m, m->b_xy.as<float>(), m->b_off.as<int64_t>(), offsets, nscans, pairs, npairs, m->b_init.as<double>(),
                          m->b_res.as<ndt2d_result>());
    if (rc) return rc;
    CK(m, cudaMemcpyAsync(res, m->b_res.p, (size_t)npairs * sizeof(ndt2d_result), cudaMemcpyDeviceToHost, m->cfg.stream));
    return align_pairs_check(m);
}

} // extern "C"
