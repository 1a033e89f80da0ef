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
    LevelDev L;
    // an unusable lattice (empty or >= 2^31 cells) is reported and left empty: every align against this target ends NO_OVERLAP
    const bool too_big = !level_geometry(L, a.res[l], a.ov, a.explicit_grid != 0, a.gox, a.goy, a.gex, a.gey, xmin, ymin, xmax, ymax);
    if (too_big) { L.nhx = L.nhy = 0; L.njx = L.njy = L.ov; }
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

// SPEC 2 auto-fit: bounding box of the target's finite points, by one warp (every lane gets the result; min and max are
// order independent). k_pairs_fused keeps its own copy of this loop inline: called from there, the helper changes its code.
__device__ __forceinline__ void target_bbox(const float2 *__restrict__ tsrc, int tn, int lane, float &xmin, float &ymin, float &xmax,
                                            float &ymax)
{
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
            const bool usable = level_geometry(L, a.res_m[l], 0, a.explicit_grid != 0, a.gox, a.goy, a.gex, a.gey, xmin, ymin, xmax, ymax);
            if (!usable) L.nhx = L.nhy = L.njx = L.njy = 0;  // as k_pairs_build: the target is reported, the pair ends NO_OVERLAP
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

// ------------------------------------------------------------------------------------------------
// submaps (SPEC 7.3): the target of a pair is several posed scans
// ------------------------------------------------------------------------------------------------

static constexpr int SUBMAP_THREADS = 256;
static constexpr int SUBMAP_LIST_CAP = 16384;   // claimed-slot list per block (u16 entries, 32 KB); longer: full-table scan

// Point q (flat index, in [start[e0], start[e1])) of the submap whose members are [e0, e1), in f64 map coordinates (SPEC 7.2);
// false for a non-finite scan point. The member is found by binary search over start[e0 .. e1-1]; the last member whose
// start is <= q holds the point, so empty members are skipped.
__device__ __forceinline__ bool submap_point(const float2 *__restrict__ xy, const SubmapDev &s, int e0, int e1, int64_t q, double &X,
                                             double &Y)
{
    int lo = e0, hi = e1 - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(s.start + mid) <= q) lo = mid;
        else hi = mid - 1;
    }
    const float2 p = __ldg(xy + __ldg(s.base + lo) + (q - __ldg(s.start + lo)));
    X = Y = 0.0;
    if (!isfinite(p.x) || !isfinite(p.y)) return false;
    posed_point(s.pose + 4 * (size_t)lo, p.x, p.y, X, Y);
    return true;
}

// k_pairs_build for a submap of up to 43 690 points: one block per (submap slot, level), its eight warps striding over the
// submap's points. SPEC 2 auto-fit box of the ((float)Xd, (float)Yd) roundings (a block reduction, as k_bbox for
// set_target_scans), the level's lattice by level_geometry, SPEC 3 accumulation into the slot's hash table (claim by
// compare-and-swap, as k_pairs_build) and, after a block barrier, the finalisation of the slots the block claimed.
// (The minimum of one block per SM lifts ptxas's register target: without it the OV = 1 form spilled at 64 registers.)
template <int OV>
__global__ void __launch_bounds__(SUBMAP_THREADS, 1) k_submap_build(const __grid_constant__ PairBuildArgs a, const __grid_constant__ SubmapDev s)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wid = blockIdx.x;
    const int t = wid / a.nlevels, l = wid % a.nlevels;
    __shared__ unsigned short s_list[SUBMAP_LIST_CAP];
    __shared__ int s_nlist;
    __shared__ float s_box[4][SUBMAP_THREADS / 32];
    const int g = __ldg(a.targets + t);
    const int e0 = (int)__ldg(s.offsets + g), e1 = (int)__ldg(s.offsets + g + 1);
    const int64_t q0 = __ldg(s.start + e0);
    const int n = (int)(__ldg(s.start + e1) - q0);

    float xmin = INFINITY, ymin = INFINITY, xmax = -INFINITY, ymax = -INFINITY;
    if (!a.explicit_grid) {
        for (int i = threadIdx.x; i < n; i += SUBMAP_THREADS) {
            double X, Y;
            if (!submap_point(a.xy, s, e0, e1, q0 + i, X, Y)) continue;
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
        if (lane == 0) { s_box[0][warp] = xmin; s_box[1][warp] = ymin; s_box[2][warp] = xmax; s_box[3][warp] = ymax; }
        __syncthreads();
#pragma unroll
        for (int w = 0; w < SUBMAP_THREADS / 32; ++w) {
            xmin = fminf(xmin, s_box[0][w]); ymin = fminf(ymin, s_box[1][w]);
            xmax = fmaxf(xmax, s_box[2][w]); ymax = fmaxf(ymax, s_box[3][w]);
        }
    }
    LevelDev L;
    // an unusable lattice is reported and left empty, as by k_pairs_build: every pair against this submap ends NO_OVERLAP
    const bool too_big = !level_geometry(L, a.res[l], a.ov, a.explicit_grid != 0, a.gox, a.goy, a.gex, a.gey, xmin, ymin, xmax, ymax);
    if (too_big) { L.nhx = L.nhy = 0; L.njx = L.njy = L.ov; }
    L.hash_mask = a.cap - 1u;
    float4 *rec = a.tab + (size_t)wid * ((size_t)a.cap + 1) * 2;
    uint32_t *cnt = a.cnt + (size_t)wid * a.cap;
    unsigned long long *sums = a.sums + (size_t)wid * a.cap * 5;
    L.cells = rec;
    L.cnt = cnt;
    L.sums = sums;
    if (threadIdx.x == 0) {
        a.geo[wid] = L;
        s_nlist = 0;
        if (too_big) atomicMax(a.error, t + 1);
    }
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 empty = make_float4(0.f, 0.f, __int_as_float((int)kEmptyKey), 0.f);
    for (unsigned sl = threadIdx.x; sl <= a.cap; sl += SUBMAP_THREADS) {
        rec[2 * (size_t)sl] = zero;
        rec[2 * (size_t)sl + 1] = sl < a.cap ? empty : zero;
    }
    __syncthreads();

    unsigned *keyword = reinterpret_cast<unsigned *>(rec);   // key of slot s = word 8 s + 6
    for (int base = warp * 32; base < n; base += SUBMAP_THREADS) {
        const int i = base + lane;
        double X = 0.0, Y = 0.0;
        const bool valid = i < n && submap_point(a.xy, s, e0, e1, q0 + i, X, Y);
        accumulate_window<OV>(L, valid, X, Y, lane, [&](int key, unsigned c, long long sx, long long sy, long long sxx, long long sxy, long long syy) {
            unsigned sl = hash_slot((unsigned)key, L.hash_mask);
            bool placed = false;
            for (unsigned probes = 0; probes <= L.hash_mask; ++probes) {
                unsigned was = atomicCAS(keyword + 8 * (size_t)sl + 6, kEmptyKey, (unsigned)key);
                if (was == kEmptyKey) {
                    const int pos = atomicAdd(&s_nlist, 1);
                    if (pos < SUBMAP_LIST_CAP) s_list[pos] = (unsigned short)sl;
                    placed = true;
                    break;
                }
                if (was == (unsigned)key) { placed = true; break; }
                sl = (sl + 1u) & L.hash_mask;
            }
            if (!placed) { atomicMax(a.error, t + 1); return; }
            atomicAdd(cnt + sl, c);
            unsigned long long *q = sums + 5 * (size_t)sl;
            atomicAdd(q + 0, (unsigned long long)sx);
            atomicAdd(q + 1, (unsigned long long)sy);
            atomicAdd(q + 2, (unsigned long long)sxx);
            atomicAdd(q + 3, (unsigned long long)sxy);
            atomicAdd(q + 4, (unsigned long long)syy);
        });
    }
    __threadfence();
    __syncthreads();

    // SPEC 3 finalisation of the claimed slots, as k_pairs_build's
    auto finish = [&](unsigned sl) {
        const unsigned key = *(volatile unsigned *)(keyword + 8 * (size_t)sl + 6);
        if (key == kEmptyKey) return;
        const unsigned nn = *(volatile uint32_t *)(cnt + sl);
        volatile long long *q = reinterpret_cast<volatile long long *>(sums + 5 * (size_t)sl);
        const long long q0_ = q[0], q1 = q[1], q2 = q[2], q3 = q[3], q4 = q[4];
        float4 ra, rb;
        finalize_record(nn, q0_, q1, q2, q3, q4, L.qu, a.min_points, a.eig_ratio, ra, rb);
        rb.z = __int_as_float((int)key);
        rec[2 * (size_t)sl] = ra;
        rec[2 * (size_t)sl + 1] = rb;
        cnt[sl] = 0u;
        q[0] = 0; q[1] = 0; q[2] = 0; q[3] = 0; q[4] = 0;
    };
    const int nlist = s_nlist;
    if (nlist <= SUBMAP_LIST_CAP) {
        for (int e = threadIdx.x; e < nlist; e += SUBMAP_THREADS) finish(s_list[e]);
    } else {
        for (unsigned sl = threadIdx.x; sl < a.cap; sl += SUBMAP_THREADS) finish(sl);
    }
}

cudaError_t launch_submap_build(const LaunchCfg &c, const PairBuildArgs &a, const SubmapDev &s, int64_t *launches)
{
    const int64_t blocks = (int64_t)a.ntargets * a.nlevels;
    if (blocks <= 0) return cudaSuccess;
    if (a.ov) k_submap_build<1><<<(int)blocks, SUBMAP_THREADS, 0, c.stream>>>(a, s);
    else k_submap_build<0><<<(int)blocks, SUBMAP_THREADS, 0, c.stream>>>(a, s);
    ++*launches;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// windowed search over pairs (ndt2d_relocalize_pairs, SPEC 6.1): k_search_sweep scores every window hypothesis of every pair
// and keeps the k best per (pair, hypothesis chunk); k_search_topk merges a pair's chunks into its exact top-k and turns it
// into refinement jobs, which k_pairs_fused (shared-memory tables) or k_align in pairs mode (per-target hash tables) align.
// The same two kernels search a batch of scans against the handle's dense target (ndt2d_relocalize_batch, SPEC 6.2), whose
// jobs k_align_block or k_align refine in job_scan mode.
// ------------------------------------------------------------------------------------------------

static constexpr int SEARCH_WARPS = 8;
static constexpr unsigned SEARCH_HEAD_BYTES = 128 + SEARCH_WARPS * 32 * 16;   // LevelDev, then the warps' top-k lists
static_assert(sizeof(LevelDev) <= 128, "k_search_sweep's head");

struct SearchCand {
    double score;
    long long idx;      // -1: no candidate
};

// A work item p is a pair (ndt2d_relocalize_pairs) or, with TABLE_DENSE, scan p of the batch against the handle's target
// (ndt2d_relocalize_batch); npairs then counts scans and pairs is unused.
struct SearchArgs {
    const float2 *xy;
    const int64_t *offsets;
    const int32_t *pairs;    // (target scan, source scan) per pair; with geo: (target slot, source scan)
    const LevelDev *geo;     // per-target tables (TABLE_GHASH): geo[slot * nlevels + level]; TABLE_DENSE: the handle's levels
    const double *centres;   // 3 per pair
    ndt2d_window win;
    long long nhyp;          // hypotheses per pair (< 2^31)
    int npairs, chunks, k, level, nlevels;
    // TABLE_SHASH: the sweep level's lattice and the layout of the table areas (from pairs_fused_layout)
    int explicit_grid;
    float res_m, gox, goy, gex, gey;
    int min_points;
    double eig_ratio;
    unsigned cap_t, hslots, off_r, off_h, off_s;   // byte offsets behind the head: records, bucket index, staged source
    SearchCand *cand;        // [npairs * chunks * k]
    unsigned int *counter;   // work queue head, zero on entry
    int *error;              // set to 1 + pair when a target's lattice would exceed 2^31 cells
};

// k_argmax_pass's order: (-score, index); an empty candidate (index -1) comes last
__device__ __forceinline__ bool search_better(double s1, long long i1, double s2, long long i2)
{
    if (i2 < 0) return i1 >= 0;
    if (i1 < 0) return false;
    return (s1 > s2) || (s1 == s2 && i1 < i2);
}

// hypothesis j of the window around c (SPEC 6.1): one f64 multiply, one f64 add, one rounding to f32 per coordinate; widened
// back to f64 as the sweep and the refinement read f32 hypotheses
__device__ __forceinline__ void window_pose(const double *__restrict__ c, const ndt2d_window &w, long long j, double p[3])
{
    const long long nt = 2 * (long long)w.nth + 1, ny = 2 * (long long)w.ny + 1;
    const long long it = j % nt - w.nth, iy = (j / nt) % ny - w.ny, ix = j / (nt * ny) - w.nx;
    p[0] = (double)__double2float_rn(__dadd_rn(__ldg(c), __dmul_rn((double)ix, w.step_x)));
    p[1] = (double)__double2float_rn(__dadd_rn(__ldg(c + 1), __dmul_rn((double)iy, w.step_y)));
    p[2] = (double)__double2float_rn(__dadd_rn(__ldg(c + 2), __dmul_rn((double)it, w.step_th)));
}

// running top-k of a warp: lane r < k holds the r-th best candidate so far (sorted, empty entries last)
__device__ __forceinline__ void topk_insert(double &ms, long long &mi, double s, long long i, int k, int lane)
{
    if (s != s || i < 0) return;        // NaN scores are skipped, as by k_argmax_pass
    const int pos = __popc(__ballot_sync(FULL_MASK, lane < k && search_better(ms, mi, s, i)));
    const double us = __shfl_up_sync(FULL_MASK, ms, 1);
    const long long ui = __shfl_up_sync(FULL_MASK, mi, 1);
    if (pos >= k) return;
    if (lane > pos) { ms = us; mi = ui; }
    else if (lane == pos) { ms = s; mi = i; }
}

// One work item = (pair, chunk of its hypotheses) from the queue. TABLE_SHASH: warp 0 builds the target's grid of the sweep
// level in shared memory (build_table_shared, as k_pairs_fused) while the other warps stage the source as f64; TABLE_GHASH:
// the prebuilt per-target table. Each warp then scores its hypotheses with the dense sweep's evaluation (the same bits as
// ndt2d_sweep on ndt2d_set_target(target scan)), keeps a running top-k, and warp 0 merges the warps' lists into the item's k
// candidates. TABLE_DENSE: item p is scan p of the batch swept over the handle's dense table geo[level] (ndt2d_relocalize_batch;
// every warp stages, the same eval_warp instantiation as k_eval_poses, so the scores are ndt2d_sweep's on that target).
// STAGED = false: sources too long for shared memory are read from global memory, as by k_eval_poses.
template <int OV, int TABLE, bool STAGED>
__global__ void __launch_bounds__(SEARCH_WARPS * 32, 3) k_search_sweep(const __grid_constant__ SearchArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned s_item;
    LevelDev *Ls = reinterpret_cast<LevelDev *>(smem_raw);
    SearchCand *lists = reinterpret_cast<SearchCand *>(smem_raw + 128);
    unsigned char *area = smem_raw + SEARCH_HEAD_BYTES;
    double2 *sp = reinterpret_cast<double2 *>(area + a.off_s);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned nitems = (unsigned)a.npairs * (unsigned)a.chunks;
    for (;;) {
        __syncthreads();                // the previous item is done with the shared memory
        if (threadIdx.x == 0) s_item = atomicAdd(a.counter, 1u);
        __syncthreads();
        const unsigned item = s_item;
        if (item >= nitems) break;
        const int p = (int)(item / (unsigned)a.chunks), c = (int)(item % (unsigned)a.chunks);
        const int tsel = TABLE == TABLE_DENSE ? 0 : __ldg(a.pairs + 2 * (size_t)p);
        const int sscan = TABLE == TABLE_DENSE ? p : __ldg(a.pairs + 2 * (size_t)p + 1);
        const int64_t s0 = __ldg(a.offsets + sscan), s1 = __ldg(a.offsets + sscan + 1);
        const int sn = (int)(s1 - s0);
        const float2 *__restrict__ ssrc = a.xy + s0;
        int stager = (int)threadIdx.x, nstagers = (int)blockDim.x;
        if (TABLE == TABLE_SHASH) {
            stager -= 32; nstagers -= 32;
            if (warp == 0) {
                const int64_t t0 = __ldg(a.offsets + tsel), t1 = __ldg(a.offsets + tsel + 1);
                const int tn = (int)(t1 - t0);
                const float2 *__restrict__ tsrc = a.xy + t0;
                float xmin = INFINITY, ymin = INFINITY, xmax = -INFINITY, ymax = -INFINITY;
                if (!a.explicit_grid) target_bbox(tsrc, tn, lane, xmin, ymin, xmax, ymax);
                LevelDev L;
                const bool usable = level_geometry(L, a.res_m, 0, a.explicit_grid != 0, a.gox, a.goy, a.gex, a.gey, xmin, ymin, xmax, ymax);
                if (!usable) L.nhx = L.nhy = L.njx = L.njy = 0;   // as k_pairs_build
                float *rec = reinterpret_cast<float *>(area + a.off_r);
                unsigned *hidx = reinterpret_cast<unsigned *>(area + a.off_h);
                L.cells = reinterpret_cast<const float4 *>(rec);
                L.cnt = hidx;
                L.sums = nullptr;
                L.hash_mask = a.hslots / 4u - 1u;
                L.zero_rec = 0u;
                if (!usable && lane == 0) atomicMax(a.error, p + 1);
                if (lane == 0) *Ls = L;
                __syncwarp();
                const int nrec = build_table_shared(Ls, tsrc, tn, a.min_points, a.eig_ratio, reinterpret_cast<unsigned *>(area), a.cap_t,
                                                    rec, hidx, a.hslots);
                if (lane == 0) Ls->zero_rec = (unsigned)nrec;
            }
        } else if (threadIdx.x == 0) {
            *Ls = a.geo[(size_t)tsel * a.nlevels + a.level];
        }
        if (STAGED && stager >= 0) {    // sanitised points as f64, padded with the far-away point (SPEC 4), as the dense sweep
            const int npad = (sn + 63) & ~63;
            for (int i = stager; i < npad; i += nstagers) {
                const float2 q = i < sn ? sanitize(__ldg(ssrc + i)) : make_float2(1e18f, 1e18f);
                sp[i] = make_double2((double)q.x, (double)q.y);
            }
        }
        __syncthreads();
        const long long h0 = (long long)c * a.nhyp / a.chunks, h1 = (long long)(c + 1) * a.nhyp / a.chunks;
        const double *cp = a.centres + 3 * (size_t)p;
        double ms = 0.0;
        long long mi = -1;
#pragma unroll 1
        for (long long j = h0 + warp; j < h1; j += SEARCH_WARPS) {
            double h[3];
            window_pose(cp, a.win, j, h);
            const Pose32 q = pose_for_level<true>(h[0], h[1], h[2], *Ls);
            Eval E;
            if (STAGED) eval_warp<OV, false, true, false, TABLE, true>(*Ls, reinterpret_cast<const float2 *>(sp), sn, q, lane, E);
            else eval_warp<OV, false, false, false, TABLE>(*Ls, ssrc, sn, q, lane, E);
            topk_insert(ms, mi, __shfl_sync(FULL_MASK, E.v[0], 0), j, a.k, lane);
        }
        if (lane < a.k) lists[warp * 32 + lane] = SearchCand{ms, mi};
        __syncthreads();
        if (warp == 0) {
#pragma unroll 1
            for (int w = 1; w < SEARCH_WARPS; ++w)
#pragma unroll 1
                for (int r = 0; r < a.k; ++r) {
                    const SearchCand e = lists[w * 32 + r];
                    if (e.idx < 0) break;
                    topk_insert(ms, mi, e.score, e.idx, a.k, lane);
                }
            if (lane < a.k) a.cand[(size_t)item * a.k + lane] = SearchCand{ms, mi};
        }
    }
}

// One block per pair: its exact top-k by (-score, index) in k passes of a block-wide arg-max over its chunks' candidates (every
// member of the pair's top-k is among its own chunk's k best), written to best_idx / best_score as by ndt2d_sweep, and the
// refinement job of each: the pair's (target, source) and the hypothesis widened to f64, as k_topk_to_jobs does. SCAN_JOBS
// (batch against the handle's target): the job is AlignArgs::job_scan[j] = p, or -1 for an empty slot (no LM work).
template <bool SCAN_JOBS>
__global__ void __launch_bounds__(256) k_search_topk(const __grid_constant__ SearchArgs a, int64_t *__restrict__ best_idx,
                                                     double *__restrict__ best_score, int32_t *__restrict__ jobs, double *__restrict__ init)
{
    __shared__ double s_val[8];
    __shared__ long long s_idx[8];
    const int p = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const SearchCand *__restrict__ cand = a.cand + (size_t)p * a.chunks * a.k;
    const int n = a.chunks * a.k;
    double pv = 0.0;
    long long pi = -1;                  // the previous pass's pick
    for (int r = 0; r < a.k; ++r) {
        double bv = 0.0;
        long long bi = -1;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const SearchCand e = cand[i];
            if ((r == 0 || search_better(pv, pi, e.score, e.idx)) && search_better(e.score, e.idx, bv, bi)) { bv = e.score; bi = e.idx; }
        }
        auto warp_best = [&]() {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double v2 = __shfl_xor_sync(FULL_MASK, bv, o);
                const long long i2 = __shfl_xor_sync(FULL_MASK, bi, o);
                if (search_better(v2, i2, bv, bi)) { bv = v2; bi = i2; }
            }
        };
        warp_best();
        if (lane == 0) { s_val[warp] = bv; s_idx[warp] = bi; }
        __syncthreads();
        bv = lane < (int)(blockDim.x >> 5) ? s_val[lane] : 0.0;
        bi = lane < (int)(blockDim.x >> 5) ? s_idx[lane] : -1;
        warp_best();                    // every warp reduces the same eight entries: every thread has the pick
        __syncthreads();
        const size_t j = (size_t)p * a.k + r;
        if (threadIdx.x == 0) {
            best_idx[j] = bi;
            if (best_score) best_score[j] = bi >= 0 ? bv : 0.0;
            if (SCAN_JOBS) {
                jobs[j] = bi >= 0 ? p : -1;
            } else {
                jobs[2 * j] = __ldg(a.pairs + 2 * (size_t)p);
                jobs[2 * j + 1] = __ldg(a.pairs + 2 * (size_t)p + 1);
            }
            double h[3] = {0.0, 0.0, 0.0};
            if (bi >= 0) window_pose(a.centres + 3 * (size_t)p, a.win, bi, h);
            init[3 * j] = h[0]; init[3 * j + 1] = h[1]; init[3 * j + 2] = h[2];
        }
        pv = bv;
        pi = bi;
    }
}

// the slots without a candidate: the all-zero NO_OVERLAP record ndt2d_relocalize returns for them
__global__ void k_search_clear(const int64_t *__restrict__ best_idx, int n, ndt2d_result *__restrict__ res)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n || best_idx[j] >= 0) return;
    ndt2d_result z;
    memset(&z, 0, sizeof(z));
    z.status = NDT2D_NO_OVERLAP;
    res[j] = z;
}

// Shared-memory layout of k_search_sweep behind its head: TABLE_SHASH: the build's sort area, records and bucket index as in
// k_pairs_fused (f.cap_t, f.rmax, f.hslots from pairs_fused_layout), then the source; TABLE_GHASH: the source only. Returns
// the dynamic shared memory per block; staged = false when the source does not fit (global reads, TABLE_GHASH only).
// TABLE_SHASH also takes the lattice of level s.level, the cell parameters and the error flag from f.
size_t search_layout(SearchArgs &s, const PairFusedArgs *f, int64_t max_source_points, int smem_optin, bool &staged)
{
    auto up16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    size_t off = 0;
    if (f) {
        s.explicit_grid = f->explicit_grid;
        s.res_m = f->res_m[s.level];
        s.gox = f->gox; s.goy = f->goy; s.gex = f->gex; s.gey = f->gey;
        s.min_points = f->prm.min_points; s.eig_ratio = f->prm.eig_ratio;
        s.error = f->error;
        s.cap_t = f->cap_t;
        s.hslots = f->hslots;
        s.off_r = (unsigned)up16((size_t)f->cap_t * 4 + 2 * ((size_t)f->cap_t + 2) * 2);
        s.off_h = (unsigned)(s.off_r + up16(std::max<size_t>(((size_t)f->rmax + 1) * 24, 1024)));
        off = s.off_h + (size_t)f->hslots * 4;
    }
    s.off_s = (unsigned)up16(off);
    const size_t with_src = SEARCH_HEAD_BYTES + s.off_s + (size_t)((std::max<int64_t>(max_source_points, 1) + 63) & ~(int64_t)63) * 16;
    staged = with_src <= (size_t)smem_optin - 1024;
    return staged ? with_src : SEARCH_HEAD_BYTES + s.off_s;
}

template <int OV, int TABLE, bool STAGED>
static cudaError_t launch_search_sweep_t(const LaunchCfg &c, const SearchArgs &a, size_t smem)
{
    auto kern = k_search_sweep<OV, TABLE, STAGED>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SEARCH_WARPS * 32, smem);
    if (e != cudaSuccess) return e;
    const int64_t need = (int64_t)a.npairs * a.chunks, cap = (int64_t)c.sm_count * std::max(per_sm, 1);
    kern<<<(int)std::min(need, cap), SEARCH_WARPS * 32, smem, c.stream>>>(a);
    return cudaGetLastError();
}

// Hypothesis chunks per pair: enough work items to keep every SM busy when there are few pairs (two items per resident block),
// but at least SEARCH_WARPS hypotheses per item, since every item builds (or loads) its target's table and stages its source.
int search_chunks(const LaunchCfg &c, int npairs, long long nhyp)
{
    const long long items = 2ll * c.sm_count * 3;   // k_search_sweep keeps three blocks per SM
    const long long want = (items + npairs - 1) / npairs, most = (nhyp + SEARCH_WARPS - 1) / SEARCH_WARPS;
    return (int)std::max(1ll, std::min(want, most));
}

// sweep (counter zeroed here), top-k and refinement jobs: two launches. table: TABLE_SHASH or TABLE_GHASH (pairs, jobs as
// pairs) or TABLE_DENSE (a batch against the handle's target, jobs as job_scan)
cudaError_t launch_search(const LaunchCfg &c, const SearchArgs &a, bool ov, int table, bool staged, size_t smem, int64_t *best_idx,
                          double *best_score, int32_t *jobs, double *init, int64_t *launches)
{
    if (a.npairs <= 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(a.counter, 0, sizeof(unsigned int), c.stream);
    if (e != cudaSuccess) return e;
    if (table == TABLE_SHASH) e = launch_search_sweep_t<0, TABLE_SHASH, true>(c, a, smem);
    else if (table == TABLE_DENSE && ov)
        e = staged ? launch_search_sweep_t<1, TABLE_DENSE, true>(c, a, smem) : launch_search_sweep_t<1, TABLE_DENSE, false>(c, a, smem);
    else if (table == TABLE_DENSE)
        e = staged ? launch_search_sweep_t<0, TABLE_DENSE, true>(c, a, smem) : launch_search_sweep_t<0, TABLE_DENSE, false>(c, a, smem);
    else if (ov) e = staged ? launch_search_sweep_t<1, TABLE_GHASH, true>(c, a, smem) : launch_search_sweep_t<1, TABLE_GHASH, false>(c, a, smem);
    else e = staged ? launch_search_sweep_t<0, TABLE_GHASH, true>(c, a, smem) : launch_search_sweep_t<0, TABLE_GHASH, false>(c, a, smem);
    if (e != cudaSuccess) return e;
    if (table == TABLE_DENSE) k_search_topk<true><<<a.npairs, 256, 0, c.stream>>>(a, best_idx, best_score, jobs, init);
    else k_search_topk<false><<<a.npairs, 256, 0, c.stream>>>(a, best_idx, best_score, jobs, init);
    *launches += 2;
    return cudaGetLastError();
}

cudaError_t launch_search_clear(const LaunchCfg &c, const int64_t *best_idx, int n, ndt2d_result *res, int64_t *launches)
{
    if (n <= 0) return cudaSuccess;
    k_search_clear<<<(n + 255) / 256, 256, 0, c.stream>>>(best_idx, n, res);
    ++*launches;
    return cudaGetLastError();
}

} // namespace ndt2d

using namespace ndt2d;

// ---- batched scan-to-scan (north_star stage 3, "batched multi-scan"): many (target scan, source scan) pairs per call ----

static unsigned next_pow2(unsigned v)
{
    unsigned p = 1;
    while (p < v) p <<= 1;
    return p;
}

// General path (overlapping grids, long scans, submaps): per-target hash tables in global memory, built for chunks of
// consecutive pairs whose distinct targets fit the table budget (NDT2D_PAIRS_BYTES, default 8 GB). A pair's target id
// is a scan of the packed batch (sub == nullptr; tables by k_pairs_build) or a submap of *sub (k_submap_build); ntargets
// is the number of ids and max_tgt the most points of any target a pair names. For chunk [p0, p1), run(p0, p1) finds the
// chunk's pairs as (target slot, source scan) in b_ppairs and the tables' geometry in b_pgeo.
template <class Run>
static int pairs_general(ndt2d_matcher *m, const char *name, const float *d_xy, const int64_t *d_offsets, int ntargets, const int32_t *pairs,
                         int npairs, int64_t max_tgt, const SubmapDev *sub, Run run)
{
    const int K = m->prm.overlap ? 4 : 1, L = m->nlevels;
    // slots per table: 1.5 x the most cells a target can occupy (every point in cells of its own), rounded up to a power
    // of two: at most 2/3 full in that worst case, typically a quarter (a 1080-beam scan occupies ~500 cells)
    const uint64_t want = 3ull * (uint64_t)std::max<int64_t>(max_tgt, 16) * K / 2;
    if (want > 65536) return fail(m, NDT2D_EINVAL, "%s: %s of %lld points need more than 65536 table slots", name,
                                  sub ? "submaps" : "target scans", (long long)max_tgt);
    const unsigned cap = next_pow2((unsigned)want);
    const size_t per_target = (size_t)L * (((size_t)cap + 1) * 32 + (size_t)cap * 44 + sizeof(LevelDev));
    size_t budget = (size_t)8 << 30;
    if (const char *e = getenv("NDT2D_PAIRS_BYTES")) budget = (size_t)strtoull(e, nullptr, 10);
    const int tmax = (int)std::max<size_t>(1, std::min<size_t>(budget / per_target, (size_t)ntargets));
    int rc;
    std::vector<int32_t> slot((size_t)ntargets, -1), targets, resolved;
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
        if (sub) CK(m, launch_submap_build(m->cfg, b, *sub, &m->launches));
        else CK(m, launch_pairs_build(m->cfg, b, &m->launches));
        if ((rc = run(p0, p1))) return rc;
        for (int32_t t : targets) slot[t] = -1;
        p0 = p1;
    }
    return NDT2D_OK;
}

extern "C" {

// ---- checks, set-up and host buffers shared by the calls over packed scans ----

// Packed scans: offsets[0] >= 0, scan b = [offsets[b], offsets[b + 1]) of at most INT_MAX points. *max_points (optional):
// the longest scan.
static int scans_validate(ndt2d_matcher *m, const char *name, const int64_t *offsets, int nscans, int64_t *max_points)
{
    if (nscans > 0 && offsets[0] < 0) return fail(m, NDT2D_EINVAL, "%s: bad offsets", name);
    int64_t longest = 0;
    for (int b = 0; b < nscans; ++b) {
        const int64_t nb = offsets[b + 1] - offsets[b];
        if (nb < 0 || nb > 0x7fffffff) return fail(m, NDT2D_EINVAL, "%s: offsets not monotone at scan %d", name, b);
        longest = std::max(longest, nb);
    }
    if (max_points) *max_points = longest;
    return NDT2D_OK;
}

// The packed scans and the (target scan, source scan) pairs of a call over pairs; *max_tgt / *max_src: the longest target
// and source scan of any pair.
static int pairs_validate(ndt2d_matcher *m, const char *name, const int64_t *offsets, int nscans, const int32_t *pairs, int npairs,
                          int64_t *max_tgt, int64_t *max_src)
{
    if (nscans < 0 || npairs < 0 || (nscans > 0 && !offsets) || (npairs > 0 && !pairs)) return fail(m, NDT2D_EINVAL, "%s: bad arguments", name);
    if (m->nlevels < 1) return fail(m, NDT2D_EINVAL, "%s: no resolution set", name);
    int rc = scans_validate(m, name, offsets, nscans, nullptr);
    if (rc) return rc;
    *max_tgt = *max_src = 0;
    for (int p = 0; p < npairs; ++p) {
        const int t = pairs[2 * p], s = pairs[2 * p + 1];
        if (t < 0 || t >= nscans || s < 0 || s >= nscans) return fail(m, NDT2D_EINVAL, "%s: pair %d: scan index out of range", name, p);
        *max_tgt = std::max(*max_tgt, offsets[t + 1] - offsets[t]);
        *max_src = std::max(*max_src, offsets[s + 1] - offsets[s]);
    }
    return NDT2D_OK;
}

// Host-buffer form: uploads the packed scans, their offsets and one pose per item (initial pose or window centre).
static int upload_scans(ndt2d_matcher *m, const char *name, const float *xy, const int64_t *offsets, int nscans, const double *poses,
                        int nitems)
{
    const int64_t total = offsets[nscans];
    if (total > 0 && !xy) return fail(m, NDT2D_EINVAL, "%s: bad offsets / xy", name);
    int rc;
    if ((rc = upload(m, m->b_xy, xy, (size_t)total * 8))) return rc;
    if ((rc = upload(m, m->b_off, offsets, (size_t)(nscans + 1) * 8))) return rc;
    return upload(m, m->b_init, poses, (size_t)nitems * 24);
}

// End of a host-buffer call: copies best_idx and best_score (when given) and the n records back, synchronises once and
// reports the device error flag d_error (nullptr: the call has none) for a target of kind `what` ("target scan", "submap").
static int finish_host_call(ndt2d_matcher *m, const char *name, size_t n, int64_t *best_idx, double *best_score, ndt2d_result *res,
                            const int *d_error, const char *what = "target scan")
{
    if (best_idx) CK(m, cudaMemcpyAsync(best_idx, m->b_tki.p, n * 8, cudaMemcpyDeviceToHost, m->cfg.stream));
    if (best_score) CK(m, cudaMemcpyAsync(best_score, m->b_tkv.p, n * 8, cudaMemcpyDeviceToHost, m->cfg.stream));
    CK(m, cudaMemcpyAsync(res, m->b_res.p, n * sizeof(ndt2d_result), cudaMemcpyDeviceToHost, m->cfg.stream));
    int err = 0;
    if (d_error) CK(m, cudaMemcpyAsync(&err, d_error, 4, cudaMemcpyDeviceToHost, m->cfg.stream));
    int rc = ndt2d_synchronize(m);
    if (rc) return rc;
    if (err) return fail(m, NDT2D_EINVAL, "%s: the auto-fitted lattice of a %s exceeds 2^31 cells "
                                          "(a point far from the rest?); its pairs were returned with status NO_OVERLAP", name, what);
    return NDT2D_OK;
}

// Whether the shared-memory path (k_pairs_fused; k_search_sweep with TABLE_SHASH) runs: grids without overlap (K = 1), the
// path not switched off by NDT2D_PAIRS_FUSED=0, and scans that fit a warp's shared-memory slice (1080-beam scans: 27 KB per
// warp, 8 warps per SM). When it does, f holds the handle's parameters, levels and lattice, the slice layout, the work-queue
// counter and the error flag; the caller sets the scans, pairs, initial poses and results.
static bool pairs_fused_setup(ndt2d_matcher *m, int64_t max_tgt, int64_t max_src, PairFusedArgs &f)
{
    memset(&f, 0, sizeof(f));
    f.prm = m->prm;
    const char *env = getenv("NDT2D_PAIRS_FUSED");
    if (m->prm.overlap || (env && atoi(env) == 0) || !pairs_fused_layout(f, max_tgt, max_src, m->cfg.max_smem_optin)) return false;
    f.nlevels = m->nlevels;
    f.explicit_grid = m->explicit_grid ? 1 : 0;
    for (int l = 0; l < m->nlevels; ++l) f.res_m[l] = m->res[l];
    f.gox = m->gox; f.goy = m->goy; f.gex = m->gex; f.gey = m->gey;
    f.counter = m->b_counter.as<unsigned int>();
    f.error = m->b_perr.as<int>();
    return true;
}

// d_xy / d_offsets / d_init / d_res: device; pairs: host (the chunking and the target list are host work). One chunk = as
// many pairs as fit the table budget. Asynchronous on the handle's stream apart from the uploads of `pairs` (shared-memory
// path) or of the small per-chunk index lists (general path); a target whose lattice exceeds 2^31 cells sets b_perr.
// sub: the pairs' targets are submaps (always the general path), and ntargets counts them; otherwise it counts the scans.
static int align_pairs_impl(ndt2d_matcher *m, const char *name, const float *d_xy, const int64_t *d_offsets, int ntargets,
                            const int32_t *pairs, int npairs, int64_t max_tgt, int64_t max_src, const double *d_init, ndt2d_result *d_res,
                            const SubmapDev *sub = nullptr)
{
    CK(m, m->b_perr.ensure(4));
    CK(m, cudaMemsetAsync(m->b_perr.p, 0, 4, m->cfg.stream));
    PairFusedArgs f;
    if (!sub && pairs_fused_setup(m, max_tgt, max_src, f)) {
        int rc;
        if ((rc = upload(m, m->b_ppairs, pairs, (size_t)npairs * 8))) return rc;
        CK(m, cudaStreamSynchronize(m->cfg.stream));     // `pairs` is the caller's buffer
        f.xy = reinterpret_cast<const float2 *>(d_xy);
        f.offsets = d_offsets;
        f.pairs = m->b_ppairs.as<int32_t>();
        f.init = d_init;
        f.res = d_res;
        f.npairs = npairs;
        CK(m, launch_pairs_fused(m->cfg, f, &m->launches));
        return NDT2D_OK;
    }
    return pairs_general(m, name, d_xy, d_offsets, ntargets, pairs, npairs, max_tgt, sub, [&](int p0, int p1) {
        AlignArgs a{};
        a.xy = reinterpret_cast<const float2 *>(d_xy);
        a.offsets = d_offsets;
        a.pairs = m->b_ppairs.as<int32_t>();
        a.geo = m->b_pgeo.as<LevelDev>();
        a.init = d_init + 3 * (size_t)p0;
        a.res = d_res + p0;
        a.nscans = p1 - p0;
        return align_device(m, a, (int)max_src);
    });
}

int ndt2d_align_pairs_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, const int64_t *offsets, int nscans,
                             const int32_t *pairs, int npairs, const double *d_init, ndt2d_result *d_res)
{
    if (!m) return NDT2D_EINVAL;
    int64_t max_tgt = 0, max_src = 0;
    int rc = pairs_validate(m, "align_pairs", offsets, nscans, pairs, npairs, &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!d_offsets || !d_init || !d_res) return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    return align_pairs_impl(m, "align_pairs", d_xy, d_offsets, nscans, pairs, npairs, max_tgt, max_src, d_init, d_res);
}

int ndt2d_align_pairs(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const int32_t *pairs, int npairs,
                      const double *init, ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    int64_t max_tgt = 0, max_src = 0;
    int rc = pairs_validate(m, "align_pairs", offsets, nscans, pairs, npairs, &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!init || !res) return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    if ((rc = upload_scans(m, "align_pairs", xy, offsets, nscans, init, npairs))) return rc;
    CK(m, m->b_res.ensure((size_t)npairs * sizeof(ndt2d_result)));
    rc = align_pairs_impl(m, "align_pairs", m->b_xy.as<float>(), m->b_off.as<int64_t>(), nscans, pairs, npairs, max_tgt, max_src,
                          m->b_init.as<double>(), m->b_res.as<ndt2d_result>());
    if (rc) return rc;
    return finish_host_call(m, "align_pairs", (size_t)npairs, nullptr, nullptr, res, m->b_perr.as<int>());
}

// ---- windowed search over pairs (SPEC 6.1): ndt2d_set_target(target) + ndt2d_relocalize(source, window) per pair ----

// k, the output size and the window (SPEC 6.1) of a windowed search over `count` items (`what`: "npairs" or "nscans"); *nhyp = H
static int search_validate(ndt2d_matcher *m, const char *name, const char *what, int count, const ndt2d_window *win, int k,
                           long long *nhyp)
{
    if (k < 1 || k > 32) return fail(m, NDT2D_EINVAL, "%s: k %d not in [1, 32]", name, k);
    if ((long long)count * k >= (1ll << 31)) return fail(m, NDT2D_EINVAL, "%s: %s * k must be below 2^31", name, what);
    if (!win) return fail(m, NDT2D_EINVAL, "%s: no window", name);
    if (win->nx < 0 || win->ny < 0 || win->nth < 0 || win->reserved != 0)
        return fail(m, NDT2D_EINVAL, "%s: window half-widths (%d, %d, %d) must be >= 0 and reserved 0", name, win->nx, win->ny, win->nth);
    if (!isfinite(win->step_x) || !isfinite(win->step_y) || !isfinite(win->step_th))
        return fail(m, NDT2D_EINVAL, "%s: window steps must be finite", name);
    long long h = 2ll * win->nx + 1;
    for (long long f : {2ll * win->ny + 1, 2ll * win->nth + 1}) {
        if (h >= (1ll << 31)) break;
        h *= f;
    }
    if (h >= (1ll << 31)) return fail(m, NDT2D_EINVAL, "%s: the window has 2^31 or more hypotheses", name);
    *nhyp = h;
    return NDT2D_OK;
}

// The SearchArgs fields of every windowed search, and room for njobs refinement jobs of job_bytes each and their initial poses
static int search_setup(ndt2d_matcher *m, SearchArgs &s, const float *d_xy, const int64_t *d_offsets, const ndt2d_window &win,
                        long long nhyp, int k, int level, size_t njobs, size_t job_bytes)
{
    CK(m, m->b_sjobs.ensure(njobs * job_bytes));
    CK(m, m->b_sinit.ensure(njobs * 24));
    memset(&s, 0, sizeof(s));
    s.xy = reinterpret_cast<const float2 *>(d_xy);
    s.offsets = d_offsets;
    s.win = win;
    s.nhyp = nhyp;
    s.k = k; s.level = level; s.nlevels = m->nlevels;
    s.counter = m->b_counter.as<unsigned int>();
    return NDT2D_OK;
}

// The hypothesis chunks of one sweep launch over `items` work items, and the candidate buffer for them
static cudaError_t search_candidates(ndt2d_matcher *m, SearchArgs &s, int items)
{
    s.chunks = search_chunks(m->cfg, items, s.nhyp);
    const cudaError_t e = m->b_scand.ensure((size_t)items * s.chunks * s.k * sizeof(SearchCand));
    s.cand = m->b_scand.as<SearchCand>();
    return e;
}

static int relocalize_pairs_validate(ndt2d_matcher *m, int level, const int64_t *offsets, int nscans, const int32_t *pairs, int npairs,
                                     const ndt2d_window *win, int k, long long *nhyp, int64_t *max_tgt, int64_t *max_src)
{
    int rc = pairs_validate(m, "relocalize_pairs", offsets, nscans, pairs, npairs, max_tgt, max_src);
    if (rc) return rc;
    if (level < 0 || level >= m->nlevels) return fail(m, NDT2D_EINVAL, "level %d out of range [0, %d)", level, m->nlevels);
    return search_validate(m, "relocalize_pairs", "npairs", npairs, win, k, nhyp);
}

// Shared-memory path (as ndt2d_align_pairs, when k_search_sweep can also stage the longest source): sweep, top-k, refinement
// by k_pairs_fused and the empty slots: four launches whatever the number of pairs. General path: per chunk of the per-target
// tables, the table build, the same sweep and top-k on the tables, k_align in pairs mode and the empty slots. sub and
// ntargets: as for align_pairs_impl.
static int relocalize_pairs_impl(ndt2d_matcher *m, const char *name, int level, const float *d_xy, const int64_t *d_offsets, int ntargets,
                                 const int32_t *pairs, int npairs, int64_t max_tgt, int64_t max_src, const double *d_centres,
                                 const ndt2d_window &win, long long nhyp, int k, int64_t *d_best_idx, double *d_best_score,
                                 ndt2d_result *d_res, const SubmapDev *sub = nullptr)
{
    const size_t njobs = (size_t)npairs * k;
    CK(m, m->b_perr.ensure(4));
    CK(m, cudaMemsetAsync(m->b_perr.p, 0, 4, m->cfg.stream));
    SearchArgs s;
    int rc = search_setup(m, s, d_xy, d_offsets, win, nhyp, k, level, njobs, 8);
    if (rc) return rc;
    int32_t *d_jobs = m->b_sjobs.as<int32_t>();
    double *d_jinit = m->b_sinit.as<double>();
    PairFusedArgs f;
    bool staged = false;
    size_t smem = 0;
    if (!sub && pairs_fused_setup(m, max_tgt, max_src, f) && (smem = search_layout(s, &f, max_src, m->cfg.max_smem_optin, staged), staged)) {
        // `pairs` is the caller's buffer: it is uploaded from a copy, so that nothing waits for the copy to finish
        m->h_spairs.assign(pairs, pairs + 2 * (size_t)npairs);
        if ((rc = upload(m, m->b_ppairs, m->h_spairs.data(), (size_t)npairs * 8))) return rc;
        s.pairs = m->b_ppairs.as<int32_t>();
        s.centres = d_centres;
        s.npairs = npairs;
        CK(m, search_candidates(m, s, npairs));
        CK(m, launch_search(m->cfg, s, false, TABLE_SHASH, true, smem, d_best_idx, d_best_score, d_jobs, d_jinit, &m->launches));
        f.xy = s.xy;
        f.offsets = d_offsets;
        f.pairs = d_jobs;
        f.init = d_jinit;
        f.res = d_res;
        f.npairs = (int)njobs;
        CK(m, launch_pairs_fused(m->cfg, f, &m->launches));
        CK(m, launch_search_clear(m->cfg, d_best_idx, (int)njobs, d_res, &m->launches));
        return NDT2D_OK;
    }
    smem = search_layout(s, nullptr, max_src, m->cfg.max_smem_optin, staged);
    return pairs_general(m, name, d_xy, d_offsets, ntargets, pairs, npairs, max_tgt, sub, [&](int p0, int p1) -> int {
        const size_t j0 = (size_t)p0 * k, nj = (size_t)(p1 - p0) * k;
        s.pairs = m->b_ppairs.as<int32_t>();
        s.geo = m->b_pgeo.as<LevelDev>();
        s.centres = d_centres + 3 * (size_t)p0;
        s.npairs = p1 - p0;
        CK(m, search_candidates(m, s, p1 - p0));
        CK(m, launch_search(m->cfg, s, m->prm.overlap != 0, TABLE_GHASH, staged, smem, d_best_idx + j0, d_best_score ? d_best_score + j0 : nullptr,
                            d_jobs, d_jinit, &m->launches));
        AlignArgs a{};
        a.xy = s.xy;
        a.offsets = d_offsets;
        a.pairs = d_jobs;
        a.geo = s.geo;
        a.init = d_jinit;
        a.res = d_res + j0;
        a.nscans = (int)nj;
        int rc = align_device(m, a, (int)max_src);
        if (rc) return rc;
        CK(m, launch_search_clear(m->cfg, d_best_idx + j0, (int)nj, d_res + j0, &m->launches));
        return NDT2D_OK;
    });
}

int ndt2d_relocalize_pairs_device(ndt2d_matcher *m, int level, const float *d_xy, const int64_t *d_offsets, const int64_t *offsets,
                                  int nscans, const int32_t *pairs, int npairs, const double *d_centres, const ndt2d_window *win, int k,
                                  int64_t *d_best_idx, double *d_best_score, ndt2d_result *d_res)
{
    if (!m) return NDT2D_EINVAL;
    long long nhyp = 0;
    int64_t max_tgt = 0, max_src = 0;
    int rc = relocalize_pairs_validate(m, level, offsets, nscans, pairs, npairs, win, k, &nhyp, &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!d_offsets || !d_centres || !d_best_idx || !d_res) return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    return relocalize_pairs_impl(m, "relocalize_pairs", level, d_xy, d_offsets, nscans, pairs, npairs, max_tgt, max_src, d_centres, *win,
                                 nhyp, k, d_best_idx, d_best_score, d_res);
}

int ndt2d_relocalize_pairs(ndt2d_matcher *m, int level, const float *xy, const int64_t *offsets, int nscans, const int32_t *pairs,
                           int npairs, const double *centres, const ndt2d_window *win, int k, int64_t *best_idx, double *best_score,
                           ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    long long nhyp = 0;
    int64_t max_tgt = 0, max_src = 0;
    int rc = relocalize_pairs_validate(m, level, offsets, nscans, pairs, npairs, win, k, &nhyp, &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!centres || !best_idx || !res) return fail(m, NDT2D_EINVAL, "bad arguments");
    DeviceGuard g(m->device);
    const size_t njobs = (size_t)npairs * k;
    if ((rc = upload_scans(m, "relocalize_pairs", xy, offsets, nscans, centres, npairs))) return rc;
    CK(m, m->b_tki.ensure(njobs * 8));
    CK(m, m->b_tkv.ensure(njobs * 8));
    CK(m, m->b_res.ensure(njobs * sizeof(ndt2d_result)));
    rc = relocalize_pairs_impl(m, "relocalize_pairs", level, m->b_xy.as<float>(), m->b_off.as<int64_t>(), nscans, pairs, npairs, max_tgt,
                               max_src, m->b_init.as<double>(), *win, nhyp, k, m->b_tki.as<int64_t>(), m->b_tkv.as<double>(),
                               m->b_res.as<ndt2d_result>());
    if (rc) return rc;
    return finish_host_call(m, "relocalize_pairs", njobs, best_idx, best_score, res, m->b_perr.as<int>());
}

// ---- pairs against submaps of posed scans (SPEC 7.3): ndt2d_set_target_scans(members) + align / relocalize per pair ----

// The scans, the submaps and the (submap, source scan) pairs of a call over submaps. host_poses: the member poses are host
// memory and are checked finite (the device forms pass nullptr and false). *max_tgt: the most points of any submap a pair
// names; *max_src: the longest source. Leaves each member's first flat point index and first point in xy in
// m->h_sm_start / m->h_sm_base, for submaps_setup.
static int submaps_validate(ndt2d_matcher *m, const char *name, const int64_t *offsets, int nscans, const int64_t *submap_offsets,
                            int nsubmaps, const int32_t *member_scans, const double *poses, bool host_poses, const int32_t *pairs,
                            int npairs, int64_t *max_tgt, int64_t *max_src)
{
    if (nscans < 0 || nsubmaps < 0 || npairs < 0 || (nscans > 0 && !offsets) || !submap_offsets || (npairs > 0 && !pairs))
        return fail(m, NDT2D_EINVAL, "%s: bad arguments", name);
    if (m->nlevels < 1) return fail(m, NDT2D_EINVAL, "%s: no resolution set", name);
    int rc = scans_validate(m, name, offsets, nscans, nullptr);
    if (rc) return rc;
    if (submap_offsets[0] != 0) return fail(m, NDT2D_EINVAL, "%s: submap_offsets[0] = %lld, not 0", name, (long long)submap_offsets[0]);
    for (int g = 0; g < nsubmaps; ++g)
        if (submap_offsets[g + 1] < submap_offsets[g] || submap_offsets[g + 1] > 0x7fffffff)
            return fail(m, NDT2D_EINVAL, "%s: submap offsets not monotone at submap %d", name, g);
    const int64_t nmembers = submap_offsets[nsubmaps];
    if (nmembers > 0 && (!member_scans || (host_poses && !poses))) return fail(m, NDT2D_EINVAL, "%s: bad arguments", name);
    m->h_sm_start.resize((size_t)nmembers + 1);
    m->h_sm_base.resize((size_t)nmembers);
    int64_t flat = 0;
    for (int64_t e = 0; e < nmembers; ++e) {
        const int32_t b = member_scans[e];
        if (b < 0 || b >= nscans) return fail(m, NDT2D_EINVAL, "%s: member %lld: scan index %d out of range", name, (long long)e, b);
        if (host_poses && (!std::isfinite(poses[3 * e]) || !std::isfinite(poses[3 * e + 1]) || !std::isfinite(poses[3 * e + 2])))
            return fail(m, NDT2D_EINVAL, "%s: pose of member %lld is not finite", name, (long long)e);
        m->h_sm_start[(size_t)e] = flat;
        m->h_sm_base[(size_t)e] = offsets[b];
        flat += offsets[b + 1] - offsets[b];
    }
    m->h_sm_start[(size_t)nmembers] = flat;
    *max_tgt = *max_src = 0;
    for (int p = 0; p < npairs; ++p) {
        const int g = pairs[2 * p], s = pairs[2 * p + 1];
        if (g < 0 || g >= nsubmaps) return fail(m, NDT2D_EINVAL, "%s: pair %d: submap index out of range", name, p);
        if (s < 0 || s >= nscans) return fail(m, NDT2D_EINVAL, "%s: pair %d: scan index out of range", name, p);
        *max_tgt = std::max(*max_tgt, m->h_sm_start[(size_t)submap_offsets[g + 1]] - m->h_sm_start[(size_t)submap_offsets[g]]);
        *max_src = std::max(*max_src, offsets[s + 1] - offsets[s]);
    }
    return NDT2D_OK;
}

// Uploads the submap offsets and the tables submaps_validate left on the host, and makes the members' pose table from the
// f64 poses on the device (one launch): *sub is then what k_submap_build reads.
static int submaps_setup(ndt2d_matcher *m, const int64_t *submap_offsets, int nsubmaps, const double *d_poses, SubmapDev *sub)
{
    const size_t nmembers = m->h_sm_base.size();
    int rc;
    if ((rc = upload(m, m->b_sm_off, submap_offsets, ((size_t)nsubmaps + 1) * 8))) return rc;
    if ((rc = upload(m, m->b_sm_start, m->h_sm_start.data(), (nmembers + 1) * 8))) return rc;
    if ((rc = upload(m, m->b_sm_base, m->h_sm_base.data(), nmembers * 8))) return rc;
    CK(m, m->b_sm_tab.ensure(std::max<size_t>(nmembers, 1) * 32));
    CK(m, launch_pose_table(m->cfg, d_poses, (int)nmembers, m->b_sm_tab.as<double>(), &m->launches));
    sub->offsets = m->b_sm_off.as<int64_t>();
    sub->start = m->b_sm_start.as<int64_t>();
    sub->base = m->b_sm_base.as<int64_t>();
    sub->pose = m->b_sm_tab.as<double>();
    return NDT2D_OK;
}

int ndt2d_align_submaps_device(ndt2d_matcher *m, const float *d_xy, const int64_t *d_offsets, const int64_t *offsets, int nscans,
                               const int64_t *submap_offsets, int nsubmaps, const int32_t *member_scans, const double *d_member_poses,
                               const int32_t *pairs, int npairs, const double *d_init, ndt2d_result *d_res)
{
    if (!m) return NDT2D_EINVAL;
    int64_t max_tgt = 0, max_src = 0;
    int rc = submaps_validate(m, "align_submaps", offsets, nscans, submap_offsets, nsubmaps, member_scans, nullptr, false, pairs, npairs,
                              &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!d_offsets || !d_init || !d_res || (!m->h_sm_base.empty() && !d_member_poses))
        return fail(m, NDT2D_EINVAL, "align_submaps: bad arguments");
    DeviceGuard g(m->device);
    SubmapDev sub;
    if ((rc = submaps_setup(m, submap_offsets, nsubmaps, d_member_poses, &sub))) return rc;
    return align_pairs_impl(m, "align_submaps", d_xy, d_offsets, nsubmaps, pairs, npairs, max_tgt, max_src, d_init, d_res, &sub);
}

int ndt2d_align_submaps(ndt2d_matcher *m, const float *xy, const int64_t *offsets, int nscans, const int64_t *submap_offsets, int nsubmaps,
                        const int32_t *member_scans, const double *member_poses, const int32_t *pairs, int npairs, const double *init,
                        ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    int64_t max_tgt = 0, max_src = 0;
    int rc = submaps_validate(m, "align_submaps", offsets, nscans, submap_offsets, nsubmaps, member_scans, member_poses, true, pairs,
                              npairs, &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!init || !res) return fail(m, NDT2D_EINVAL, "align_submaps: bad arguments");
    DeviceGuard g(m->device);
    if ((rc = upload_scans(m, "align_submaps", xy, offsets, nscans, init, npairs))) return rc;
    if ((rc = upload(m, m->b_sm_pose, member_poses, m->h_sm_base.size() * 24))) return rc;
    CK(m, m->b_res.ensure((size_t)npairs * sizeof(ndt2d_result)));
    SubmapDev sub;
    if ((rc = submaps_setup(m, submap_offsets, nsubmaps, m->b_sm_pose.as<double>(), &sub))) return rc;
    rc = align_pairs_impl(m, "align_submaps", m->b_xy.as<float>(), m->b_off.as<int64_t>(), nsubmaps, pairs, npairs, max_tgt, max_src,
                          m->b_init.as<double>(), m->b_res.as<ndt2d_result>(), &sub);
    if (rc) return rc;
    return finish_host_call(m, "align_submaps", (size_t)npairs, nullptr, nullptr, res, m->b_perr.as<int>(), "submap");
}

static int relocalize_submaps_validate(ndt2d_matcher *m, int level, const int64_t *offsets, int nscans, const int64_t *submap_offsets,
                                       int nsubmaps, const int32_t *member_scans, const double *poses, bool host_poses, const int32_t *pairs,
                                       int npairs, const ndt2d_window *win, int k, long long *nhyp, int64_t *max_tgt, int64_t *max_src)
{
    int rc = submaps_validate(m, "relocalize_submaps", offsets, nscans, submap_offsets, nsubmaps, member_scans, poses, host_poses, pairs,
                              npairs, max_tgt, max_src);
    if (rc) return rc;
    if (level < 0 || level >= m->nlevels)
        return fail(m, NDT2D_EINVAL, "relocalize_submaps: level %d out of range [0, %d)", level, m->nlevels);
    return search_validate(m, "relocalize_submaps", "npairs", npairs, win, k, nhyp);
}

int ndt2d_relocalize_submaps_device(ndt2d_matcher *m, int level, const float *d_xy, const int64_t *d_offsets, const int64_t *offsets,
                                    int nscans, const int64_t *submap_offsets, int nsubmaps, const int32_t *member_scans,
                                    const double *d_member_poses, const int32_t *pairs, int npairs, const double *d_centres,
                                    const ndt2d_window *win, int k, int64_t *d_best_idx, double *d_best_score, ndt2d_result *d_res)
{
    if (!m) return NDT2D_EINVAL;
    long long nhyp = 0;
    int64_t max_tgt = 0, max_src = 0;
    int rc = relocalize_submaps_validate(m, level, offsets, nscans, submap_offsets, nsubmaps, member_scans, nullptr, false, pairs, npairs,
                                         win, k, &nhyp, &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!d_offsets || !d_centres || !d_best_idx || !d_res || (!m->h_sm_base.empty() && !d_member_poses))
        return fail(m, NDT2D_EINVAL, "relocalize_submaps: bad arguments");
    DeviceGuard g(m->device);
    SubmapDev sub;
    if ((rc = submaps_setup(m, submap_offsets, nsubmaps, d_member_poses, &sub))) return rc;
    return relocalize_pairs_impl(m, "relocalize_submaps", level, d_xy, d_offsets, nsubmaps, pairs, npairs, max_tgt, max_src, d_centres,
                                 *win, nhyp, k, d_best_idx, d_best_score, d_res, &sub);
}

int ndt2d_relocalize_submaps(ndt2d_matcher *m, int level, const float *xy, const int64_t *offsets, int nscans, const int64_t *submap_offsets,
                             int nsubmaps, const int32_t *member_scans, const double *member_poses, const int32_t *pairs, int npairs,
                             const double *centres, const ndt2d_window *win, int k, int64_t *best_idx, double *best_score,
                             ndt2d_result *res)
{
    if (!m) return NDT2D_EINVAL;
    long long nhyp = 0;
    int64_t max_tgt = 0, max_src = 0;
    int rc = relocalize_submaps_validate(m, level, offsets, nscans, submap_offsets, nsubmaps, member_scans, member_poses, true, pairs,
                                         npairs, win, k, &nhyp, &max_tgt, &max_src);
    if (rc) return rc;
    if (npairs == 0) return NDT2D_OK;
    if (!centres || !best_idx || !res) return fail(m, NDT2D_EINVAL, "relocalize_submaps: bad arguments");
    DeviceGuard g(m->device);
    const size_t njobs = (size_t)npairs * k;
    if ((rc = upload_scans(m, "relocalize_submaps", xy, offsets, nscans, centres, npairs))) return rc;
    if ((rc = upload(m, m->b_sm_pose, member_poses, m->h_sm_base.size() * 24))) return rc;
    CK(m, m->b_tki.ensure(njobs * 8));
    CK(m, m->b_tkv.ensure(njobs * 8));
    CK(m, m->b_res.ensure(njobs * sizeof(ndt2d_result)));
    SubmapDev sub;
    if ((rc = submaps_setup(m, submap_offsets, nsubmaps, m->b_sm_pose.as<double>(), &sub))) return rc;
    rc = relocalize_pairs_impl(m, "relocalize_submaps", level, m->b_xy.as<float>(), m->b_off.as<int64_t>(), nsubmaps, pairs, npairs,
                               max_tgt, max_src, m->b_init.as<double>(), *win, nhyp, k, m->b_tki.as<int64_t>(), m->b_tkv.as<double>(),
                               m->b_res.as<ndt2d_result>(), &sub);
    if (rc) return rc;
    return finish_host_call(m, "relocalize_submaps", njobs, best_idx, best_score, res, m->b_perr.as<int>(), "submap");
}

// ---- windowed search of a batch of scans against the handle's target (SPEC 6.2): ndt2d_relocalize(scan, window) per scan ----

// Sweep of every scan over its window on the dense table of `level`, top-k, refinement of the nscans * k jobs by align_device
// (k_align_block or k_align, job_scan mode) and the empty slots: four launches whatever the number of scans.
static int relocalize_batch_impl(ndt2d_matcher *m, int level, const float *d_xy, const int64_t *d_offsets, int nscans, int max_points,
                                 const double *d_centres, const ndt2d_window &win, long long nhyp, int k, int64_t *d_best_idx,
                                 double *d_best_score, ndt2d_result *d_res)
{
    const size_t njobs = (size_t)nscans * k;
    SearchArgs s;
    int rc = search_setup(m, s, d_xy, d_offsets, win, nhyp, k, level, njobs, 4);
    if (rc) return rc;
    // the sweep reads the level from the device (SearchArgs::geo); the copy is taken now, so a later set_target cannot reach it
    if ((rc = upload(m, m->b_slevels, m->lv, (size_t)m->nlevels * sizeof(LevelDev)))) return rc;
    s.geo = m->b_slevels.as<LevelDev>();
    s.centres = d_centres;
    s.npairs = nscans;
    // every item stages only its scan (no table build), so the chunking is the pairs' one without a table to amortise
    CK(m, search_candidates(m, s, nscans));
    bool staged = false;
    const size_t smem = search_layout(s, nullptr, max_points, m->cfg.max_smem_optin, staged);
    int32_t *d_jobs = m->b_sjobs.as<int32_t>();
    double *d_jinit = m->b_sinit.as<double>();
    CK(m, launch_search(m->cfg, s, m->prm.overlap != 0, TABLE_DENSE, staged, smem, d_best_idx, d_best_score, d_jobs, d_jinit, &m->launches));
    AlignArgs a{};
    a.xy = s.xy;
    a.offsets = d_offsets;
    a.job_scan = d_jobs;
    a.init = d_jinit;
    a.res = d_res;
    a.nscans = (int)njobs;
    if ((rc = align_device(m, a, max_points))) return rc;
    CK(m, launch_search_clear(m->cfg, d_best_idx, (int)njobs, d_res, &m->launches));
    return NDT2D_OK;
}

int ndt2d_relocalize_batch_device(ndt2d_matcher *m, int level, const float *d_xy, const int64_t *d_offsets, int nscans, int max_points,
                                  const double *d_centres, const ndt2d_window *win, int k, int64_t *d_best_idx, double *d_best_score,
                                  ndt2d_result *d_res)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    long long nhyp = 0;
    if ((rc = search_validate(m, "relocalize_batch", "nscans", nscans, win, k, &nhyp))) return rc;
    if (nscans < 0 || max_points < 0 || (nscans > 0 && (!d_offsets || !d_centres || !d_best_idx || !d_res)))
        return fail(m, NDT2D_EINVAL, "relocalize_batch: bad arguments");
    if (nscans == 0) return NDT2D_OK;
    DeviceGuard g(m->device);
    return relocalize_batch_impl(m, level, d_xy, d_offsets, nscans, max_points, d_centres, *win, nhyp, k, d_best_idx, d_best_score, d_res);
}

int ndt2d_relocalize_batch(ndt2d_matcher *m, int level, const float *xy, const int64_t *offsets, int nscans, const double *centres,
                           const ndt2d_window *win, int k, int64_t *best_idx, double *best_score, ndt2d_result *res)
{
    int rc = check_level(m, level);
    if (rc) return rc;
    long long nhyp = 0;
    if ((rc = search_validate(m, "relocalize_batch", "nscans", nscans, win, k, &nhyp))) return rc;
    if (nscans < 0 || (nscans > 0 && (!offsets || !centres || !best_idx || !res))) return fail(m, NDT2D_EINVAL, "relocalize_batch: bad arguments");
    if (nscans == 0) return NDT2D_OK;
    int64_t max_points = 0;
    if ((rc = scans_validate(m, "relocalize_batch", offsets, nscans, &max_points))) return rc;
    DeviceGuard g(m->device);
    const size_t njobs = (size_t)nscans * k;
    if ((rc = upload_scans(m, "relocalize_batch", xy, offsets, nscans, centres, nscans))) return rc;
    CK(m, m->b_tki.ensure(njobs * 8));
    CK(m, m->b_tkv.ensure(njobs * 8));
    CK(m, m->b_res.ensure(njobs * sizeof(ndt2d_result)));
    rc = relocalize_batch_impl(m, level, m->b_xy.as<float>(), m->b_off.as<int64_t>(), nscans, (int)max_points, m->b_init.as<double>(), *win,
                               nhyp, k, m->b_tki.as<int64_t>(), m->b_tkv.as<double>(), m->b_res.as<ndt2d_result>());
    if (rc) return rc;
    return finish_host_call(m, "relocalize_batch", njobs, best_idx, best_score, res, nullptr);
}

} // extern "C"
