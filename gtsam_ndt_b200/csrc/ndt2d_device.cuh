// Device-side building blocks of the 2D NDT path: lattice index (SPEC 2, f64), per-pair terms (SPEC 4, cell-local f32),
// expneg (SPEC 4.1), the warp evaluation with SPEC 4's fixed summation order, and the damped closed-form 3x3 solve
// (SPEC 5). Compiled with -fmad=false: only the explicit fma calls below fuse, exactly as SPEC.md writes them.
// Reference file:line: none exists (/root/reference/README.md:1 is the whole mount).
//
// The evaluation is written for Blackwell's packed f32x2 instructions (FFMA2 / FMUL2 / FADD2): SPEC.md v2
// arranges every per-point quantity as a pair — (rx,ry), (jx,jy), (X,Y), (qx,qy), (ux,uy), (vx,vy), the record
// pairs (mux,muy) (B00,B01) (B01,B11) — so one packed instruction does both components with the scalar of
// the other operand broadcast, and the scalar chains (exp, dot-product sums) of the two points a lane owns
// are packed across the points. Each packed op is the IEEE round-to-nearest op on both halves: results are
// bit-identical to the scalar oracle.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "ndt2d_internal.h"

namespace ndt2d {

typedef unsigned long long u64;

// ---- packed f32x2 helpers --------------------------------------------------------------------------
__device__ __forceinline__ u64 pk(float lo, float hi)
{
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk(u64 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ float lo32(u64 v) { float a, b; upk(v, a, b); return a; }
__device__ __forceinline__ float hi32(u64 v) { float a, b; upk(v, a, b); return b; }
__device__ __forceinline__ u64 bc(float c) { return pk(c, c); } // broadcast; ptxas folds it into an .F32 operand
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
// acc = fma(a, b, acc) / acc = acc + a, accumulator tied to the destination
__device__ __forceinline__ void fma2_acc(u64 &acc, u64 a, u64 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b)); }
__device__ __forceinline__ void add2_acc(u64 &acc, u64 a) { asm("add.rn.f32x2 %0, %0, %1;" : "+l"(acc) : "l"(a)); }
// lo + hi of a packed product pair: the "a*b + c*d" of SPEC 4 (two rounded products, one add)
__device__ __forceinline__ float hsum(u64 v) { float a, b; upk(v, a, b); return __fadd_rn(a, b); }

// ---- SPEC 2 (v4): lattice index in f64 -------------------------------------------------------------------
// f: a coordinate in cell units relative to the lattice origin. h = floor(f) comes from the "magic number" sum
// t = f + 1.5 * 2^52 rounded towards -infinity: for 0 <= floor(f) < 2^32 the high word of t is the magic constant's and
// the low word is floor(f), so the lattice test is two integer compares and NaN, infinities and huge values fail it.
// df = (float)(f - h): the position inside the lattice square, in [0, 1] (the subtraction is exact).
// Returns hi(t), which equals hi(magic) = 0x43380000 iff 0 <= floor(f) < 2^32.
__device__ __forceinline__ unsigned node_of(double f, unsigned &h, float &df)
{
    const double MAGIC = 6755399441055744.0; // 1.5 * 2^52
    const double t = __dadd_rd(f, MAGIC);
    const double n = __dadd_rn(t, -MAGIC);
    df = __double2float_rn(__dsub_rn(f, n));
    h = (unsigned)__double2loint(t);
    return (unsigned)__double2hiint(t);
}

// Index of table entry (hx, hy) if both coordinates are inside the lattice, else `outside`. Written in PTX so that the
// test stays one LOP3 ((wx ^ C) | (wy ^ C)), three chained ISETP, one IMAD and one SEL: the compiler's own expansion of the
// same expression is four compares feeding four dependent selects per point.
__device__ __forceinline__ unsigned lattice_base(unsigned wx, unsigned wy, unsigned hx, unsigned hy, unsigned nhx, unsigned nhy,
                                                 unsigned njx, unsigned outside)
{
    unsigned r;
    asm("{\n\t.reg .pred p;\n\t.reg .b32 bad, idx;\n\t"
        "lop3.b32 bad, %1, %2, 0x43380000, 0x7e;\n\t"
        "setp.eq.u32 p, bad, 0;\n\t"
        "setp.lt.and.u32 p, %3, %5, p;\n\t"
        "setp.lt.and.u32 p, %4, %6, p;\n\t"
        "mad.lo.u32 idx, %4, %7, %3;\n\t"
        "selp.u32 %0, idx, %8, p;\n\t}"
        : "=r"(r)
        : "r"(wx), "r"(wy), "r"(hx), "r"(hy), "r"(nhx), "r"(nhy), "r"(njx), "r"(outside));
    return r;
}

__device__ __forceinline__ bool lattice_of(double fx, double fy, unsigned nhx, unsigned nhy, unsigned &hx, unsigned &hy, float &dfx,
                                           float &dfy)
{
    const unsigned wx = node_of(fx, hx, dfx), wy = node_of(fy, hy, dfy);
    return (wx == 0x43380000u) & (wy == 0x43380000u) & (hx < nhx) & (hy < nhy);
}

// a target point (no pose): f = (X - (double)origin) * inv_st, X = (double) of an f32 map point or the f64 map coordinate of
// a posed scan point (SPEC 7.2)
__device__ __forceinline__ bool lattice_of_point(const LevelDev &L, double X, double Y, int &hx, int &hy)
{
    unsigned ux, uy;
    float dfx, dfy;
    const bool in = lattice_of(__dmul_rn(__dsub_rn(X, (double)L.ox), L.inv_std), __dmul_rn(__dsub_rn(Y, (double)L.oy), L.inv_std),
                               (unsigned)L.nhx, (unsigned)L.nhy, ux, uy, dfx, dfy);
    hx = (int)ux;
    hy = (int)uy;
    return in;
}

// SPEC 7.2: the f64 map coordinates of the finite scan point (x, y) under its scan's pose P = {cos, sin, p0, p1}
// (launch_pose_table), never rounded to f32. Every build from posed scans (k_accumulate, k_bbox, k_submap_build) goes
// through here.
__device__ __forceinline__ void posed_point(const double *__restrict__ P, float x, float y, double &X, double &Y)
{
    const double cs = __ldg(P), sn = __ldg(P + 1), p0 = __ldg(P + 2), p1 = __ldg(P + 3);
    const double xd = (double)x, yd = (double)y;
    X = __fma_rn(cs, xd, __fma_rn(-sn, yd, p0));
    Y = __fma_rn(sn, xd, __fma_rn(cs, yd, p1));
}

// ---- SPEC 3: finalisation of one cell from its integer sums; f64, operations in the order the spec lists ----
__device__ __forceinline__ void finalize_record(unsigned n, long long s0, long long s1, long long s2, long long s3, long long s4,
                                                double U, int min_points, double eig_ratio, float4 &ra, float4 &rb)
{
    ra = make_float4(0.f, 0.f, 0.f, 0.f);
    rb = ra;
    if (n < (unsigned)min_points) return;
    double N = (double)n;
    double mx = (double)s0 / N, my = (double)s1 / N;
    double cxx = ((double)s2 - (double)s0 * mx) / (N - 1.0);
    double cxy = ((double)s3 - (double)s0 * my) / (N - 1.0);
    double cyy = ((double)s4 - (double)s1 * my) / (N - 1.0);
    mx *= U; my *= U; cxx *= U * U; cxy *= U * U; cyy *= U * U;
    double tr = cxx + cyy, hd = 0.5 * (cxx - cyy), rad = sqrt(hd * hd + cxy * cxy);
    double l1 = 0.5 * tr + rad, l2 = 0.5 * tr - rad;
    if (!(l1 > 1e-10)) return;
    if (l2 < eig_ratio * l1) {
        double l2n = eig_ratio * l1, vx, vy;
        if (hd >= 0.0) { vx = hd + rad; vy = cxy; } else { vx = cxy; vy = rad - hd; }
        double nn = vx * vx + vy * vy, dl = l1 - l2n;
        cxx = l2n + dl * (vx * vx) / nn;
        cxy = dl * (vx * vy) / nn;
        cyy = l2n + dl * (vy * vy) / nn;
    }
    double det = cxx * cyy - cxy * cxy;
    const float b01 = (float)(-(cxy / det));
    ra = make_float4((float)mx, (float)my, (float)(cyy / det), b01); // the mean relative to the cell centre
    rb = make_float4(b01, (float)(cxx / det), (float)n, 1.0f);
}

// ---- SPEC 3: accumulation of one warp-wide window of target points ---------------------------------------------
// One point per lane (valid == false: no point). For each of the K cells of the point, lanes holding the same cell in
// consecutive positions (laser scans are spatially coherent) are combined with a segmented shuffle reduction and the
// head of each run hands the run's count and five integer sums to `sink(key, count, sx, sy, sxx, sxy, syy)`, key being
// the table index jy * njx + jx. Integer sums are associative, so any sink (global atomics into the dense table,
// compare-and-swap into a hash table, ...) gives the cells SPEC 3 defines. Used by k_accumulate and k_pairs_build.
// (X, Y): the map coordinates in f64 - an f32 point widened, or a posed scan point's unrounded transform (SPEC 7.2).
template <int OV, class Sink>
__device__ __forceinline__ void accumulate_window(const LevelDev &L, bool valid, double X, double Y, int lane, Sink sink)
{
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int K = OV ? 2 : 1;
    int hx = 0, hy = 0;
    const bool inside = valid && lattice_of_point(L, X, Y, hx, hy);
#pragma unroll
    for (int b = 0; b < K; ++b) {
#pragma unroll
        for (int a = 0; a < K; ++a) {
            const int jx = hx + a, jy = hy + b;
            const int key = inside ? jy * L.njx + jx : -1;
            const double cx = (double)L.ox + ((double)(jx - L.ov)) * (double)L.st + 0.5 * (double)L.res;
            const double cy = (double)L.oy + ((double)(jy - L.ov)) * (double)L.st + 0.5 * (double)L.res;
            const double dx = X - cx, dy = Y - cy;
            const long long qx = inside ? __double2ll_rn(dx * L.qs) : 0;
            const long long qy = inside ? __double2ll_rn(dy * L.qs) : 0;
            int c = inside ? 1 : 0;
            long long sx = qx, sy = qy, sxx = qx * qx, sxy = qx * qy, syy = qy * qy;
            // run id: number of run heads at or below this lane
            const int prev = __shfl_up_sync(FULL, key, 1);
            const bool head = (lane == 0) || (prev != key);
            const unsigned heads = __ballot_sync(FULL, head);
            const int rid = __popc(heads & (0xffffffffu >> (31 - lane)));
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int rid2 = __shfl_down_sync(FULL, rid, d);
                const int c2 = __shfl_down_sync(FULL, c, d);
                const long long sx2 = __shfl_down_sync(FULL, sx, d);
                const long long sy2 = __shfl_down_sync(FULL, sy, d);
                const long long sxx2 = __shfl_down_sync(FULL, sxx, d);
                const long long sxy2 = __shfl_down_sync(FULL, sxy, d);
                const long long syy2 = __shfl_down_sync(FULL, syy, d);
                if (lane + d < 32 && rid2 == rid) {
                    c += c2; sx += sx2; sy += sy2; sxx += sxx2; sxy += sxy2; syy += syy2;
                }
            }
            if (head && key >= 0) sink(key, (unsigned)c, sx, sy, sxx, sxy, syy);
        }
    }
}

// ---- SPEC 4.1: exp(-h), bit-exact sequence of f32 operations -----------------------------------------
__device__ __forceinline__ float expneg(float h)
{
    float t = __fmaf_rn(h, 1.44269502f, 12582912.0f);
    float nf = __fsub_rn(t, 12582912.0f);
    int ni = __float_as_int(t) - 0x4B400000;
    float r = __fmaf_rn(nf, -0.693145752f, h);
    r = __fmaf_rn(nf, -1.42860677e-6f, r);
    float y = -r;
    float p = 1.38888889e-3f;
    p = __fmaf_rn(p, y, 8.33333333e-3f);
    p = __fmaf_rn(p, y, 4.16666667e-2f);
    p = __fmaf_rn(p, y, 1.66666667e-1f);
    p = __fmaf_rn(p, y, 0.5f);
    p = __fmaf_rn(p, y, 1.0f);
    p = __fmaf_rn(p, y, 1.0f);
    return __fmul_rn(p, __int_as_float(0x3F800000 - ni * 0x800000));
}

// The same on two values; nh = -h. Uses fma(h,L,M) == fma(-h,-L,M) and fma(n,-C,h) == -fma(n,C,-h), both exact
// under round-to-nearest-even, so both halves equal expneg(h) bit for bit.
// NOTE (ptxas 12.9): mul.rn.f32x2 followed by add/sub.rn.f32x2 is contracted into FFMA2 even with -fmad=false
// and explicit .rn, unlike the scalar forms. SPEC.md v2 is written so that every packed multiply that feeds a
// packed add IS an fma; never write mul2 -> add2/sub2 in this file.
__device__ __forceinline__ u64 expneg2(u64 nh)
{
    const u64 MAGIC = bc(12582912.0f);
    // The magic sum taken with the sign of n flipped: t = M - n (fma(-h, L, M); exact mirror of M + n, M's mantissa is even), so
    // that the bits of t are 0x4B400000 - n and 2^-n's bit pattern 0x3F800000 - (n << 23) is 0x3F800000 + (bits(t) << 23)
    // (0x4B400000 << 23 vanishes mod 2^32): one shift-add on the integer pipe per value, where n * -0x800000 + 0x3F800000 was
    // an IMAD - two cycles of the FMA pipe, the loop's busiest unit (tools/mix_probe.py) - plus a constant move per step.
    u64 t = fma2(nh, bc(1.44269502f), MAGIC);
    u64 nf = sub2(t, MAGIC);                       // -n, exactly
    float t0, t1;
    upk(t, t0, t1);
    unsigned s0, s1;
    asm("{\n\t.reg .b32 x;\n\tshl.b32 x, %1, 23;\n\tadd.s32 %0, x, 0x3F800000;\n\t}" : "=r"(s0) : "r"(__float_as_int(t0)));
    asm("{\n\t.reg .b32 x;\n\tshl.b32 x, %1, 23;\n\tadd.s32 %0, x, 0x3F800000;\n\t}" : "=r"(s1) : "r"(__float_as_int(t1)));
    u64 y = fma2(nf, bc(-0.693145752f), nh);       // -h + n ln2: fma(-n, -C, y) == fma(n, C, y)
    y = fma2(nf, bc(-1.42860677e-6f), y);
    u64 p = fma2(bc(1.38888889e-3f), y, bc(8.33333333e-3f));
    p = fma2(p, y, bc(4.16666667e-2f));
    p = fma2(p, y, bc(1.66666667e-1f));
    p = fma2(p, y, bc(0.5f));
    p = fma2(p, y, bc(1.0f));
    p = fma2(p, y, bc(1.0f));
    return mul2(p, pk(__int_as_float((int)s0), __int_as_float((int)s1)));
}

// ---- SPEC 4: pose and point -----------------------------------------------------------------------------
// The pose as one evaluation on one level uses it (SPEC 4, v4): the point-to-cell geometry runs in f64 and in cell
// units relative to the lattice origin (ci, si, txi, tyi); the derivative terms use the f32 roundings (c, s).
struct Pose32 {
    double ci, si, txi, tyi;
    float c, s;
};

// SPEC 4.2: sin and cos of the pose angle as a fixed sequence of f64 operations (two-constant Cody-Waite reduction,
// fdlibm kernel polynomials, quadrant from the low bits of the magic sum): the oracle's bits, and about a third of
// the instructions of the library sincos with its Payne-Hanek branch.
// CM: the polynomial coefficients come from constant memory - a DFMA takes a constant-bank operand directly, whereas a 64-bit
// literal costs two uniform moves in front of it (36 per evaluation). The sweep kernel uses it (233 -> 218 instructions per
// hypothesis outside the point loop); in k_align the literals stay, because with the constant-bank form ptxas's register
// allocation of the point loop came out twelve moves longer (tools/looplen.py: 129 -> 141 instructions).
static __constant__ double kSinCos[15] = {
    0.63661977236758138, 1.5707963267948966, 6.123233995736766e-17,
    1.58969099521155010221e-10, -2.50507602534068634195e-08, 2.75573137070700676789e-06, -1.98412698298579493134e-04,
    8.33333333332248946124e-03, -1.66666666666666324348e-01,
    -1.13596475577881948265e-11, 2.08757232129817482790e-09, -2.75573143513906633035e-07, 2.48015872894767294178e-05,
    -1.38888888888741095749e-03, 4.16666666666666019037e-02};
template <bool CM = false>
__device__ __forceinline__ void sincos_spec(double th, double &sn_out, double &cs_out)
{
    const double MAGIC = 6755399441055744.0; // 1.5 * 2^52
    const double K[15] = {CM ? kSinCos[0] : 0.63661977236758138, CM ? kSinCos[1] : 1.5707963267948966, CM ? kSinCos[2] : 6.123233995736766e-17,
                          CM ? kSinCos[3] : 1.58969099521155010221e-10, CM ? kSinCos[4] : -2.50507602534068634195e-08,
                          CM ? kSinCos[5] : 2.75573137070700676789e-06, CM ? kSinCos[6] : -1.98412698298579493134e-04,
                          CM ? kSinCos[7] : 8.33333333332248946124e-03, CM ? kSinCos[8] : -1.66666666666666324348e-01,
                          CM ? kSinCos[9] : -1.13596475577881948265e-11, CM ? kSinCos[10] : 2.08757232129817482790e-09,
                          CM ? kSinCos[11] : -2.75573143513906633035e-07, CM ? kSinCos[12] : 2.48015872894767294178e-05,
                          CM ? kSinCos[13] : -1.38888888888741095749e-03, CM ? kSinCos[14] : 4.16666666666666019037e-02};
    const double t = __fma_rn(th, K[0], MAGIC);
    const double k = __dadd_rn(t, -MAGIC);
    const int q = __double2loint(t) & 3;
    double r = __fma_rn(-k, K[1], th);
    r = __fma_rn(-k, K[2], r);
    const double z = __dmul_rn(r, r);
    double ps = __fma_rn(z, K[3], K[4]);
    ps = __fma_rn(z, ps, K[5]);
    ps = __fma_rn(z, ps, K[6]);
    ps = __fma_rn(z, ps, K[7]);
    ps = __fma_rn(z, ps, K[8]);
    const double sn = __fma_rn(__dmul_rn(r, z), ps, r);
    double pc = __fma_rn(z, K[9], K[10]);
    pc = __fma_rn(z, pc, K[11]);
    pc = __fma_rn(z, pc, K[12]);
    pc = __fma_rn(z, pc, K[13]);
    pc = __fma_rn(z, pc, K[14]);
    const double cs = __fma_rn(__dmul_rn(z, z), pc, __fma_rn(z, -0.5, 1.0));
    const double s4 = (q & 1) ? cs : sn, c4 = (q & 1) ? sn : cs;
    sn_out = (q & 2) ? -s4 : s4;
    cs_out = ((q + 1) & 2) ? -c4 : c4;
}

template <bool CM = false>
__device__ __forceinline__ Pose32 pose_for_level(double tx, double ty, double th, const LevelDev &L)
{
    double sn, cs;
    sincos_spec<CM>(th, sn, cs);
    Pose32 q;
    q.c = (float)cs;
    q.s = (float)sn;
    q.ci = __dmul_rn(cs, L.inv_std);
    q.si = __dmul_rn(sn, L.inv_std);
    q.txi = __dmul_rn(__dsub_rn(tx, (double)L.ox), L.inv_std);
    q.tyi = __dmul_rn(__dsub_rn(ty, (double)L.oy), L.inv_std);
    return q;
}

// SPEC 4: a point that cannot lie in any lattice becomes the finite far-away point (1e18, 1e18)
__device__ __forceinline__ float2 sanitize(float2 p)
{
    bool bad = !(fabsf(p.x) <= 1e18f) || !(fabsf(p.y) <= 1e18f); // also true for NaN
    return bad ? make_float2(1e18f, 1e18f) : p;
}

struct PosePk {
    u64 cs, nsc, ncns;        // (c,s) (-s,c) (-c,-s): f32, for r = R x and j = dr/dtheta
    double ci, si, txi, tyi;  // f64, cell units: the lattice coordinates of the transformed point
};
__device__ __forceinline__ PosePk pose_pack(const Pose32 &q)
{
    PosePk P;
    P.cs = pk(q.c, q.s);
    P.nsc = pk(-q.s, q.c);
    P.ncns = pk(-q.c, -q.s);
    P.ci = q.ci; P.si = q.si; P.txi = q.txi; P.tyi = q.tyi;
    return P;
}

struct PointPk {
    u64 r, j;      // (rx,ry) (jx,jy), f32
    u64 XY;        // the point relative to the centre of the cell being evaluated (lx, ly), metres, f32
    u64 df;        // position inside the lattice square, in [0,1]^2
};
// JR: take j from r instead of computing it. SPEC 4: jx = fma(ns,x,nc*y) = -ry and jy = fma(c,x,ns*y) = rx bit for bit
// (round-to-nearest is symmetric under negation), so j is r with its halves swapped and one sign flipped; ptxas folds
// that into operand modifiers (.HI_LO.NP) and four packed instructions per step disappear. Measured: +2.3 % at K = 4 (v3), where j
// is used by four cells; at K = 1 it was -2 % under SPEC v3 and is +5 % under v4 (x8: 20.31 vs 19.33 M matches/s - the f64
// geometry made the loop longer and the four instructions count), so every evaluation uses it now. The diagnostic kernel
// k_point_terms computes j as SPEC 4 writes it (JR = false), which the parity tests compare against.
template <bool JR = false>
__device__ __forceinline__ void rotate_point(const PosePk &P, float x, float y, PointPk &p)
{
    p.r = fma2(P.cs, bc(x), mul2(P.nsc, bc(y)));   // rx = fma(c,x,ns*y), ry = fma(s,x,c*y)
    if (JR) p.j = pk(-hi32(p.r), lo32(p.r));
    else p.j = fma2(P.nsc, bc(x), mul2(P.ncns, bc(y))); // jx = fma(ns,x,nc*y), jy = fma(c,x,ns*y)
}

// SPEC 4 (v4): lattice coordinates of the transformed point in f64, f = R x / st + (t - origin) / st; the lattice square
// (hx, hy) and the f32 position inside it. Returns false outside the lattice (hx, hy are then meaningless).
__device__ __forceinline__ bool locate_point(const PosePk &P, float x, float y, unsigned nhx, unsigned nhy, unsigned &hx, unsigned &hy,
                                             u64 &df)
{
    const double xd = (double)x, yd = (double)y;
    const double fx = __fma_rn(P.ci, xd, __fma_rn(-P.si, yd, P.txi));
    const double fy = __fma_rn(P.si, xd, __fma_rn(P.ci, yd, P.tyi));
    float dfx, dfy;
    const bool in = lattice_of(fx, fy, nhx, nhy, hx, hy, dfx, dfy);
    df = pk(dfx, dfy);
    return in;
}

// The same for the gather path: the index of the point's first cell in the table, or G.outside outside the lattice.
struct LatticePk;
__device__ __forceinline__ unsigned locate_base(const PosePk &P, float x, float y, const LatticePk &G, u64 &df);

// ---- cell record: four f32 pairs in one 256-bit load ------------------------------------------------------
struct Cell4 {
    u64 mu, B0, B1, nv; // (mux,muy) (B00,B01) (B01,B11) (n,valid)
};
__device__ __forceinline__ Cell4 load_cell(const float4 *__restrict__ cells, unsigned idx)
{
    Cell4 r;
    const float4 *p = cells + 2 * (size_t)idx;
    // L1::no_allocate (measured best of the gather forms): a gathered record is rarely reused before L1 evicts it, and not
    // allocating spares the fill bandwidth
    asm("ld.global.nc.L1::no_allocate.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(r.mu), "=l"(r.B0), "=l"(r.B1), "=l"(r.nv) : "l"(p));
    return r;
}

// ---- SPEC 4 per-pair terms, scalar form (diagnostic kernel k_point_terms) --------------------------------
__device__ __forceinline__ bool pair_terms_scalar(const Cell4 &c, const PointPk &p, float T[10])
{
    float mux, muy, B00, B01, B01b, B11, nn, valid, rx, ry, jx, jy, X, Y;
    upk(c.mu, mux, muy); upk(c.B0, B00, B01); upk(c.B1, B01b, B11); upk(c.nv, nn, valid);
    upk(p.r, rx, ry); upk(p.j, jx, jy); upk(p.XY, X, Y);
    if (valid == 0.0f) return false;
    float qx = __fsub_rn(X, mux), qy = __fsub_rn(Y, muy);
    float ux = __fmaf_rn(B00, qx, __fmul_rn(B01, qy)), uy = __fmaf_rn(B01, qx, __fmul_rn(B11, qy));
    float mm = __fadd_rn(__fmul_rn(qx, ux), __fmul_rn(qy, uy));
    float h = __fmul_rn(0.5f, mm);
    if (!(h < 30.0f)) return false;
    float e = expneg(h);
    float a2 = __fadd_rn(__fmul_rn(ux, jx), __fmul_rn(uy, jy));
    float vx = __fmaf_rn(B00, jx, __fmul_rn(B01, jy)), vy = __fmaf_rn(B01, jx, __fmul_rn(B11, jy));
    float w = __fadd_rn(__fmul_rn(ux, rx), __fmul_rn(uy, ry));
    float k = __fadd_rn(__fmul_rn(jx, vx), __fmul_rn(jy, vy));
    k = __fsub_rn(k, w);
    k = __fmaf_rn(-a2, a2, k);
    T[0] = e; // the factors (e, c1..c9) that SPEC 4 accumulates with acc_t = fma(e, c_t, acc_t)
    T[1] = ux; T[2] = uy; T[3] = a2;
    T[4] = __fmaf_rn(-ux, ux, B00); T[5] = __fmaf_rn(-ux, uy, B01); T[6] = __fmaf_rn(-a2, ux, vx);
    T[7] = __fmaf_rn(-uy, uy, B11); T[8] = __fmaf_rn(-a2, uy, vy);
    T[9] = k;
    return true;
}

// ---- SPEC 4 evaluation for one warp -------------------------------------------------------------------------
// Result of one evaluation, held redundantly by every lane.
struct Eval {
    double v[10];
    int count;
    int slot; // transposed finish only: v[0] is sum number `slot`
};

__device__ __forceinline__ double warp_sum(double x)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x; // SPEC 4's butterfly: D[l] + D[l xor o] is commutative, every lane ends with the same bits
}

// The same ten butterflies, transposed: in every round a lane keeps half of the sums it still holds and hands the
// other half to its partner, so 12 exchange-and-add steps replace 50. Sum t of lane l goes through exactly the
// additions of SPEC 4's butterfly (D[l] + D[l xor o] with the operands possibly swapped, and IEEE addition
// commutes), so the bits are the butterfly's. Returns the one finished sum this lane ends up with; `t` is its index.
__device__ __forceinline__ double xchg_add(double keep, double send, int o) { return keep + __shfl_xor_sync(0xffffffffu, send, o); }

__device__ __forceinline__ double warp_sum10_transposed(const double V[10], int lane, int &t)
{
    const bool h4 = lane & 16, h3 = lane & 8, h2 = lane & 4, h1 = lane & 2;
    double W[5], X[3], Y[2];
#pragma unroll
    for (int i = 0; i < 5; ++i) W[i] = xchg_add(h4 ? V[i + 5] : V[i], h4 ? V[i] : V[i + 5], 16);
#pragma unroll
    for (int i = 0; i < 2; ++i) X[i] = xchg_add(h3 ? W[i + 3] : W[i], h3 ? W[i] : W[i + 3], 8);
    X[2] = xchg_add(W[2], W[2], 8);
    Y[0] = xchg_add(h2 ? X[2] : X[0], h2 ? X[0] : X[2], 4);
    Y[1] = xchg_add(X[1], X[1], 4);
    double Z = xchg_add(h1 ? Y[1] : Y[0], h1 ? Y[0] : Y[1], 2);
    Z = xchg_add(Z, Z, 1);
    const int xi = h1 ? 1 : (h2 ? 2 : 0);           // which X this lane finished
    const int wi = xi == 2 ? 2 : xi + (h3 ? 3 : 0); // which W
    t = wi + (h4 ? 5 : 0);
    return Z;
}

// f32 partial sums of one lane = SPEC 4's partials p = lane (point A) and lane + 32 (point B)
struct Partials {
    u64 s12[2], s45[2], s68[2]; // per point: (T1,T2) (T4,T5) (T6,T8)
    u64 s0, s3, s9;             // (A,B): T0 T3 T9
    float s7[2];                // T7 per point (scalar: its operands (uy, B11) sit in the high halves of two pairs)
};

// The SPEC 4 factors of one cell for the lane's two points A and B. Skipped pairs have e = 0.
struct Factors {
    u64 e;                 // (eA, eB)
    u64 c12[2], c45[2], c68[2]; // per point: (c1,c2) (c4,c5) (c6,c8)
    u64 c3, c9;            // (A,B)
    float c7[2];           // per point
};

// SPEC 4's two tests of a pair (the cell is valid, h < 30): returns e if the pair counts, else 0; COUNT: cnt += 1 if it counts
template <bool COUNT>
__device__ __forceinline__ float select_count(float valid, float nh, float e, int &cnt)
{
    float r;
    if (COUNT) {
        asm("{\n\t.reg .pred p;\n\t"
            "setp.neu.f32 p, %2, 0f00000000;\n\t"
            "setp.gt.and.f32 p, %3, 0fC1F00000, p;\n\t"
            "selp.f32 %0, %4, 0f00000000, p;\n\t"
            "@p add.s32 %1, %1, 1;\n\t}"
            : "=f"(r), "+r"(cnt)
            : "f"(valid), "f"(nh), "f"(e));
    } else {
        asm("{\n\t.reg .pred p;\n\t"
            "setp.neu.f32 p, %1, 0f00000000;\n\t"
            "setp.gt.and.f32 p, %2, 0fC1F00000, p;\n\t"
            "selp.f32 %0, %3, 0f00000000, p;\n\t}"
            : "=f"(r)
            : "f"(valid), "f"(nh), "f"(e));
    }
    return r;
}

// A point outside the lattice was given the all-zero sentinel record (fetch()), so `valid` covers both tests of SPEC 4.
template <bool FULL>
__device__ __forceinline__ void cell_factors(const Cell4 &cA, const Cell4 &cB, const PointPk &A, const PointPk &B, Factors &F,
                                             int &cnt)
{
    // q = XY - mu ; u = B q ; m = q.u ; nh = -0.5 m
    u64 qA = sub2(A.XY, cA.mu), qB = sub2(B.XY, cB.mu);
    u64 uA = fma2(cA.B0, bc(lo32(qA)), mul2(cA.B1, bc(hi32(qA))));
    u64 uB = fma2(cB.B0, bc(lo32(qB)), mul2(cB.B1, bc(hi32(qB))));
    u64 nh = mul2(bc(-0.5f), pk(hsum(mul2(qA, uA)), hsum(mul2(qB, uB))));
    u64 e = expneg2(nh);
    // skipped pairs get e = 0: fma(0, c, acc) == acc bit for bit (every c is finite, see sanitize())
    // the two tests, the select and the count in PTX: one SEL and one predicated add per point (the compiler's own
    // expansion is a zero move plus a predicated move for the select and an add plus a predicated move for the count)
    F.e = pk(select_count<FULL>(hi32(cA.nv), lo32(nh), lo32(e), cnt), select_count<FULL>(hi32(cB.nv), hi32(nh), hi32(e), cnt));
    if (FULL) {
        float a2A = hsum(mul2(uA, A.j)), a2B = hsum(mul2(uB, B.j));
        u64 vA = fma2(cA.B0, bc(lo32(A.j)), mul2(cA.B1, bc(hi32(A.j))));
        u64 vB = fma2(cB.B0, bc(lo32(B.j)), mul2(cB.B1, bc(hi32(B.j))));
        float wA = hsum(mul2(uA, A.r)), wB = hsum(mul2(uB, B.r));
        u64 k = sub2(pk(hsum(mul2(A.j, vA)), hsum(mul2(B.j, vB))), pk(wA, wB));
        F.c3 = pk(a2A, a2B);
        F.c9 = fma2(pk(-a2A, -a2B), F.c3, k);
        F.c12[0] = uA;
        F.c12[1] = uB;
        F.c45[0] = fma2(bc(-lo32(uA)), uA, cA.B0);
        F.c45[1] = fma2(bc(-lo32(uB)), uB, cB.B0);
        F.c68[0] = fma2(bc(-a2A), uA, vA);
        F.c68[1] = fma2(bc(-a2B), uB, vB);
        F.c7[0] = __fmaf_rn(-hi32(uA), hi32(uA), hi32(cA.B1));
        F.c7[1] = __fmaf_rn(-hi32(uB), hi32(uB), hi32(cB.B1));
    }
}

// acc_t = fma(e, c_t, acc_t) for the factors of one cell (SPEC 4's update of the lane's two partials)
template <bool FULL>
__device__ __forceinline__ void apply_factors(const Factors &F, Partials &S)
{
    add2_acc(S.s0, F.e);
    if (FULL) {
        const float eA = lo32(F.e), eB = hi32(F.e);
        fma2_acc(S.s12[0], F.c12[0], bc(eA));
        fma2_acc(S.s12[1], F.c12[1], bc(eB));
        fma2_acc(S.s45[0], F.c45[0], bc(eA));
        fma2_acc(S.s45[1], F.c45[1], bc(eB));
        fma2_acc(S.s68[0], F.c68[0], bc(eA));
        fma2_acc(S.s68[1], F.c68[1], bc(eB));
        fma2_acc(S.s3, F.e, F.c3);
        S.s7[0] = __fmaf_rn(eA, F.c7[0], S.s7[0]);
        S.s7[1] = __fmaf_rn(eB, F.c7[1], S.s7[1]);
        fma2_acc(S.s9, F.e, F.c9);
    }
}

// Parked factors: the SPEC 4 factors of one (64-point step, cell) for all 32 lanes, written to shared memory by one warp and
// applied by another in SPEC order (k_align_block's eight warps; the helper warps of k_align). FACTOR_WORDS u64 per lane,
// word-major: a warp's store or load of one word is one conflict-free 256-byte row. o = base of the entry + lane.
static constexpr int FACTOR_WORDS = 10; // e, c12[2], c45[2], c68[2], c3, c9, c7 pair
static constexpr unsigned kFactorBytes = FACTOR_WORDS * 32 * sizeof(u64);
__device__ __forceinline__ void park_factors(const Factors &X, u64 *o)
{
    o[0 * 32] = X.e;
    o[1 * 32] = X.c12[0]; o[2 * 32] = X.c12[1];
    o[3 * 32] = X.c45[0]; o[4 * 32] = X.c45[1];
    o[5 * 32] = X.c68[0]; o[6 * 32] = X.c68[1];
    o[7 * 32] = X.c3; o[8 * 32] = X.c9;
    o[9 * 32] = pk(X.c7[0], X.c7[1]);
}
__device__ __forceinline__ void apply_parked(const u64 *o, Partials &S, int &cnt)
{
    Factors X;
    X.e = o[0 * 32];
    X.c12[0] = o[1 * 32]; X.c12[1] = o[2 * 32];
    X.c45[0] = o[3 * 32]; X.c45[1] = o[4 * 32];
    X.c68[0] = o[5 * 32]; X.c68[1] = o[6 * 32];
    X.c3 = o[7 * 32]; X.c9 = o[8 * 32];
    upk(o[9 * 32], X.c7[0], X.c7[1]);
    // a contributing pair has e = exp(-h) with h < 30, never zero; a skipped pair has e = 0 exactly
    cnt += (lo32(X.e) != 0.0f ? 1 : 0) + (hi32(X.e) != 0.0f ? 1 : 0);
    apply_factors<true>(X, S);
}

// one cell for the lane's two points, accumulated into the lane's partials: acc_t = fma(e, c_t, acc_t)
template <bool FULL>
__device__ __forceinline__ void accumulate_cell(const Cell4 &cA, const Cell4 &cB, const PointPk &A, const PointPk &B, Partials &S,
                                                int &cnt)
{
    Factors F;
    cell_factors<FULL>(cA, cB, A, B, F, cnt);
    apply_factors<FULL>(F, S);
}

// Where the warp's points come from: AoS float2 in shared memory, sanitised and padded with the far-away
// point to a multiple of 64 (SMEM), or global memory with bounds checks (scans too long for the slot).
// ADDR (SMEM only): i is not a point index but the shared-window byte address of point A (see eval_warp)
template <bool SMEM, bool ADDR = false>
__device__ __forceinline__ void load_two(const float2 *pts, int n, int i, float2 &a, float2 &b)
{
    if (SMEM) {
        const unsigned sa = ADDR ? (unsigned)i : (unsigned)__cvta_generic_to_shared(pts) + 8u * (unsigned)i;
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(a.x), "=f"(a.y) : "r"(sa));
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2+256];" : "=f"(b.x), "=f"(b.y) : "r"(sa));
    } else {
        const float2 far = make_float2(1e18f, 1e18f);
        a = i < n ? sanitize(__ldg(pts + i)) : far;
        b = i + 32 < n ? sanitize(__ldg(pts + i + 32)) : far;
    }
}

// One iteration's worth of fetched state for a lane: its two transformed points and the K cell records of each
// (loads may still be in flight when the struct is handed on).
template <int OV>
struct Fetched {
    static constexpr int NC = OV ? 4 : 1;
    PointPk A, B;
    Cell4 cA[NC], cB[NC];
};

// How a level's cell records are stored (template parameter TABLE of the evaluation):
//   TABLE_DENSE  L.cells is the dense row-major table (scan-to-map, set_target)
//   TABLE_GHASH  L.cells is an open-addressing hash table in global memory keyed by the dense index (ndt2d_align_pairs,
//                general path): hash_mask + 1 records, key in the record's `n` word, sentinel record behind them
//   TABLE_SHASH  the valid cells of one target scan in SHARED memory (ndt2d_align_pairs, fused path): L.cells is the compact
//                array of 24-byte records, L.cnt the index of hash_mask + 1 four-entry buckets (see lookup_shared), and
//                L.zero_rec the number of the all-zero record that a failed lookup returns
enum { TABLE_DENSE = 0, TABLE_GHASH = 1, TABLE_SHASH = 2 };

struct LatticePk {
    unsigned nhx, nhy, njx;
    unsigned sentinel; // dense tables: index of the first of the njx + 2 all-zero records that follow the cells (the gather target of
                       // a point outside the lattice; sentinel + {0, 1, njx, njx + 1} are all zero records, so the four cells
                       // of an outside point need no test of their own). Global hash tables: the one zero record after the
                       // slots. Shared tables: the number of the zero record behind the compact array.
    unsigned mask;     // hash tables only: slots - 1
    unsigned outside;  // what lattice_base() returns for a point outside the lattice: `sentinel` for dense tables (the gather
                       // goes straight to the zero records); 0xffffffff for hash tables, where every smaller value is a cell key
    unsigned srec, sidx; // TABLE_SHASH: shared-window addresses of the record array and of the u32 slot index
    float st;          // stride in metres: local coordinate = fma(df, st, off)
    u64 off[4];        // per cell of the point: minus the cell centre relative to node (hx, hy): (-st/2, -st/2) for one
                       // grid; (-a st, -b st) for cell (a, b) of the four half-shifted grids
};

template <int OV>
__device__ __forceinline__ LatticePk lattice_pack(const LevelDev &L, int table)
{
    LatticePk G;
    G.nhx = (unsigned)L.nhx; G.nhy = (unsigned)L.nhy; G.njx = (unsigned)L.njx;
    G.mask = L.hash_mask;
    G.sentinel = table == TABLE_DENSE ? (unsigned)L.njx * (unsigned)L.njy : table == TABLE_GHASH ? L.hash_mask + 1u : L.zero_rec;
    G.outside = table != TABLE_DENSE ? 0xffffffffu : G.sentinel;
    G.srec = G.sidx = 0u;
    if (table == TABLE_SHASH) {
        G.srec = (unsigned)__cvta_generic_to_shared(L.cells);
        G.sidx = (unsigned)__cvta_generic_to_shared(L.cnt);
    }
    G.st = L.st;
    if (OV) {
#pragma unroll
        for (int k = 0; k < 4; ++k) G.off[k] = pk(-__fmul_rn((float)(k & 1), L.st), -__fmul_rn((float)(k >> 1), L.st));
    } else {
        const float h2 = __fmul_rn(0.5f, L.st);
        G.off[0] = G.off[1] = G.off[2] = G.off[3] = pk(-h2, -h2);
    }
    return G;
}

__device__ __forceinline__ unsigned locate_base(const PosePk &P, double xd, double yd, const LatticePk &G, u64 &df);
__device__ __forceinline__ unsigned locate_base(const PosePk &P, float x, float y, const LatticePk &G, u64 &df)
{
    return locate_base(P, (double)x, (double)y, G, df);
}
// (xd, yd): the point already widened to f64 (the sweep kernel stages the scan that way: the conversions are done once)
__device__ __forceinline__ unsigned locate_base(const PosePk &P, double xd, double yd, const LatticePk &G, u64 &df)
{
    const double fx = __fma_rn(P.ci, xd, __fma_rn(-P.si, yd, P.txi));
    const double fy = __fma_rn(P.si, xd, __fma_rn(P.ci, yd, P.tyi));
    float dfx, dfy;
    unsigned hx, hy;
    const unsigned wx = node_of(fx, hx, dfx), wy = node_of(fy, hy, dfy);
    df = pk(dfx, dfy);
    return lattice_base(wx, wy, hx, hy, G.nhx, G.nhy, G.njx, G.outside);
}

// slot of a cell key in a per-target hash table: Fibonacci hashing, bits 15.. of the product (tables have <= 2^16 slots)
__device__ __forceinline__ unsigned hash_slot(unsigned key, unsigned mask) { return ((key * 0x9E3779B1u) >> 15) & mask; }

// the point relative to the centre of its cell k (SPEC 4, v4): one f32 fma per coordinate
__device__ __forceinline__ u64 local_xy(const LatticePk &G, u64 df, int k) { return fma2(df, bc(G.st), G.off[k]); }

// TABLE_SHASH: the valid cells of one target in shared memory. Records are 24 bytes {mux, muy, B00, B01, B11, key}
// (B01 once, no count: the evaluation needs neither), appended in key order, followed by one all-zero record (key word
// 0xffffffff) for lookups that find nothing. The index is made of hash_mask + 1 BUCKETS of four u32 entries (one 128-bit
// shared load): a used entry is (key & 0x7fff) << 16 | record id, an empty one 0xffffffff, entries fill from the front;
// a key whose bucket hash_slot(key) is full goes to the next bucket. The common lookup is therefore branch-free - one
// bucket load, four tag compares, one record load, the record's own key word as the verdict - and only a full bucket or
// a false tag match (both rare: about one bucket in 300 overflows) sends the lane to the probing slow path.
static constexpr unsigned kSharedRecordBytes = 24;
__device__ __forceinline__ void lds_record(unsigned a, u64 &mu, u64 &b0, u64 &b1k)
{
    asm volatile("ld.shared.b64 %0, [%1];" : "=l"(mu) : "r"(a));
    asm volatile("ld.shared.b64 %0, [%1+8];" : "=l"(b0) : "r"(a));
    asm volatile("ld.shared.b64 %0, [%1+16];" : "=l"(b1k) : "r"(a));
}
__device__ __forceinline__ void lds_bucket(unsigned a, unsigned &e0, unsigned &e1, unsigned &e2, unsigned &e3)
{
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(e0), "=r"(e1), "=r"(e2), "=r"(e3) : "r"(a));
}
__device__ __forceinline__ Cell4 record_to_cell(u64 mu, u64 b0, u64 b1k, bool valid)
{
    Cell4 c;
    c.mu = mu;
    c.B0 = b0;
    c.B1 = pk(hi32(b0), lo32(b1k));            // (B01, B11)
    c.nv = pk(0.0f, valid ? 1.0f : 0.0f);
    return c;
}
// the probing lookup: buckets from hash_slot(key) on, every tag match verified against the record's key
static __device__ __noinline__ Cell4 lookup_shared_slow(unsigned srec, unsigned sidx, unsigned mask, unsigned zid, unsigned key)
{
    const unsigned tag = key & 0x7fffu;
    unsigned b = hash_slot(key, mask);
    u64 mu, b0, b1k;
    for (unsigned probes = 0; probes <= mask; ++probes) {
        unsigned e[4];
        lds_bucket(sidx + b * 16u, e[0], e[1], e[2], e[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if ((e[j] >> 16) == tag) {
                lds_record(srec + (e[j] & 0xffffu) * kSharedRecordBytes, mu, b0, b1k);
                if ((unsigned)__float_as_int(hi32(b1k)) == key) return record_to_cell(mu, b0, b1k, true);
            }
        }
        if (e[3] == 0xffffffffu) break;        // the bucket never filled up: the key is not in the table
        b = (b + 1u) & mask;
    }
    lds_record(srec + zid * kSharedRecordBytes, mu, b0, b1k);
    return record_to_cell(mu, b0, b1k, false);
}
// common path; `slow` is set when this lane has to take the probing path (key 0xffffffff = outside the lattice: no record)
__device__ __forceinline__ Cell4 lookup_shared(const LatticePk &G, unsigned key, bool &slow)
{
    const unsigned tagword = (key & 0x7fffu) << 16;
    unsigned e0, e1, e2, e3;
    lds_bucket(G.sidx + hash_slot(key, G.mask) * 16u, e0, e1, e2, e3);
    // entry ^ tagword is the bare record id (< 2^16) for an entry with this tag and >= 2^16 for every other one (an empty
    // entry keeps bit 31): the minimum of the four is the match, if there is one - 4 LOP3 + 3 VIMNMX instead of 12 compare/selects
    const unsigned m = min(min(e0 ^ tagword, e1 ^ tagword), min(e2 ^ tagword, e3 ^ tagword));
    const bool inside = key != 0xffffffffu;
    const bool tagged = inside && m < 0x10000u;
    u64 mu, b0, b1k;
    lds_record(G.srec + (tagged ? m : G.sentinel) * kSharedRecordBytes, mu, b0, b1k);
    const bool ok = tagged && (unsigned)__float_as_int(hi32(b1k)) == key;
    slow = inside && !ok && (tagged || e3 != 0xffffffffu);   // a false tag match, or a full bucket without a match
    return record_to_cell(mu, b0, b1k, ok);
}

// P64 (score-only kernels with the scan staged in shared memory): pts holds double2 per point, r and j are not needed
template <int OV, bool SMEM, int TABLE = TABLE_DENSE, bool P64 = false, bool ADDR = false>
__device__ __forceinline__ void fetch(const float4 *__restrict__ cells, const LatticePk &G, const PosePk &P, const float2 *pts,
                                      int n, int i, Fetched<OV> &F)
{
    unsigned bA, bB;
    if (P64) {
        double2 a, b;
        if (ADDR) {     // i is the shared-window byte address of point A, 16 bytes per point
            asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a.x), "=d"(a.y) : "r"((unsigned)i));
            asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+512];" : "=d"(b.x), "=d"(b.y) : "r"((unsigned)i));
        } else {
            a = reinterpret_cast<const double2 *>(pts)[i];
            b = reinterpret_cast<const double2 *>(pts)[i + 32];
        }
        F.A.r = F.A.j = F.B.r = F.B.j = 0ull;
        bA = locate_base(P, a.x, a.y, G, F.A.df);
        bB = locate_base(P, b.x, b.y, G, F.B.df);
    } else {
        float2 a, b;
        load_two<SMEM, ADDR>(pts, n, i, a, b);
        rotate_point<true>(P, a.x, a.y, F.A);
        rotate_point<true>(P, b.x, b.y, F.B);
        bA = locate_base(P, a.x, a.y, G, F.A.df);
        bB = locate_base(P, b.x, b.y, G, F.B.df);
    }
    // K = 1: one record per point. K = 4: two rows of two adjacent records (64 contiguous bytes per row).
    // Outside the lattice: the zero records behind the table (invalid), so the gather needs no predicate.
    if (TABLE == TABLE_DENSE) {
#pragma unroll
        for (int k = 0; k < Fetched<OV>::NC; ++k) {
            const unsigned o = (k & 1) + (k >> 1) * G.njx;
            F.cA[k] = load_cell(cells, bA + o);
            F.cB[k] = load_cell(cells, bB + o);
        }
    } else if (TABLE == TABLE_SHASH) {
#pragma unroll
        for (int k = 0; k < Fetched<OV>::NC; ++k) {
            const unsigned o = (k & 1) + (k >> 1) * G.njx;
            const unsigned kA = bA == G.outside ? bA : bA + o, kB = bB == G.outside ? bB : bB + o;
            bool slowA, slowB;
            F.cA[k] = lookup_shared(G, kA, slowA);
            F.cB[k] = lookup_shared(G, kB, slowB);
            if (__any_sync(0xffffffffu, slowA || slowB)) {
                if (slowA) F.cA[k] = lookup_shared_slow(G.srec, G.sidx, G.mask, G.sentinel, kA);
                if (slowB) F.cB[k] = lookup_shared_slow(G.srec, G.sidx, G.mask, G.sentinel, kB);
            }
        }
    } else {
        const bool inA = bA != G.outside, inB = bB != G.outside;
        // hash tables: the first probes of all cells go out together; only then are the (rare) collisions chased
        unsigned sA[Fetched<OV>::NC], sB[Fetched<OV>::NC];
#pragma unroll
        for (int k = 0; k < Fetched<OV>::NC; ++k) {
            const unsigned o = (k & 1) + (k >> 1) * G.njx;
            sA[k] = inA ? hash_slot(bA + o, G.mask) : G.sentinel;
            sB[k] = inB ? hash_slot(bB + o, G.mask) : G.sentinel;
            F.cA[k] = load_cell(cells, sA[k]);
            F.cB[k] = load_cell(cells, sB[k]);
        }
#pragma unroll
        for (int k = 0; k < Fetched<OV>::NC; ++k) {
            const unsigned o = (k & 1) + (k >> 1) * G.njx;
            // (tables are at most 2/3 full, so an empty slot ends every chain; the bound only guards against a corrupt table)
            if (inA) {
                for (unsigned probes = 0; probes <= G.mask; ++probes) {
                    const unsigned key = (unsigned)__float_as_int(lo32(F.cA[k].nv));
                    if (key == bA + o || key == kEmptyKey) break;
                    sA[k] = (sA[k] + 1u) & G.mask;
                    F.cA[k] = load_cell(cells, sA[k]);
                }
                if ((unsigned)__float_as_int(lo32(F.cA[k].nv)) != bA + o) F.cA[k].nv = 0ull;   // not found: invalid
            }
            if (inB) {
                for (unsigned probes = 0; probes <= G.mask; ++probes) {
                    const unsigned key = (unsigned)__float_as_int(lo32(F.cB[k].nv));
                    if (key == bB + o || key == kEmptyKey) break;
                    sB[k] = (sB[k] + 1u) & G.mask;
                    F.cB[k] = load_cell(cells, sB[k]);
                }
                if ((unsigned)__float_as_int(lo32(F.cB[k].nv)) != bB + o) F.cB[k].nv = 0ull;
            }
        }
    }
}

// one step's cells for the lane's two points, accumulated in cell order (SPEC 4)
template <int OV, bool FULL>
__device__ __forceinline__ void accumulate_step(const LatticePk &G, Fetched<OV> &F, Partials &S, int &cnt)
{
#pragma unroll
    for (int k = 0; k < Fetched<OV>::NC; ++k) {
        F.A.XY = local_xy(G, F.A.df, k);
        F.B.XY = local_xy(G, F.B.df, k);
        accumulate_cell<FULL>(F.cA[k], F.cB[k], F.A, F.B, S, cnt);
    }
}

// SPEC 4 for one warp. Lane l owns points 64 j + l (A) and 64 j + 32 + l (B), i.e. partials l and l + 32: each of the
// two gather requests of an iteration then covers 32 consecutive beams (few distinct cache lines per request).
// TR (FULL only): finish with the transposed reduction; E.v[0] is then sum number E.slot, the other E.v are unset.
template <bool FULL, bool TR>
__device__ __forceinline__ void finish_partials(const Partials &S, int cnt, int lane, Eval &E);

// No helper warps (every caller but k_align<..., HELP>): the warp evaluates all its steps itself.
struct NoHelp {
    static constexpr bool on = false;
    __device__ __forceinline__ unsigned own_steps(unsigned nsteps) const { return nsteps; }
    __device__ __forceinline__ void finish(Partials &, int &, int) const {}
};

// TABLE: how L's records are stored (TABLE_DENSE / TABLE_GHASH / TABLE_SHASH), resolved in fetch().
// Help (SMEM only): the warp evaluates the first help.own_steps(steps) 64-point steps; help.finish()
// then applies the factors of the remaining steps, computed and parked by other warps, in step order (HelpPlan in
// ndt2d_align.cuh) - SPEC 4's summation order is kept, so the sums are the same bits.
template <int OV, bool FULL, bool SMEM, bool TR = false, int TABLE = TABLE_DENSE, bool P64 = false, class Help = NoHelp>
__device__ __forceinline__ void eval_warp(const LevelDev &L, const float2 *pts, int n, const Pose32 &q, int lane, Eval &E,
                                          const Help help = Help())
{
    Partials S;
    S.s0 = S.s3 = S.s9 = 0ull;
    S.s7[0] = S.s7[1] = 0.0f;
#pragma unroll
    for (int k = 0; k < 2; ++k) S.s12[k] = S.s45[k] = S.s68[k] = 0ull;
    int cnt = 0;
    const float4 *__restrict__ cells = L.cells;
    const PosePk P = pose_pack(q);
    const LatticePk G = lattice_pack<OV>(L, TABLE);
    const int npad = (n + 63) & ~63;
    if (SMEM) {
        // the staged scan is walked by its shared-window address: one register is loop counter and load address at once (as
        // pts[i] the compiler recomputed slot base + warp * capacity + i with two multiply-adds and a constant load per step)
        constexpr unsigned PB = P64 ? 16u : 8u;     // bytes per staged point
        const unsigned s0 = (unsigned)__cvta_generic_to_shared(pts) + PB * (unsigned)lane;
        const unsigned s1 = s0 + PB * (Help::on ? 64u * help.own_steps((unsigned)npad >> 6) : (unsigned)npad);
#pragma unroll 1
        for (unsigned sa = s0; sa < s1; sa += 64u * PB) {
            Fetched<OV> cur;
            fetch<OV, SMEM, TABLE, P64, true>(cells, G, P, pts, n, (int)sa, cur);
            accumulate_step<OV, FULL>(G, cur, S, cnt);
        }
        if (Help::on) help.finish(S, cnt, lane);
    } else {
#pragma unroll 1
        for (int i = lane; i < npad; i += 64) {
            Fetched<OV> cur;
            fetch<OV, SMEM, TABLE, P64>(cells, G, P, pts, n, i, cur);
            accumulate_step<OV, FULL>(G, cur, S, cnt);
        }
    }
    finish_partials<FULL, TR>(S, cnt, lane, E);
}

// SPEC 4: D[l] = (double)P[l] + (double)P[l+32], then the butterfly (plain: every lane gets all ten sums; TR: the
// transposed form, E.v[0] = sum number E.slot)
template <bool FULL, bool TR>
__device__ __forceinline__ void finish_partials(const Partials &S, int cnt, int lane, Eval &E)
{
    E.slot = 0;
    if (FULL) {
        double D[10];
        D[0] = (double)lo32(S.s0) + (double)hi32(S.s0);
        D[1] = (double)lo32(S.s12[0]) + (double)lo32(S.s12[1]);
        D[2] = (double)hi32(S.s12[0]) + (double)hi32(S.s12[1]);
        D[3] = (double)lo32(S.s3) + (double)hi32(S.s3);
        D[4] = (double)lo32(S.s45[0]) + (double)lo32(S.s45[1]);
        D[5] = (double)hi32(S.s45[0]) + (double)hi32(S.s45[1]);
        D[6] = (double)lo32(S.s68[0]) + (double)lo32(S.s68[1]);
        D[7] = (double)S.s7[0] + (double)S.s7[1];
        D[8] = (double)hi32(S.s68[0]) + (double)hi32(S.s68[1]);
        D[9] = (double)lo32(S.s9) + (double)hi32(S.s9);
        if (TR) {
            E.v[0] = warp_sum10_transposed(D, lane, E.slot);
        } else {
#pragma unroll
            for (int t = 0; t < 10; ++t) E.v[t] = warp_sum(D[t]);
        }
    } else {
        E.v[0] = warp_sum((double)lo32(S.s0) + (double)hi32(S.s0));
#pragma unroll
        for (int t = 1; t < 10; ++t) E.v[t] = 0.0;
    }
    E.count = __reduce_add_sync(0xffffffffu, cnt);
}

// ---- SPEC 5: damped 3x3 solve in f64, closed form, no contraction (-fmad=false). g = v[1..3], H6 = v[4..9] ----
// Adjugate over determinant with Sylvester's criterion as the positive-definiteness test: about 60 instructions
// and one reciprocal, where a Cholesky factorisation costs three square roots and twelve divisions (each ~25
// instructions in f64). __drcp_rn is the correctly rounded reciprocal, i.e. the oracle's 1.0 / det bit for bit.
__device__ __forceinline__ bool solve3(const double *g, const double *H6, double lambda, double d[3])
{
    const double A00 = H6[0] + lambda * fmax(fabs(H6[0]), 1e-9);
    const double A11 = H6[3] + lambda * fmax(fabs(H6[3]), 1e-9);
    const double A22 = H6[5] + lambda * fmax(fabs(H6[5]), 1e-9);
    const double A01 = H6[1], A02 = H6[2], A12 = H6[4];
    const double C00 = A11 * A22 - A12 * A12;
    const double C01 = A02 * A12 - A01 * A22;
    const double C02 = A01 * A12 - A02 * A11;
    const double C11 = A00 * A22 - A02 * A02;
    const double C12 = A01 * A02 - A00 * A12;
    const double C22 = A00 * A11 - A01 * A01;
    const double det = (A00 * C00 + A01 * C01) + A02 * C02;
    if (!(A00 > 0.0) || !(C22 > 0.0) || !(det > 0.0)) return false;
    const double r = __drcp_rn(det);
    d[0] = -(((C00 * g[0] + C01 * g[1]) + C02 * g[2]) * r);
    d[1] = -(((C01 * g[0] + C11 * g[1]) + C12 * g[2]) * r);
    d[2] = -(((C02 * g[0] + C12 * g[1]) + C22 * g[2]) * r);
    return true;
}

} // namespace ndt2d
