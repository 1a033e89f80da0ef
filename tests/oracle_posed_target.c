/*
 * SPEC 7.2 (target from posed scans) on top of the CPU spec oracle - test infrastructure, NOT product code.
 *
 * The oracle's source is compiled into this library unchanged, so every oracle_* entry point is here with the oracle's
 * own lattice, level set-up and finalisation; this file adds the one thing SPEC 7.2 changes: the points reach SPEC 2-3
 * as f64 map coordinates (the scan point transformed by its pose, not rounded to f32) instead of widened f32 points.
 * Built by tests/posed_oracle.py with the oracle's flags (-ffp-contract=off -mfma: fma() is one rounding).
 */
#include "ndt2d_oracle.c"

/* SPEC 3 for one point given in f64 map coordinates: the oracle's accumulate() with (double)X replaced by X */
static void accumulate_point_f64(level_t *L, double X, double Y)
{
    const int K = L->ov ? 2 : 1;
    int hx, hy;
    if (!lattice(L, (X - (double)L->ox) * L->inv_std, (Y - (double)L->oy) * L->inv_std, &hx, &hy, NULL, NULL)) return;
    for (int b = 0; b < K; ++b) for (int a = 0; a < K; ++a) {
        int jx = hx + a, jy = hy + b;
        double cx = (double)L->ox + ((double)(jx - L->ov)) * (double)L->st + 0.5 * (double)L->res;
        double cy = (double)L->oy + ((double)(jy - L->ov)) * (double)L->st + 0.5 * (double)L->res;
        double dx = X - cx, dy = Y - cy;
        int64_t qx = llrint(dx * L->qs), qy = llrint(dy * L->qs);
        size_t c = (size_t)jy * (size_t)L->njx + (size_t)jx;
        L->n[c] += 1;
        int64_t *s = L->s + 5 * c;
        s[0] += qx; s[1] += qy; s[2] += qx * qx; s[3] += qx * qy; s[4] += qy * qy;
    }
}

/* SPEC 7.2: XY[2i], XY[2i+1] = the f64 map coordinates of posed scan point i; NaN for a point with a non-finite coordinate
 * (outside every lattice, not part of the bounding box). Returns the point count, or -1 on bad arguments. */
static int64_t posed_points(const float *xy, const int64_t *offsets, int nscans, const double *poses, double **XY)
{
    *XY = NULL;
    if (nscans < 0 || (nscans > 0 && offsets[0] != 0)) return -1;
    for (int b = 0; b < nscans; ++b) {
        if (offsets[b + 1] < offsets[b]) return -1;
        for (int t = 0; t < 3; ++t) if (!isfinite(poses[3 * b + t])) return -1;
    }
    const int64_t n = nscans > 0 ? offsets[nscans] : 0;
    *XY = (double *)malloc((size_t)(n > 0 ? n : 1) * 2 * sizeof(double));
    if (!*XY) return -1;
    for (int b = 0; b < nscans; ++b) {
        double sn, cs;
        oracle_sincos(poses[3 * b + 2], &sn, &cs);
        const double p0 = poses[3 * b], p1 = poses[3 * b + 1];
        for (int64_t i = offsets[b]; i < offsets[b + 1]; ++i) {
            const float x = xy[2 * i], y = xy[2 * i + 1];
            double X = NAN, Y = NAN;
            if (isfinite(x) && isfinite(y)) {
                const double xd = (double)x, yd = (double)y;
                X = fma(cs, xd, fma(-sn, yd, p0));
                Y = fma(sn, xd, fma(cs, yd, p1));
            }
            (*XY)[2 * i] = X; (*XY)[2 * i + 1] = Y;
        }
    }
    return n;
}

/* set (add == 0) or add (SPEC 7; without a target: set). Auto-fit: SPEC 2 on the f32 roundings of the map coordinates -
 * the oracle's level_setup() takes the bounding box of the two corner points of that box, which is the box itself. */
static int target_scans(oracle_matcher *m, int add, const float *xy, const int64_t *offsets, int nscans, const double *poses)
{
    double *XY;
    const int64_t n = posed_points(xy, offsets, nscans, poses, &XY);
    if (n < 0) { free(XY); return 1; }
    int rc = 0;
    if (!add || !m->has_target) {
        drop_target(m);
        float xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
        for (int64_t i = 0; i < n; ++i) {
            const float x = (float)XY[2 * i], y = (float)XY[2 * i + 1];
            if (!isfinite(x) || !isfinite(y)) continue;
            if (x < xmin) xmin = x;
            if (x > xmax) xmax = x;
            if (y < ymin) ymin = y;
            if (y > ymax) ymax = y;
        }
        const float corners[4] = {xmin, ymin, xmax, ymax};
        const int ncorners = xmin <= xmax ? 2 : 0;
        for (int l = 0; l < m->nlevels && !rc; ++l) rc = level_setup(m, l, corners, ncorners);
        if (rc) drop_target(m);
        else m->has_target = 1;
    }
    for (int l = 0; l < m->nlevels && !rc; ++l) {
        for (int64_t i = 0; i < n; ++i) accumulate_point_f64(&m->lv[l], XY[2 * i], XY[2 * i + 1]);
        finalize(&m->lv[l], &m->prm);
    }
    free(XY);
    return rc;
}

int oracle_set_target_scans(oracle_matcher *m, const float *xy, const int64_t *offsets, int nscans, const double *poses)
{
    return target_scans(m, 0, xy, offsets, nscans, poses);
}

int oracle_add_target_scans(oracle_matcher *m, const float *xy, const int64_t *offsets, int nscans, const double *poses)
{
    return target_scans(m, 1, xy, offsets, nscans, poses);
}
