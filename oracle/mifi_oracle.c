/*
 * oracle/mifi_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement (plain C99) of the reference's
 * horizontal-regridding hot path.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load the library built from this file; the product library
 * (libfimex_b200.so) never links, loads or calls it.
 *
 * Every function names the reference lines it follows (paths relative to /root/reference).  The
 * restatement is validated two ways (tests/test_oracle_*.py):
 *   1. against the reference's own known-answer tests (test/testInterpolation.cc:49-155, 265-654);
 *   2. bit-for-bit against oracle/_ref/libmifi_ref.so = the reference's src/interpolation.c compiled
 *      unmodified where it lies (oracle/Makefile), on seeded random and adversarial inputs; golden
 *      vectors produced from that library are committed under tests/golden/.
 * The C++ classes CachedInterpolation / CachedForwardInterpolation / CachedVectorReprojection and the
 * coord-NN search of CDMInterpolator cannot be compiled here (Boost, libxml2, udunits2, NetCDF absent),
 * so for them this restatement is pinned only by the reference's scalar kernels they call.
 *
 * Build: gcc -std=gnu99 -O2 -ffp-contract=off -fopenmp (no FMA contraction: x86-64 -O2 emits none for
 * the reference either, SURVEY.md 8a trap 7).
 */
#include "shim/proj_api.h"

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_OK 1
#define ORC_ERROR (-1)
#define ORC_PI 3.1415926535897932384626433832795 /* MIFI_PI, include/fimex/mifi_constants.h:42 */
#define ORC_PROJ_AXIS 0
#define ORC_LONGITUDE 1
#define ORC_LATITUDE 2

/* method numbering of include/fimex/mifi_constants.h:52-147 */
enum {
    ORC_NN = 0,
    ORC_BILINEAR,
    ORC_BICUBIC,
    ORC_COORD_NN,
    ORC_COORD_NN_KD,
    ORC_FWD_SUM,
    ORC_FWD_MEAN,
    ORC_FWD_MEDIAN,
    ORC_FWD_MAX,
    ORC_FWD_MIN,
    ORC_FWD_UNDEF_SUM,
    ORC_FWD_UNDEF_MEAN,
    ORC_FWD_UNDEF_MEDIAN,
    ORC_FWD_UNDEF_MAX,
    ORC_FWD_UNDEF_MIN
};

static float orc_undef_f(void)
{
    return nanf(""); /* MIFI_UNDEFINED_F, mifi_constants.h:254: canonical quiet NaN 0x7fc00000 */
}

/* src/interpolation.c:66-101 (including the forward_undef_min -> FORWARD_MIN quirk, :97-98) */
int orc_string_to_method(const char* s)
{
    static const struct {
        const char* name;
        int m;
    } tab[] = {{"bilinear", ORC_BILINEAR},
               {"nearestneighbor", ORC_NN},
               {"bicubic", ORC_BICUBIC},
               {"coord_nearestneighbor", ORC_COORD_NN},
               {"coord_kdtree", ORC_COORD_NN_KD},
               {"forward_sum", ORC_FWD_SUM},
               {"forward_mean", ORC_FWD_MEAN},
               {"forward_median", ORC_FWD_MEDIAN},
               {"forward_max", ORC_FWD_MAX},
               {"forward_min", ORC_FWD_MIN},
               {"forward_undef_sum", ORC_FWD_UNDEF_SUM},
               {"forward_undef_mean", ORC_FWD_UNDEF_MEAN},
               {"forward_undef_median", ORC_FWD_UNDEF_MEDIAN},
               {"forward_undef_max", ORC_FWD_UNDEF_MAX},
               {"forward_undef_min", ORC_FWD_MIN}};
    for (size_t i = 0; i < sizeof(tab) / sizeof(tab[0]); ++i)
        if (strcmp(tab[i].name, s) == 0)
            return tab[i].m;
    return -1;
}

/* ------------------------------------------------------------------------------------------------
 * A9  mifi_points2position, src/interpolation.c:148-217 (+ bsearchDoubleIndex :124-146)
 * ---------------------------------------------------------------------------------------------- */
void orc_points2position(double* pts, long n, const double* axis, int num, int axis_type)
{
    const int ascending = axis[0] < axis[num - 1];
    int circular = 0;
    if (axis_type == ORC_LONGITUDE) {
        if (axis[0] < 0 || axis[num - 1] < 0) { /* axis is -180..180: fold points > pi (:157-161) */
            for (long i = 0; i < n; ++i)
                if (pts[i] > ORC_PI)
                    pts[i] -= 2 * ORC_PI;
        } else { /* axis is 0..360: fold negative points (:163-166) */
            for (long i = 0; i < n; ++i)
                if (pts[i] < 0)
                    pts[i] += 2 * ORC_PI;
        }
        double next = axis[num - 1] + (axis[1] - axis[0]) * 1.01; /* :168 */
        if (ascending) {
            next -= 2 * ORC_PI;
            circular = (next >= axis[0]);
        } else {
            next += 2 * ORC_PI;
            circular = (next <= axis[0]);
        }
    }
    for (long i = 0; i < n; ++i) {
        const double key = pts[i];
        if (!isfinite(key)) { /* :183-186 */
            pts[i] = -999.;
            continue;
        }
        /* binary search with the reference's exact probe sequence (:127-145) */
        int first = 0, last = num - 1, pos = 0, cmp = 0;
        while (first <= last) {
            pos = (first + last) / 2;
            const double b = axis[pos];
            cmp = (key > b) ? 1 : ((key == b) ? 0 : -1);
            if (!ascending)
                cmp = -cmp;
            if (cmp > 0)
                first = pos + 1;
            else if (cmp < 0)
                last = pos - 1;
            else
                break;
        }
        if (cmp == 0) {
            pts[i] = (double)pos;
            continue;
        }
        int seg = (cmp > 0) ? pos + 1 : pos; /* index of the first axis element "after" key */
        if (seg == num)
            seg--; /* extrapolate right (:193-194) */
        else if (seg == 0)
            seg++; /* extrapolate left (:195-196) */
        const double slope = axis[seg] - axis[seg - 1];
        const double offset = axis[seg] - (slope * seg);
        double apos = (key - offset) / slope;
        if (circular && apos <= -0.5)
            apos += num;
        if (circular && apos > (num - 0.5))
            apos -= num;
        pts[i] = apos;
    }
}

/* ------------------------------------------------------------------------------------------------
 * A6-A8  per-point gathers, src/interpolation.c:862-1028.  `lvl` = ix*iy is the level stride of the
 * [z][y][x] array (mifi_3d_array_position, include/fimex/interpolation.h:423-426).
 * ---------------------------------------------------------------------------------------------- */
static void orc_fill_undef(float* out, int iz)
{
    for (int z = 0; z < iz; ++z)
        out[z] = orc_undef_f();
}

/* A6 :862-879 */
void orc_get_values_nn(const float* in, float* out, double x, double y, int ix, int iy, int iz)
{
    const int rx = (int)lround(x), ry = (int)lround(y); /* the reference narrows to int (:864-865) */
    if (rx < 0 || rx >= ix || ry < 0 || ry >= iy) {
        orc_fill_undef(out, iz);
        return;
    }
    const size_t lvl = (size_t)ix * iy;
    const float* p = in + (size_t)ry * ix + rx;
    for (int z = 0; z < iz; ++z, p += lvl)
        out[z] = *p;
}

/* A7 :881-957.  Trap 4 (:936 `y0 <= iy`): the reference reads row iy (out of bounds) for x in an edge
 * strip and y in [iy-0.5, iy+0.5); that is undefined behaviour, so this restatement (and the GPU path)
 * return NaN there.  orc_bilinear_is_ub() reports exactly that set so parity checks can mask it. */
int orc_bilinear_is_ub(double x, double y, int ix, int iy)
{
    const int x0 = (int)floor(x), y0 = (int)floor(y);
    if (0 <= x0 && x0 + 1 < ix)
        return 0;
    const int rx = (int)lround(x);
    if (rx < 0 || rx >= ix)
        return 0;
    if (0 <= y0 && y0 + 1 < iy)
        return 0;
    return lround(y) == iy;
}

void orc_get_values_bilinear(const float* in, float* out, double x, double y, int ix, int iy, int iz)
{
    const size_t lvl = (size_t)ix * iy;
    const int x0 = (int)floor(x), y0 = (int)floor(y);
    const float xf = (float)(x - x0), yf = (float)(y - y0); /* :885,888: fp64 subtract, then to float */
    const int x_in = (0 <= x0) && (x0 + 1 < ix);
    const int y_in = (0 <= y0) && (y0 + 1 < iy);
    if (x_in && y_in) { /* :889-902 */
        const float* p = in + (size_t)y0 * ix + x0;
        for (int z = 0; z < iz; ++z, p += lvl) {
            const float top = (1.f - xf) * p[0] + xf * p[1];
            const float bot = (1.f - xf) * p[ix] + xf * p[ix + 1];
            out[z] = (1.f - yf) * top + yf * bot;
        }
    } else if (x_in) { /* :903-920: outer half cell in y -> linear in x on the nearest row */
        const int ry = (int)lround(y);
        if (ry < 0 || ry >= iy) {
            orc_fill_undef(out, iz);
            return;
        }
        const float* p = in + (size_t)ry * ix + x0;
        for (int z = 0; z < iz; ++z, p += lvl)
            out[z] = (1.f - xf) * p[0] + xf * p[1];
    } else {
        const int rx = (int)lround(x); /* :922 */
        if (rx < 0 || rx >= ix) {
            orc_fill_undef(out, iz);
            return;
        }
        if (y_in) { /* :925-933: nearest in x, linear in y */
            const float* p = in + (size_t)y0 * ix + rx;
            for (int z = 0; z < iz; ++z, p += lvl)
                out[z] = (1 - yf) * p[0] + (yf * p[ix]);
        } else { /* :935-947: nearest in both; ry == iy is the reference's out-of-bounds read */
            const int ry = (int)lround(y);
            if (ry < 0 || ry >= iy) {
                orc_fill_undef(out, iz);
                return;
            }
            const float* p = in + (size_t)ry * ix + rx;
            for (int z = 0; z < iz; ++z, p += lvl)
                out[z] = *p;
        }
    }
}

/* weights of the a = -0.5 cubic convolution: w[i] = sum_j T[j] * M[j][i], M as :962-968 (already *0.5),
 * accumulated from 0 in j order exactly like :985-990 / :995-1000 */
static void orc_cubic_weights(double t, double w[4])
{
    static const double M[4][4] = {{0, 2, 0, 0}, {-1, 0, 1, 0}, {2, -5, 4, -1}, {-1, 3, -3, 1}};
    double T[4];
    T[0] = 1;
    T[1] = t;
    T[2] = t * t;
    T[3] = T[2] * t;
    for (int i = 0; i < 4; ++i) {
        double acc = 0;
        for (int j = 0; j < 4; ++j)
            acc += T[j] * (M[j][i] * .5);
        w[i] = acc;
    }
}

/* A8 :959-1028 */
void orc_get_values_bicubic(const float* in, float* out, double x, double y, int ix, int iy, int iz)
{
    const int x0 = (int)floor(x), y0 = (int)floor(y);
    if (!(1 <= x0 && x0 + 2 < ix && 1 <= y0 && y0 + 2 < iy)) { /* :975-976, no edge fallback */
        orc_fill_undef(out, iz);
        return;
    }
    double wx[4], wy[4];
    orc_cubic_weights(x - x0, wx);
    orc_cubic_weights(y - y0, wy);
    const size_t lvl = (size_t)ix * iy;
    const float* p = in + (size_t)(y0 - 1) * ix + (x0 - 1);
    for (int z = 0; z < iz; ++z, p += lvl) {
        float acc = 0; /* :1005: the accumulator is a float, re-rounded after every row (:1019) */
        for (int r = 0; r < 4; ++r) {
            const float* row = p + (size_t)r * ix;
            double rowval = 0; /* XMF[r], :1012-1016 */
            for (int c = 0; c < 4; ++c)
                rowval += wx[c] * (double)row[c];
            acc = (float)(acc + rowval * wy[r]);
        }
        out[z] = acc;
    }
}

/* ------------------------------------------------------------------------------------------------
 * A10  mifi_project_values / mifi_project_axes, src/interpolation.c:1158-1244 (arithmetic is PROJ's;
 * see oracle/pj_oracle.c)
 * ---------------------------------------------------------------------------------------------- */
static int orc_open_pair(const char* a, const char* b, projPJ* pa, projPJ* pb)
{
    *pa = pj_init_plus(a);
    if (!*pa)
        return ORC_ERROR;
    *pb = pj_init_plus(b);
    if (!*pb) {
        pj_free(*pa);
        return ORC_ERROR;
    }
    return ORC_OK;
}

int orc_project_values(const char* proj_in, const char* proj_out, double* x, double* y, long n)
{
    projPJ pi, po;
    if (orc_open_pair(proj_in, proj_out, &pi, &po) != ORC_OK)
        return ORC_ERROR;
    double* z = (double*)calloc((size_t)(n > 0 ? n : 1), sizeof(double));
    int rc = pj_transform(pi, po, n, 0, x, y, z);
    free(z);
    pj_free(pi);
    pj_free(po);
    return rc == 0 ? ORC_OK : ORC_ERROR;
}

int orc_project_axes(const char* proj_in, const char* proj_out, const double* xax, const double* yax, int ix, int iy, double* xo,
                     double* yo)
{
    for (int y = 0; y < iy; ++y)
        for (int x = 0; x < ix; ++x) {
            xo[(size_t)y * ix + x] = xax[x];
            yo[(size_t)y * ix + x] = yax[y];
        }
    return orc_project_values(proj_in, proj_out, xo, yo, (long)ix * iy);
}

/* A11 convertAxis :221-229 */
static void orc_convert_axis(const double* in, int n, int type, double* out)
{
    for (int i = 0; i < n; ++i)
        out[i] = (type == ORC_LONGITUDE || type == ORC_LATITUDE) ? DEG_TO_RAD * in[i] : in[i];
}

/* A12 mifi_interpolate_f :231-297 (heap instead of the reference's stack VLAs) */
int orc_interpolate_f(int method, const char* proj_in, const float* in, const double* in_x, const double* in_y, int in_xt, int in_yt,
                      int ix, int iy, int iz, const char* proj_out, float* out, const double* out_x, const double* out_y, int out_xt,
                      int out_yt, int ox, int oy)
{
    if (method != ORC_NN && method != ORC_BILINEAR && method != ORC_BICUBIC)
        return ORC_ERROR;
    const size_t on = (size_t)ox * oy;
    double* ax = (double*)malloc(sizeof(double) * (size_t)(ix + iy + ox + oy));
    double* px = (double*)malloc(sizeof(double) * on);
    double* py = (double*)malloc(sizeof(double) * on);
    float* col = (float*)malloc(sizeof(float) * (size_t)iz);
    double *ixa = ax, *iya = ax + ix, *oxa = iya + iy, *oya = oxa + ox;
    orc_convert_axis(in_x, ix, in_xt, ixa);
    orc_convert_axis(in_y, iy, in_yt, iya);
    orc_convert_axis(out_x, ox, out_xt, oxa);
    orc_convert_axis(out_y, oy, out_yt, oya);
    /* :257: the reference ignores the return value of mifi_project_axes */
    orc_project_axes(proj_out, proj_in, oxa, oya, ox, oy, px, py);
    orc_points2position(px, (long)on, ixa, ix, in_xt);
    orc_points2position(py, (long)on, iya, iy, in_yt);
    for (size_t i = 0; i < on; ++i) {
        if (method == ORC_NN)
            orc_get_values_nn(in, col, px[i], py[i], ix, iy, iz);
        else if (method == ORC_BILINEAR)
            orc_get_values_bilinear(in, col, px[i], py[i], ix, iy, iz);
        else
            orc_get_values_bicubic(in, col, px[i], py[i], ix, iy, iz);
        for (int z = 0; z < iz; ++z)
            out[(size_t)z * on + i] = col[z];
    }
    free(ax);
    free(px);
    free(py);
    free(col);
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------------
 * A15  vector-rotation matrix, src/interpolation.c:311-438 (points_proj_delta), :441-521 (delta
 * selection), :607-788 (the three public entry points)
 * ---------------------------------------------------------------------------------------------- */
static double orc_bearing(double lat0, double lon0, double lat1, double lon1)
{
    /* :311-329 */
    const double dlon = lon0 - lon1;
    return atan2(sin(dlon) * cos(lat1), cos(lat0) * sin(lat1) - sin(lat0) * cos(lat1) * cos(dlon));
}

static int orc_matrix_from_deltas(projPJ in_pj, projPJ out_pj, const double* in_x, const double* in_y, const double* out_x,
                                  const double* out_y, double dx, double dy, long on, double* matrix)
{
    double* tx = (double*)malloc(sizeof(double) * (size_t)on);
    double* ty = (double*)malloc(sizeof(double) * (size_t)on);
    double* tz = (double*)calloc((size_t)on, sizeof(double));
    const int ll = pj_is_latlong(out_pj);
    int rc = ORC_OK;
    /* step along x (:350-381) */
    for (long i = 0; i < on; ++i) {
        tx[i] = in_x[i] + dx;
        ty[i] = in_y[i];
    }
    if (pj_transform(in_pj, out_pj, on, 0, tx, ty, tz) != 0) {
        rc = ORC_ERROR;
        goto done;
    }
    for (long i = 0; i < on; ++i) {
        double phi;
        if (ll) {
            phi = orc_bearing(out_y[i], out_x[i], ty[i], tx[i]);
        } else {
            phi = atan2(ty[i] - out_y[i], tx[i] - out_x[i]);
            if (!(dx > 0))
                phi += ORC_PI;
        }
        matrix[4 * i] = phi;
    }
    /* step along y (:391-433) */
    for (long i = 0; i < on; ++i) {
        tx[i] = in_x[i];
        ty[i] = in_y[i] + dy;
        tz[i] = 0;
    }
    if (pj_transform(in_pj, out_pj, on, 0, tx, ty, tz) != 0) {
        rc = ORC_ERROR;
        goto done;
    }
    for (long i = 0; i < on; ++i) {
        double phi0;
        if (ll) { /* x-step result is discarded for lat/long targets (:408-412) */
            phi0 = orc_bearing(out_y[i], out_x[i], ty[i], tx[i]);
            if (!(dy > 0))
                phi0 += ORC_PI;
        } else {
            double phix = -1 * atan2(tx[i] - out_x[i], ty[i] - out_y[i]);
            if (!(dy > 0))
                phix += ORC_PI;
            phi0 = .5 * (phix + matrix[4 * i]); /* :424, no wrap handling */
        }
        const double c = cos(phi0), s = sin(phi0);
        matrix[4 * i + 0] = c;
        matrix[4 * i + 1] = s;
        matrix[4 * i + 2] = -1 * s;
        matrix[4 * i + 3] = phi0;
    }
done:
    free(tx);
    free(ty);
    free(tz);
    return rc;
}

/* :441-521: both deltas are derived from the x field (trap 11) */
static void orc_pick_deltas(const double* in_x, int ox, int oy, double* dx, double* dy)
{
    const double eps = 1e-3;
    double d;
    if (ox > 1 && oy > 1) {
        d = eps * (in_x[(size_t)ox + 1] - in_x[0]);
        const size_t hx = (size_t)ox / 2, hy = (size_t)oy / 2;
        const double d2 = eps * (in_x[(hy + 1) * ox + (hx + 1)] - in_x[hy * ox + hx]);
        d += d2;
        d /= 2;
    } else if (ox > 1) {
        d = eps * (in_x[1] - in_x[0]);
    } else if (oy > 1) {
        d = eps * (in_x[(size_t)ox] - in_x[0]);
    } else {
        d = (in_x[0] > 1) ? (in_x[0] * eps) : eps;
    }
    *dx = d;
    *dy = d;
    if (fabs(*dx) < 1e-9 || fabs(*dy) < 1e-9) { /* :509-513 */
        *dx = eps;
        *dy = eps;
    }
}

/* mifi_get_vector_reproject_matrix :719-788 */
int orc_vector_matrix(const char* proj_in, const char* proj_out, const double* out_x_axis, const double* out_y_axis, int xt, int yt, int ox,
                      int oy, double* matrix)
{
    projPJ pi, po;
    if (orc_open_pair(proj_in, proj_out, &pi, &po) != ORC_OK)
        return ORC_ERROR;
    const size_t on = (size_t)ox * oy;
    double* xa = (double*)malloc(sizeof(double) * (size_t)(ox + oy));
    double* ya = xa + ox;
    orc_convert_axis(out_x_axis, ox, xt, xa);
    orc_convert_axis(out_y_axis, oy, yt, ya);
    double* buf = (double*)malloc(sizeof(double) * on * 4);
    double *inx = buf, *iny = buf + on, *outx = buf + 2 * on, *outy = buf + 3 * on;
    double* z = (double*)calloc(on, sizeof(double));
    for (int y = 0; y < oy; ++y)
        for (int x = 0; x < ox; ++x) {
            const size_t i = (size_t)y * ox + x;
            inx[i] = outx[i] = xa[x];
            iny[i] = outy[i] = ya[y];
        }
    int rc = ORC_ERROR;
    if (pj_transform(po, pi, (long)on, 0, inx, iny, z) == 0) {
        double dx, dy;
        orc_pick_deltas(inx, ox, oy, &dx, &dy);
        rc = orc_matrix_from_deltas(pi, po, inx, iny, outx, outy, dx, dy, (long)on, matrix);
    }
    pj_free(pi);
    pj_free(po);
    free(xa);
    free(buf);
    free(z);
    return rc;
}

/* mifi_get_vector_reproject_matrix_field :667-717 */
int orc_vector_matrix_field(const char* proj_in, const char* proj_out, const double* in_x_field, const double* in_y_field, int ox, int oy,
                            double* matrix)
{
    projPJ pi, po;
    if (orc_open_pair(proj_in, proj_out, &pi, &po) != ORC_OK)
        return ORC_ERROR;
    const size_t on = (size_t)ox * oy;
    double* ox_f = (double*)malloc(sizeof(double) * on * 2);
    double* oy_f = ox_f + on;
    double* z = (double*)calloc(on, sizeof(double));
    memcpy(ox_f, in_x_field, sizeof(double) * on);
    memcpy(oy_f, in_y_field, sizeof(double) * on);
    int rc = ORC_ERROR;
    if (pj_transform(pi, po, (long)on, 0, ox_f, oy_f, z) == 0) {
        double dx, dy;
        orc_pick_deltas(in_x_field, ox, oy, &dx, &dy);
        rc = orc_matrix_from_deltas(pi, po, in_x_field, in_y_field, ox_f, oy_f, dx, dy, (long)on, matrix);
    }
    pj_free(pi);
    pj_free(po);
    free(ox_f);
    free(z);
    return rc;
}

/* mifi_get_vector_reproject_matrix_points :607-665.  As in the reference the projections are not
 * released (:660-664 frees the arrays only). */
int orc_vector_matrix_points(const char* proj_in, const char* proj_out, int input_is_metric, const double* out_x, const double* out_y, int on,
                             double* matrix)
{
    projPJ pi, po;
    if (orc_open_pair(proj_in, proj_out, &pi, &po) != ORC_OK)
        return ORC_ERROR;
    double* inx = (double*)malloc(sizeof(double) * (size_t)on * 2);
    double* iny = inx + on;
    double* z = (double*)calloc((size_t)on, sizeof(double));
    memcpy(inx, out_x, sizeof(double) * (size_t)on);
    memcpy(iny, out_y, sizeof(double) * (size_t)on);
    int rc = ORC_ERROR;
    if (pj_transform(po, pi, on, 0, inx, iny, z) == 0) {
        const double delta = input_is_metric ? 100 : 0.00001;
        rc = orc_matrix_from_deltas(pi, po, inx, iny, out_x, out_y, delta, delta, on, matrix);
    }
    pj_free(pi);
    pj_free(po);
    free(inx);
    free(z);
    return rc;
}

/* A14 mifi_vector_reproject_values_by_matrix_f :790-812 */
void orc_vector_reproject_by_matrix(const double* matrix, float* u, float* v, int ox, int oy, int oz)
{
    const size_t layer = (size_t)ox * oy;
    for (int z = 0; z < oz; ++z) {
        float* uz = u + (size_t)z * layer;
        float* vz = v + (size_t)z * layer;
        for (size_t i = 0; i < layer; ++i) {
            const double c = matrix[4 * i], s = matrix[4 * i + 1];
            const double un = uz[i] * c - vz[i] * s;
            const double vn = uz[i] * s + vz[i] * c;
            uz[i] = (float)un;
            vz[i] = (float)vn;
        }
    }
}

/* mifi_vector_reproject_direction_by_matrix_f :814-835 */
void orc_vector_reproject_direction(const double* matrix, float* angle, int ox, int oy, int oz)
{
    const size_t layer = (size_t)ox * oy;
    for (int z = 0; z < oz; ++z)
        for (size_t i = 0; i < layer; ++i) {
            float* a = angle + (size_t)z * layer + i;
            double an = *a - RAD_TO_DEG * matrix[4 * i + 3];
            if (an < 0)
                an += 360;
            if (an > 360)
                an -= 360;
            *a = (float)an;
        }
}

/* mifi_vector_reproject_values_f :837-859 */
int orc_vector_reproject_values(const char* proj_in, const char* proj_out, float* u, float* v, const double* out_x_axis,
                                const double* out_y_axis, int xt, int yt, int ox, int oy, int oz)
{
    double* m = (double*)malloc(sizeof(double) * 4 * (size_t)ox * oy);
    int rc = orc_vector_matrix(proj_in, proj_out, out_x_axis, out_y_axis, xt, yt, ox, oy, m);
    if (rc == ORC_OK)
        orc_vector_reproject_by_matrix(m, u, v, ox, oy, oz);
    free(m);
    return rc;
}

/* ------------------------------------------------------------------------------------------------
 * A4/A5  CachedInterpolation, src/CachedInterpolation.cc:118-147 (loop) and :149-200 (crop)
 * ---------------------------------------------------------------------------------------------- */
static long long orc_clamp_ll(long long lo, double dv, long long hi)
{
    const long long v = (long long)dv; /* :151-158 */
    if (v < lo)
        return lo;
    if (v < hi)
        return v;
    return hi;
}

/* returns 1 and updates px/py/inX/inY/minX/minY when the domain was reduced, 0 when left alone */
int orc_reduced_domain(double* px, double* py, size_t n, size_t* inX, size_t* inY, long long* minX_out, long long* minY_out)
{
    if (n == 0)
        return 0;
    double lox = px[0], hix = px[0], loy = py[0], hiy = py[0];
    for (size_t i = 1; i < n; ++i) { /* std::min_element / max_element semantics with operator< */
        if (px[i] < lox)
            lox = px[i];
        if (hix < px[i])
            hix = px[i];
        if (py[i] < loy)
            loy = py[i];
        if (hiy < py[i])
            hiy = py[i];
    }
    const long long EXT = 2;
    const long long x0 = orc_clamp_ll(0, floor(lox) - EXT, (long long)*inX - 1);
    const long long y0 = orc_clamp_ll(0, floor(loy) - EXT, (long long)*inY - 1);
    const long long x1 = orc_clamp_ll(0, ceil(hix) + EXT, (long long)*inX - 1);
    const long long y1 = orc_clamp_ll(0, ceil(hiy) + EXT, (long long)*inY - 1);
    if ((x1 - x0) < 1 || (y1 - y0) < 1)
        return 0;
    for (size_t i = 0; i < n; ++i) {
        px[i] -= x0;
        py[i] -= y0;
    }
    *minX_out = x0;
    *minY_out = y0;
    *inX = (size_t)(x1 - x0 + 1);
    *inY = (size_t)(y1 - y0 + 1);
    return 1;
}

/* interpolateValues :118-147: OpenMP over target points, per-thread column buffer, z-strided scatter.
 * `method` selects the function pointer as the constructor does (:104-114). */
int orc_cached_interpolate(int method, const double* px, const double* py, size_t inX, size_t inY, size_t outX, size_t outY,
                           const float* in, size_t size, float* out, int nthreads)
{
    void (*fn)(const float*, float*, double, double, int, int, int);
    switch (method) {
    case ORC_BILINEAR:
        fn = orc_get_values_bilinear;
        break;
    case ORC_BICUBIC:
        fn = orc_get_values_bicubic;
        break;
    case ORC_NN:
    case ORC_COORD_NN:
    case ORC_COORD_NN_KD:
        fn = orc_get_values_nn;
        break;
    default:
        return ORC_ERROR;
    }
    const size_t layer = outX * outY;
    const size_t inZ = size / (inX * inY);
#ifdef _OPENMP
    if (nthreads <= 0)
        nthreads = omp_get_max_threads();
#pragma omp parallel num_threads(nthreads)
#endif
    {
        float* col = (float*)malloc(sizeof(float) * (inZ ? inZ : 1));
#ifdef _OPENMP
#pragma omp for
#endif
        for (long long xy = 0; xy < (long long)layer; ++xy) {
            fn(in, col, px[xy], py[xy], (int)inX, (int)inY, (int)inZ);
            float* o = out + xy;
            for (size_t z = 0; z < inZ; ++z, o += layer)
                *o = col[z];
        }
        free(col);
    }
    (void)nthreads;
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------------
 * A16/A17  CachedForwardInterpolation, src/CachedForwardInterpolation.cc:38-59, 62-90, 92-131 and
 * RoundAndClamp, src/Utils.cc:42-58
 * ---------------------------------------------------------------------------------------------- */
void orc_round_and_clamp(const double* pos, size_t n, int maxi, int* idx)
{
    for (size_t i = 0; i < n; ++i) {
        const double r = round(pos[i]);
        /* the reference converts round(d) to int implicitly; out-of-int-range / NaN is UB there and
         * yields INT_MIN on x86-64, i.e. "invalid" */
        int v = (r >= -2147483648.0 && r <= 2147483647.0) ? (int)r : INT32_MIN;
        idx[i] = (v >= 0 && v <= maxi) ? v : -1;
    }
}

/* std::nth_element(first, nth, last) on floats with operator<, restated from libstdc++'s bits/stl_algo.h (__introselect,
 * __unguarded_partition_pivot, __move_median_to_first, __insertion_sort, __heap_select) and bits/stl_heap.h (__make_heap,
 * __adjust_heap, __push_heap, __pop_heap).  The C++ standard leaves the result undefined when the range holds NaN (< is then
 * no strict weak order) and does not say which of several equal elements lands at nth (+0 == -0); this restatement makes
 * the same comparisons and moves in the same order as that library, so it picks the same element bit for bit. */
static void orc_swapf(float* a, float* b)
{
    const float t = *a;
    *a = *b;
    *b = t;
}

static void orc_push_heap(float* v, ptrdiff_t hole, ptrdiff_t top, float value)
{
    ptrdiff_t parent = (hole - 1) / 2;
    while (hole > top && v[parent] < value) {
        v[hole] = v[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    v[hole] = value;
}

static void orc_adjust_heap(float* v, ptrdiff_t hole, ptrdiff_t len, float value)
{
    const ptrdiff_t top = hole;
    ptrdiff_t child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (v[child] < v[child - 1])
            child--;
        v[hole] = v[child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        v[hole] = v[child - 1];
        hole = child - 1;
    }
    orc_push_heap(v, hole, top, value);
}

static void orc_heap_select(float* first, float* middle, float* last)
{
    const ptrdiff_t len = middle - first;
    if (len >= 2) { /* __make_heap */
        for (ptrdiff_t parent = (len - 2) / 2;; parent--) {
            orc_adjust_heap(first, parent, len, first[parent]);
            if (parent == 0)
                break;
        }
    }
    for (float* i = middle; i < last; ++i)
        if (*i < *first) { /* __pop_heap(first, middle, i) */
            const float value = *i;
            *i = *first;
            orc_adjust_heap(first, 0, len, value);
        }
}

static void orc_insertion_sort(float* first, float* last)
{
    if (first == last)
        return;
    for (float* i = first + 1; i != last; ++i) {
        const float val = *i;
        if (val < *first) {
            memmove(first + 1, first, sizeof(float) * (size_t)(i - first));
            *first = val;
        } else { /* __unguarded_linear_insert */
            float* hole = i;
            float* next = i - 1;
            while (val < *next) {
                *hole = *next;
                hole = next;
                --next;
            }
            *hole = val;
        }
    }
}

static void orc_move_median_to_first(float* result, float* a, float* b, float* c)
{
    if (*a < *b) {
        if (*b < *c)
            orc_swapf(result, b);
        else if (*a < *c)
            orc_swapf(result, c);
        else
            orc_swapf(result, a);
    } else if (*a < *c)
        orc_swapf(result, a);
    else if (*b < *c)
        orc_swapf(result, c);
    else
        orc_swapf(result, b);
}

static float* orc_unguarded_partition_pivot(float* first, float* last)
{
    float* mid = first + (last - first) / 2;
    orc_move_median_to_first(first, first + 1, mid, last - 1);
    float* lo = first + 1;
    float* hi = last;
    const float* pivot = first;
    for (;;) {
        while (*lo < *pivot)
            ++lo;
        --hi;
        while (*pivot < *hi)
            --hi;
        if (!(lo < hi))
            return lo;
        orc_swapf(lo, hi);
        ++lo;
    }
}

void orc_nth_element(float* first, size_t nth_index, size_t n)
{
    float* last = first + n;
    float* nth = first + nth_index;
    if (first == last || nth == last)
        return;
    int depth_limit = 0; /* std::__lg(n) * 2 */
    for (size_t m = n; m > 1; m >>= 1)
        depth_limit += 2;
    while (last - first > 3) {
        if (depth_limit == 0) {
            orc_heap_select(first, nth + 1, last);
            orc_swapf(first, nth);
            return;
        }
        --depth_limit;
        float* cut = orc_unguarded_partition_pivot(first, last);
        if (cut <= nth)
            first = cut;
        else
            last = cut;
    }
    orc_insertion_sort(first, last);
}

static float orc_aggregate(int method, float* v, size_t n)
{
    switch (method) {
    case ORC_FWD_SUM:
    case ORC_FWD_UNDEF_SUM:
    case ORC_FWD_MEAN:
    case ORC_FWD_UNDEF_MEAN: {
        float s = 0.f; /* std::accumulate(..., 0.f): sequential fp32 sum in input order (:38-48) */
        for (size_t i = 0; i < n; ++i)
            s = s + v[i];
        if (method == ORC_FWD_MEAN || method == ORC_FWD_UNDEF_MEAN)
            s = s / n; /* float / size_t -> the count is converted to float */
        return s;
    }
    case ORC_FWD_MEDIAN:
    case ORC_FWD_UNDEF_MEDIAN:
        orc_nth_element(v, n / 2, n); /* nth_element(v.begin(), v.begin() + n/2, v.end()); v[n/2] (:49-53) */
        return v[n / 2];
    case ORC_FWD_MAX:
    case ORC_FWD_UNDEF_MAX: {
        size_t best = 0; /* std::max_element: first largest under operator< (:54-56) */
        for (size_t i = 1; i < n; ++i)
            if (v[best] < v[i])
                best = i;
        return v[best];
    }
    default: { /* MIN */
        size_t best = 0;
        for (size_t i = 1; i < n; ++i)
            if (v[i] < v[best])
                best = i;
        return v[best];
    }
    }
}

int orc_forward_interpolate(int method, const int* xi, const int* yi, size_t inX, size_t inY, size_t outX, size_t outY, const float* in,
                            size_t size, float* out)
{
    if (method < ORC_FWD_SUM || method > ORC_FWD_UNDEF_MIN)
        return ORC_ERROR;
    const int undef = method >= ORC_FWD_UNDEF_SUM;
    const size_t nin = inX * inY, layer = outX * outY, inZ = size / nin;
    size_t* start = (size_t*)malloc(sizeof(size_t) * (layer + 1));
    size_t* fill = (size_t*)malloc(sizeof(size_t) * (layer ? layer : 1));
    float* bucket = (float*)malloc(sizeof(float) * (nin ? nin : 1));
    for (size_t z = 0; z < inZ; ++z) {
        const float* lv = in + z * nin;
        /* bucket the level's values per target cell, preserving input (row-major) order (:99-115) */
        memset(start, 0, sizeof(size_t) * (layer + 1));
        for (size_t i = 0; i < nin; ++i)
            if ((undef || !isnan(lv[i])) && xi[i] >= 0 && yi[i] >= 0)
                start[(size_t)yi[i] * outX + xi[i] + 1]++;
        for (size_t c = 0; c < layer; ++c)
            start[c + 1] += start[c];
        memcpy(fill, start, sizeof(size_t) * layer);
        for (size_t i = 0; i < nin; ++i)
            if ((undef || !isnan(lv[i])) && xi[i] >= 0 && yi[i] >= 0)
                bucket[fill[(size_t)yi[i] * outX + xi[i]]++] = lv[i];
        float* o = out + z * layer;
        for (size_t c = 0; c < layer; ++c) { /* :118-128 */
            const size_t cnt = start[c + 1] - start[c];
            o[c] = cnt ? orc_aggregate(method, bucket + start[c], cnt) : orc_undef_f();
        }
    }
    free(start);
    free(fill);
    free(bucket);
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------------
 * A2  bad<->NaN adapters: mifi_bad2nanf src/interpolation.c:1775-1783; ScaleValue<float,OUT> with
 * scale 1 / offset 0, include/fimex/Utils.h:444-464 (NaN -> fill; integers round, floats cast)
 * ---------------------------------------------------------------------------------------------- */
size_t orc_bad2nan(float* p, size_t n, float bad)
{
    if (isnan(bad))
        return 0;
    const float nanv = orc_undef_f();
    for (size_t i = 0; i < n; ++i)
        if (p[i] == bad)
            p[i] = nanv;
    return 0;
}

/* data2InterpolationArray, src/CDMInterpolator.cc:115-119: Data::asFloat() is a static_cast per element
 * (src/DataImpl.h:385-389, include/fimex/Utils.h:88-113: no rounding towards a floating-point type), then
 * mifi_bad2nanf with the fill value narrowed to float (src/interpolation.c:1775-1783). */
#define ORC_AS_FLOAT(NAME, T)                                                                                  \
    void orc_as_float_##NAME(const T* in, size_t n, double bad, float* out)                                    \
    {                                                                                                          \
        const float b = (float)bad;                                                                            \
        const float nanv = orc_undef_f();                                                                      \
        for (size_t i = 0; i < n; ++i) {                                                                       \
            const float f = (float)in[i];                                                                      \
            out[i] = (!isnan(b) && f == b) ? nanv : f;                                                         \
        }                                                                                                      \
    }
ORC_AS_FLOAT(i8, signed char)
ORC_AS_FLOAT(i16, short)
ORC_AS_FLOAT(i32, int)
ORC_AS_FLOAT(f32, float)
ORC_AS_FLOAT(f64, double)
ORC_AS_FLOAT(u8, unsigned char)
ORC_AS_FLOAT(u16, unsigned short)
ORC_AS_FLOAT(u32, unsigned int)
ORC_AS_FLOAT(i64, long long)
ORC_AS_FLOAT(u64, unsigned long long)

/* interpolationArray2Data, src/CDMInterpolator.cc:121-124: convertDataType(MIFI_UNDEFINED_F, 1., 0., type, badValue, 1., 0.)
 * = ScaleValue<float, OUT> (include/fimex/Utils.h:444-464): NaN -> static_cast<OUT>(badValue); otherwise
 * data_caster<OUT, double>(1. * in + 0.), which rounds through MetNoFimex::round(double) -> int (::lround narrowed to int,
 * Utils.h:72-75, 98-99) for integer OUT and is a plain static_cast for float / double. */
#define ORC_FROM_FLOAT_INT(NAME, T)                                                                            \
    void orc_from_float_##NAME(const float* in, size_t n, double fill, T* out)                                 \
    {                                                                                                          \
        for (size_t i = 0; i < n; ++i)                                                                         \
            out[i] = isnan(in[i]) ? (T)fill : (T)(int)lround(1. * in[i] + 0.);                                 \
    }
#define ORC_FROM_FLOAT_FP(NAME, T)                                                                             \
    void orc_from_float_##NAME(const float* in, size_t n, double fill, T* out)                                 \
    {                                                                                                          \
        for (size_t i = 0; i < n; ++i)                                                                         \
            out[i] = isnan(in[i]) ? (T)fill : (T)(1. * in[i] + 0.);                                            \
    }
ORC_FROM_FLOAT_INT(i8, signed char)
ORC_FROM_FLOAT_INT(i16, short)
ORC_FROM_FLOAT_INT(i32, int)
ORC_FROM_FLOAT_FP(f32, float)
ORC_FROM_FLOAT_FP(f64, double)
ORC_FROM_FLOAT_INT(u8, unsigned char)
ORC_FROM_FLOAT_INT(u16, unsigned short)
ORC_FROM_FLOAT_INT(u32, unsigned int)
ORC_FROM_FLOAT_INT(i64, long long)
ORC_FROM_FLOAT_INT(u64, unsigned long long)

/* ------------------------------------------------------------------------------------------------
 * 8f rank 3: the 2-D pre/post-processes.  mifi_fill2d_f (src/interpolation.c:1246-1376): undefined cells get the mean of the
 * defined ones, then lexicographic Gauss-Seidel relaxation of the Laplace equation on those cells (weight 1 on undefined
 * cells, times corrEff in the interior), a convergence test every 10th sweep, one-sided relaxation of the border after each
 * sweep.  mifi_creepfill(val)2d_f (:1378-1525): undefined cells creep in from defined neighbours, `repeat` times per cell.
 * Restated sweep by sweep; pinned bit for bit against the compiled reference (tests/test_oracle_golden.py).
 * ---------------------------------------------------------------------------------------------- */
int orc_fill2d(size_t nx, size_t ny, float* field, float relaxCrit, float corrEff, size_t maxLoop, size_t* nChanged)
{
    const size_t n = nx * ny;
    if (n == 0)
        return ORC_OK;
    double sum = 0;
    size_t nundef = 0;
    for (size_t i = 0; i < n; ++i) {
        if (isnan(field[i]))
            ++nundef;
        else
            sum += field[i];
    }
    *nChanged = nundef;
    const size_t ndef = n - nundef;
    if (ndef == 0 || nundef == 0)
        return ORC_OK;
    float* w = (float*)malloc(n * sizeof(float));
    const double average = sum / ndef;
    double dev = 0;
    for (size_t i = 0; i < n; ++i) {
        if (isnan(field[i])) {
            w[i] = 1.f;
            field[i] = average;
        } else {
            dev += fabs(field[i] - average);
            w[i] = 0.f;
        }
    }
    dev /= ndef;
    const double crit = relaxCrit * dev;
    const size_t xl = nx - 1, yl = ny - 1; /* last column / row */
    for (size_t y = 1; y < yl; ++y)
        for (size_t x = 1; x < xl; ++x)
            w[y * nx + x] *= corrEff;
    for (size_t loop = 0; loop < maxLoop; ++loop) {
        int bad = 0;
        const int test = (loop < (maxLoop - 5)) && (loop % 10 == 0);
        const float crtest = crit * corrEff;
        for (size_t y = 1; y < yl; ++y) {
            for (size_t x = 1; x < xl; ++x) {
                float* f = field + y * nx + x;
                const float e = (f[1] + f[-1] + f[nx] + f[-(long)nx]) * 0.25 - *f;
                const float ew = e * w[y * nx + x];
                *f += ew;
                if (test && fabs(ew) > crtest)
                    bad = 1;
            }
        }
        if (test && !bad)
            break;
        for (size_t y = 1; y < yl; ++y) {
            float* r = field + y * nx;
            r[0] += (r[1] - r[0]) * w[y * nx];
            r[xl] += (r[xl - 1] - r[xl]) * w[y * nx + xl];
        }
        for (size_t x = 0; x < nx; ++x) {
            field[x] += (field[nx + x] - field[x]) * w[x];
            field[yl * nx + x] += (field[(yl - 1) * nx + x] - field[yl * nx + x]) * w[yl * nx + x];
        }
    }
    free(w);
    return ORC_OK;
}

/* use_mean != 0: mifi_creepfill2d_f (first guess = float mean of the defined values); else mifi_creepfillval2d_f */
int orc_creepfill2d(size_t nx, size_t ny, float* field, int use_mean, float defaultVal, unsigned short repeat, char setWeight,
                    size_t* nChanged)
{
    const size_t n = nx * ny;
    if (n == 0)
        return ORC_OK;
    double sum = 0;
    size_t nundef = 0;
    for (size_t i = 0; i < n; ++i) {
        if (isnan(field[i]))
            ++nundef;
        else
            sum += field[i];
    }
    *nChanged = nundef;
    const size_t ndef = n - nundef;
    if (ndef == 0 || nundef == 0)
        return ORC_OK;
    float guess = defaultVal;
    if (use_mean)
        guess = sum / ndef;
    char* w = (char*)malloc(n);
    unsigned short* r = (unsigned short*)malloc(n * sizeof(unsigned short));
    for (size_t i = 0; i < n; ++i) {
        if (isnan(field[i])) {
            w[i] = 0;
            r[i] = 0;
            field[i] = guess;
        } else {
            w[i] = setWeight;
            r[i] = repeat;
        }
    }
    const size_t xl = nx - 1, yl = ny - 1;
    size_t changed = 1, loops = 0;
    while (changed > 0 && loops < ndef) {
        changed = 0;
        ++loops;
        for (size_t y = 1; y < yl; ++y) {
            for (size_t x = 1; x < xl; ++x) {
                const size_t p = y * nx + x;
                if (r[p] >= repeat)
                    continue;
                const size_t wsum = w[p + 1] + w[p - 1] + w[p + nx] + w[p - nx];
                if (wsum == 0)
                    continue;
                field[p] += w[p + 1] * field[p + 1] + w[p - 1] * field[p - 1] + w[p + nx] * field[p + nx] + w[p - nx] * field[p - nx];
                field[p] /= (1 + wsum);
                w[p] = 1;
                r[p]++;
                ++changed;
            }
        }
    }
    for (size_t k = 0; k < repeat; ++k) {
        for (size_t y = 1; y < yl; ++y) {
            const size_t a = y * nx, b = y * nx + xl;
            if (r[a] < repeat) {
                field[a] += field[a + 1] * w[a + 1];
                field[a] /= (1 + w[a + 1]);
                w[a] = 1;
            }
            if (r[b] < repeat) {
                field[b] += field[b - 1] * w[b - 1];
                field[b] /= (1 + w[b - 1]);
                w[b] = 1;
            }
        }
        for (size_t x = 0; x < nx; ++x) {
            const size_t a = x, b = yl * nx + x;
            if (r[a] < repeat) {
                field[a] += field[a + nx] * w[a + nx];
                field[a] /= (1 + w[a + nx]);
                w[a] = 1;
            }
            if (r[b] < repeat) {
                field[b] += field[b - nx] * w[b - nx];
                field[b] /= (1 + w[b - nx]);
                w[b] = 1;
            }
        }
    }
    free(r);
    free(w);
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------------
 * A18  coord_nearestneighbor search, src/CDMInterpolator.cc:1064-1125 (getGridDistance) and
 * :1141-1220 (fastTranslatePointsToClosestInputCell).  The reference sorts with std::sort (unstable);
 * the order among equal latitudes is libstdc++-specific and only matters for exact cos_d ties.  Here a
 * stable sort on (lat, insertion order) is used and ties are reported by orc_coordnn's return value.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    double lat, lon, x, y;
    double coslat, sinlat;
    size_t seq;
} orc_llpt;

static int orc_cmp_llpt(const void* a, const void* b)
{
    const orc_llpt *p = (const orc_llpt*)a, *q = (const orc_llpt*)b;
    if (p->lat < q->lat)
        return -1;
    if (q->lat < p->lat)
        return 1;
    return (p->seq > q->seq) - (p->seq < q->seq);
}

double orc_grid_distance(const double* lon, const double* lat, size_t nx, size_t ny)
{
    /* :1064-1125 */
    int steps;
    size_t step;
    if (nx * ny > 1000) {
        steps = 53;
        step = nx * ny / steps;
    } else {
        step = 1;
        steps = (int)(nx * ny);
    }
    double worst = 2; /* min over samples of their max cos_d */
    int have = 0;
    for (int k = 0; k < steps; ++k) {
        const size_t sp = (size_t)k * step;
        const double lon0 = lon[sp], lat0 = lat[sp];
        if (isnan(lon0) || isnan(lat0))
            continue;
        double best = -2;
        for (size_t ix = 0; ix < nx; ++ix)
            for (size_t iy = 0; iy < ny; ++iy) {
                const size_t pos = ix + iy * nx;
                if (pos == sp || isnan(lon[pos]) || isnan(lat[pos]))
                    continue;
                const double dlon = lon0 - lon[pos];
                const double cd = cos(lat0) * cos(lat[pos]) * cos(dlon) + sin(lat0) * sin(lat[pos]);
                if (cd > best)
                    best = cd;
            }
        if (!have || best < worst)
            worst = best;
        have = 1;
    }
    double d = acos(worst);
    d *= 1.414;
    if (d > ORC_PI)
        d = ORC_PI;
    return d;
}

/* px = target longitudes, py = target latitudes (radians), overwritten with source (ix, iy) or (-1,-1).
 * Returns the number of targets whose winner had an exact cos_d tie with another candidate. */
long orc_coordnn(double* px, double* py, size_t n, const double* lon, const double* lat, size_t nx, size_t ny)
{
    const double roi = orc_grid_distance(lon, lat, nx, ny);
    const double min_grid_cos = cos(roi);
    orc_llpt* pts = (orc_llpt*)malloc(sizeof(orc_llpt) * ((nx * ny) > 0 ? nx * ny : 1));
    size_t m = 0;
    for (size_t ix = 0; ix < nx; ++ix)
        for (size_t iy = 0; iy < ny; ++iy) {
            const size_t pos = ix + iy * nx;
            if (isnan(lon[pos]) || isnan(lat[pos]))
                continue;
            pts[m].lat = lat[pos];
            pts[m].lon = lon[pos];
            pts[m].x = (double)ix;
            pts[m].y = (double)iy;
            pts[m].seq = m;
            ++m;
        }
    qsort(pts, m, sizeof(orc_llpt), orc_cmp_llpt);
    long ties = 0;
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : ties) schedule(dynamic, 1024)
#endif
    for (long long i = 0; i < (long long)n; ++i) {
        const double plat = py[i], plon = px[i];
        double rx = -1., ry = -1.;
        double best = min_grid_cos;
        double min_d = acos(best);
        int tie = 0;
        /* lower_bound on latitude */
        size_t lo = 0, hi = m;
        while (lo < hi) {
            const size_t mid = lo + (hi - lo) / 2;
            if (pts[mid].lat < plat)
                lo = mid + 1;
            else
                hi = mid;
        }
        for (size_t k = lo; k < m; ++k) { /* upwards (:1173-1189) */
            if (fabs(pts[k].lat - plat) > min_d)
                break;
            const double dlon = pts[k].lon - plon;
            const double cd = cos(pts[k].lat) * cos(plat) * cos(dlon) + sin(pts[k].lat) * sin(plat);
            if (cd > best) {
                best = cd;
                min_d = acos(best);
                rx = pts[k].x;
                ry = pts[k].y;
                tie = 0;
            } else if (cd == best && rx >= 0) {
                tie = 1;
            }
        }
        for (size_t k = lo; k-- > 0;) { /* downwards (:1191-1209) */
            if (fabs(pts[k].lat - plat) > min_d)
                break;
            const double dlon = pts[k].lon - plon;
            const double cd = cos(pts[k].lat) * cos(plat) * cos(dlon) + sin(pts[k].lat) * sin(plat);
            if (cd > best) {
                best = cd;
                min_d = acos(best);
                rx = pts[k].x;
                ry = pts[k].y;
                tie = 0;
            } else if (cd == best && rx >= 0) {
                tie = 1;
            }
        }
        py[i] = ry;
        px[i] = rx;
        ties += tie;
    }
    free(pts);
    return ties;
}

/* lonLatVals2Matrix :1226-1239 */
/* coord_kdtree: flannTranslatePointsToClosestInputCell, src/CDMInterpolator.cc:991-1062.  nanoflann (vendored in the reference,
 * include/nanoflann/nanoflann.hpp) only prunes the search: radiusSearch(sorted) returns the matches with
 * dist < radius (RadiusResultSet::addPoint, :150-153) ordered by distance, and the reference takes the first, i.e. the exact
 * nearest neighbour by PointCloud::kdtree_distance = d0*d0 + d1*d1 + d2*d2 (CDMInterpolator.cc:967-973).  Brute force here.
 * Equal distances are ordered by std::sort (unspecified); the lowest source position wins here and the count is returned.
 * Pinned against the reference's nanoflann itself (oracle/ref_kd_driver.cc, tests/test_oracle_golden.py).  Declared deviation:
 * source points with NaN coordinates are skipped; in the reference they enter the tree as NaN points and corrupt its
 * bounding boxes (many targets then lose their match). */
long orc_coordkd(double* px, double* py, size_t n, const double* lon, const double* lat, size_t nx, size_t ny, double max_dist_m)
{
    const size_t ns = nx * ny;
    double* c = (double*)malloc(sizeof(double) * 3 * ns);
    for (size_t ix = 0; ix < nx; ++ix) {
        for (size_t iy = 0; iy < ny; ++iy) {
            const size_t pos = ix + iy * nx;
            if (!(isnan(lat[pos]) || isnan(lon[pos]))) {
                const double sinLat = sin(lat[pos]), cosLat = cos(lat[pos]), sinLon = sin(lon[pos]), cosLon = cos(lon[pos]);
                c[3 * pos] = cosLat * cosLon;
                c[3 * pos + 1] = cosLat * sinLon;
                c[3 * pos + 2] = sinLat;
            } else {
                c[3 * pos] = c[3 * pos + 1] = c[3 * pos + 2] = NAN;
            }
        }
    }
    double maxDist = max_dist_m / 6371000.;
    const double search_radius = maxDist * maxDist;
    long ties = 0;
#pragma omp parallel for reduction(+ : ties)
    for (size_t i = 0; i < n; ++i) {
        const double sinLat = sin(py[i]), cosLat = cos(py[i]), sinLon = sin(px[i]), cosLon = cos(px[i]);
        const double q[3] = {cosLat * cosLon, cosLat * sinLon, sinLat};
        double best = search_radius;
        long bestpos = -1;
        int tie = 0;
        for (size_t p = 0; p < ns; ++p) {
            const double d0 = q[0] - c[3 * p], d1 = q[1] - c[3 * p + 1], d2 = q[2] - c[3 * p + 2];
            const double dist = d0 * d0 + d1 * d1 + d2 * d2;
            if (dist < best) {
                best = dist;
                bestpos = (long)p;
                tie = 0;
            } else if (dist == best && bestpos >= 0) {
                tie = 1;
            }
        }
        if (bestpos >= 0) {
            px[i] = (double)(bestpos % (long)nx);
            py[i] = (double)(bestpos / (long)nx);
        } else {
            px[i] = -1000;
            py[i] = -1000;
        }
        ties += tie;
    }
    free(c);
    return ties;
}

/* getMaxDistanceOfInterest, src/CDMInterpolator.cc:304-326 (axis values as given, times the earth radius unless metric) */
double orc_max_distance_of_interest(const double* xa, size_t nx, const double* ya, size_t ny, int is_metric)
{
    const double factor = is_metric ? 1. : 6371000.;
    double maxX = 0, maxY = 0;
    for (size_t i = 0; i + 1 < nx; ++i)
        maxX = fmax(factor * fabs(xa[i + 1] - xa[i]), maxX);
    for (size_t j = 0; j + 1 < ny; ++j)
        maxY = fmax(factor * fabs(ya[j + 1] - ya[j]), maxY);
    return fmax(maxX, maxY);
}

void orc_lonlat_to_matrix(const double* lonv, const double* latv, size_t nlon, size_t nlat, double* lon2d, double* lat2d)
{
    for (size_t ix = 0; ix < nlon; ++ix)
        for (size_t iy = 0; iy < nlat; ++iy) {
            lon2d[ix + iy * nlon] = lonv[ix];
            lat2d[ix + iy * nlon] = latv[iy];
        }
}
