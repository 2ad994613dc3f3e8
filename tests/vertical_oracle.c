/*
 * tests/vertical_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement (plain C99) of vertical interpolation to pressure
 * levels, the pressure branch of the reference's CDMVerticalInterpolator, written out as DESIGN.md section 2 states it (the
 * reference's C++ side is not compiled here; the per-column step follows mifi_get_values_linear_f / _log_f / _log_log_f,
 * src/interpolation.c:1030-1156).  Only tests/ and profiles/tools/vertical_time.py load the library built from this file
 * (tests/vertical_oracle.py compiles it on demand); libfimex_b200.so never links, loads or calls it.
 *
 * Build: gcc -std=gnu99 -O2 -ffp-contract=off -fPIC -fopenmp (no FMA contraction), as oracle/liboracle.so.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_OK 1
#define ORC_ERROR (-1)

static float orc_undef_f(void)
{
    return nanf(""); /* MIFI_UNDEFINED_F, mifi_constants.h:254: canonical quiet NaN 0x7fc00000 */
}

enum { ORC_VINT_LIN = 0, ORC_VINT_LOG = 1, ORC_VINT_LOGLOG = 2, ORC_VINT_NN = 3 }; /* MIFI_VINT_METHOD_* */
enum { ORC_VCOORD_PRESSURE = 0, ORC_VCOORD_HYBRID = 1, ORC_VCOORD_SIGMA = 2 };

/* ln(x): fdlibm 5.3 __ieee754_log (e_log.c), four arithmetic operations only, so that the library's kernel
 * (vertical_kernels.cu, vlog) rounds every step identically */
double orc_vlog(double x)
{
    static const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, two54 = 1.80143985094819840000e+16;
    static const double Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                        Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                        Lg7 = 1.479819860511658591e-01;
    double hfsq, f, s, z, R, w, t1, t2, dk;
    int k, hx, i, j;
    uint32_t lx;
    uint64_t bits;
    memcpy(&bits, &x, 8);
    hx = (int)(uint32_t)(bits >> 32);
    lx = (uint32_t)bits;
    k = 0;
    if (hx < 0x00100000) {
        if (((hx & 0x7fffffff) | lx) == 0)
            return -INFINITY;
        if (hx < 0)
            return NAN;
        k -= 54;
        x *= two54;
        memcpy(&bits, &x, 8);
        hx = (int)(uint32_t)(bits >> 32);
    }
    if (hx >= 0x7ff00000)
        return x + x;
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    i = (hx + 0x95f64) & 0x100000;
    memcpy(&bits, &x, 8);
    bits = ((uint64_t)(uint32_t)(hx | (i ^ 0x3ff00000)) << 32) | (bits & 0xffffffffu);
    memcpy(&x, &bits, 8);
    k += (i >> 20);
    f = x - 1.0;
    dk = (double)k;
    if ((0x000fffff & (2 + hx)) < 3) {
        if (f == 0.0)
            return k == 0 ? 0.0 : dk * ln2_hi + dk * ln2_lo;
        R = f * f * (0.5 - 0.33333333333333333 * f);
        return k == 0 ? f - R : dk * ln2_hi - ((R - dk * ln2_lo) - f);
    }
    s = f / (2.0 + f);
    z = s * s;
    i = hx - 0x6147a;
    w = z * z;
    j = 0x6b851 - hx;
    t1 = w * (Lg2 + w * (Lg4 + w * Lg6));
    t2 = z * (Lg1 + w * (Lg3 + w * (Lg5 + w * Lg7)));
    i |= j;
    R = t2 + t1;
    if (i > 0) {
        hfsq = 0.5 * f * f;
        if (k == 0)
            return f - (hfsq - s * (hfsq + R));
        return dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f);
    }
    if (k == 0)
        return f - s * (f - R);
    return dk * ln2_hi - ((s * (f - R) - dk * ln2_lo) - f);
}

/* the coordinate the weights are linear in: p, ln p, ln ln p */
static double orc_vcoord(int method, double p)
{
    if (method == ORC_VINT_LOG)
        return orc_vlog(p);
    if (method == ORC_VINT_LOGLOG)
        return orc_vlog(orc_vlog(p));
    return p;
}

/* one value between the levels at pressures pa (value A) and pb (value B) for the target pressure x */
static float orc_vint_value(int method, float A, float B, double pa, double pb, double x)
{
    double xa, xb, w;
    if (method == ORC_VINT_NN)
        return fabs(x - pb) < fabs(x - pa) ? B : A; /* a tie takes the lower level */
    xa = orc_vcoord(method, pa);
    xb = orc_vcoord(method, pb);
    w = xa == xb ? 0.0 : (orc_vcoord(method, x) - xa) / (xb - xa);
    return (float)((double)A + w * ((double)B - (double)A));
}

/* the two-level step for n values, with the argument list of the reference's mifi_get_values_linear_f (a, b: pressures of the
 * levels of A and B, x: target pressure) */
void orc_vint_values(int method, const float* A, const float* B, float* out, size_t n, double a, double b, double x)
{
    size_t i;
    for (i = 0; i < n; ++i)
        out[i] = orc_vint_value(method, A[i], B[i], a, b, x);
}

/* in [nt][nk][nxy], ps [nt][nxy] (unused for pressure levels), out [nt][np][nxy] */
int orc_vinterp_pressure(int method, int kind, const double* ap, const double* b, int nk, double ptop, double ps_scale, const double* levels,
                         int np, int extrapolate, const float* in, const float* ps, long nxy, long nt, float* out)
{
    long long ncol = (long long)nxy * nt;
    if (nk < 2 || np < 1 || method < ORC_VINT_LIN || method > ORC_VINT_NN)
        return ORC_ERROR;
#pragma omp parallel
    {
        double* p = (double*)malloc(sizeof(double) * nk);
        long long col;
#pragma omp for schedule(static)
        for (col = 0; col < ncol; ++col) {
            const long long t = col / nxy, c = col % nxy;
            const float* v = in + t * nk * nxy + c;
            float* o = out + t * np * nxy + c;
            double psd = 0.0, lo, hi;
            int k, i, incr, flat;
            if (kind != ORC_VCOORD_PRESSURE)
                psd = (double)ps[t * nxy + c] * ps_scale;
            for (k = 0; k < nk; ++k) {
                if (kind == ORC_VCOORD_HYBRID)
                    p[k] = ap[k] + b[k] * psd;
                else if (kind == ORC_VCOORD_SIGMA)
                    p[k] = ptop + b[k] * (psd - ptop);
                else
                    p[k] = ap[k];
            }
            incr = p[0] < p[nk - 1];
            flat = !(p[0] < p[nk - 1]) && !(p[0] > p[nk - 1]);
            lo = incr ? p[0] : p[nk - 1];
            hi = incr ? p[nk - 1] : p[0];
            for (i = 0; i < np; ++i) {
                const double P = levels[i];
                float r = orc_undef_f();
                int kk = -1;
                if (!flat) {
                    if (P < lo || P > hi) {
                        if (extrapolate)
                            kk = ((P < lo) == incr) ? 0 : nk - 2; /* the end pair on that side */
                    } else {
                        for (k = 0; k < nk - 1; ++k) { /* the smallest k with P between p_k and p_k+1, endpoints included */
                            const double a = p[k] < p[k + 1] ? p[k] : p[k + 1], z = p[k] < p[k + 1] ? p[k + 1] : p[k];
                            if (a <= P && P <= z) {
                                kk = k;
                                break;
                            }
                        }
                    }
                }
                if (kk >= 0)
                    r = orc_vint_value(method, v[(long long)kk * nxy], v[(long long)(kk + 1) * nxy], p[kk], p[kk + 1], P);
                o[(long long)i * nxy] = r;
            }
        }
        free(p);
    }
    return ORC_OK;
}
