/*
 * tests/vertical_height_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement (plain C99) of vertical interpolation to height and
 * altitude levels, the height branch of the reference's CDMVerticalInterpolator, written out as DESIGN.md section 2 states it (the
 * reference's converters, ToVLevelConverter and the mifi_barometric_* helpers, are C++ and not compiled here).  It includes
 * tests/vertical_oracle.c so that ln() (orc_vlog) and the undefined value are the very code the pressure branch's restatement uses.  Only tests/ and profiles/tools/vertical_height_time.py load the library built from this file
 * (tests/vertical_height_oracle.py compiles it on demand); libfimex_b200.so never links, loads or calls it.
 *
 * Build: gcc -std=gnu99 -O2 -ffp-contract=off -fPIC -fopenmp (no FMA contraction), as tests/vertical_oracle.c.
 */
#include "vertical_oracle.c"


enum { ORC_VZ_STANDARD = 0, ORC_VZ_HYPSOMETRIC = 1, ORC_VZ_FIELD = 2 };
enum { ORC_VZ_ALTITUDE = 0, ORC_VZ_HEIGHT = 1 };

/* exp(x): fdlibm 5.3 __ieee754_exp (e_exp.c): reduction x = k ln2 + r, |r| <= ln2 / 2, and a degree-5 rational approximation;
 * < 1 ulp.  Four arithmetic operations and bit operations only, as orc_vlog, so that vexp (vertical_kernels.cu) rounds alike. */
double orc_vexp(double x)
{
    static const double halF[2] = {0.5, -0.5}, huge = 1.0e+300, twom1000 = 9.33263618503218878990e-302,
                        o_threshold = 7.09782712893383973096e+02, u_threshold = -7.45133219101941108420e+02,
                        ln2HI[2] = {6.93147180369123816490e-01, -6.93147180369123816490e-01},
                        ln2LO[2] = {1.90821492927058770002e-10, -1.90821492927058770002e-10}, invln2 = 1.44269504088896338700e+00,
                        P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03, P3 = 6.61375632143793436117e-05,
                        P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
    double y, hi = 0.0, lo = 0.0, c, t;
    int k = 0, xsb;
    uint32_t hx, lx;
    uint64_t bits;
    memcpy(&bits, &x, 8);
    hx = (uint32_t)(bits >> 32);
    lx = (uint32_t)bits;
    xsb = (int)((hx >> 31) & 1);
    hx &= 0x7fffffff;
    if (hx >= 0x40862E42) { /* |x| >= 709.78... */
        if (hx >= 0x7ff00000) {
            if (((hx & 0xfffff) | lx) != 0)
                return x + x;              /* NaN */
            return (xsb == 0) ? x : 0.0; /* exp(+-inf) = {inf, 0} */
        }
        if (x > o_threshold)
            return huge * huge;
        if (x < u_threshold)
            return twom1000 * twom1000;
    }
    if (hx > 0x3fd62e42) {     /* |x| > 0.5 ln2 */
        if (hx < 0x3FF0A2B2) { /* and |x| < 1.5 ln2 */
            hi = x - ln2HI[xsb];
            lo = ln2LO[xsb];
            k = 1 - xsb - xsb;
        } else {
            k = (int)(invln2 * x + halF[xsb]);
            t = k;
            hi = x - t * ln2HI[0]; /* t * ln2HI is exact here */
            lo = t * ln2LO[0];
        }
        x = hi - lo;
    } else if (hx < 0x3e300000) { /* |x| < 2^-28 */
        return 1.0 + x;
    }
    t = x * x;
    c = x - t * (P1 + t * (P2 + t * (P3 + t * (P4 + t * P5))));
    if (k == 0)
        return 1.0 - ((x * c) / (c - 2.0) - x);
    y = 1.0 - ((lo - (x * c) / (2.0 - c)) - hi);
    memcpy(&bits, &y, 8);
    if (k >= -1021) {
        bits += (uint64_t)(int64_t)k << 52; /* add k to y's exponent */
        memcpy(&y, &bits, 8);
        return y;
    }
    bits += (uint64_t)(int64_t)(k + 1000) << 52;
    memcpy(&y, &bits, 8);
    return y * twom1000;
}

/* The converter constants, formed once (the library forms them with the same expressions in fimex_b200/csrc/api.cu).  US Standard
 * Atmosphere 1976 / ICAO, seven geopotential layers: base altitude h_b [m], base temperature T_b [K], lapse rate L_b [K/m], the
 * published base pressures p_b [hPa]; R* [J/(mol K)], M (dry air) and M_w (water) [kg/mol], g0 [m/s2]. */
#define ORC_NLAYER 7
static const double orc_hb[ORC_NLAYER] = {0.0, 11000.0, 20000.0, 32000.0, 47000.0, 51000.0, 71000.0};
static const double orc_Tb[ORC_NLAYER] = {288.15, 216.65, 216.65, 228.65, 270.65, 270.65, 214.65};
static const double orc_Lb[ORC_NLAYER] = {-6.5e-3, 0.0, 1e-3, 2.8e-3, 0.0, -2.8e-3, -2e-3};
static const double orc_pb[ORC_NLAYER] = {1013.25, 226.3206, 54.74889, 8.680187, 1.109063, 0.6693887, 0.03956420};
static const double orc_R = 8.31432, orc_M = 0.0289644, orc_Mw = 0.01801528, orc_g0 = 9.80665;

static double orc_H(void) /* R* / (M g0) [m/K] */
{
    return orc_R / (orc_M * orc_g0);
}

/* standard-atmosphere altitude [m] of the pressure p [hPa] */
double orc_zstd(double p)
{
    int b = 0, l;
    for (l = 1; l < ORC_NLAYER; ++l) /* the last layer with p <= p_b */
        if (p <= orc_pb[l])
            b = l;
    if (orc_Lb[b] != 0.0) {
        const double e = -(orc_R * orc_Lb[b]) / (orc_g0 * orc_M), c = orc_Tb[b] / orc_Lb[b];
        return orc_hb[b] + c * (orc_vexp(e * orc_vlog(p / orc_pb[b])) - 1.0);
    }
    return orc_hb[b] + (orc_H() * orc_Tb[b]) * orc_vlog(orc_pb[b] / p);
}

/* The coordinate zc[k] of every level k of one column (altitude, or height above z_s for the height target) and the column's
 * direction: 1 when level 0 is the surface end, 0 when level nk - 1 is, -1 for equal or NaN ends (a NaN column).  psd: ps * ps_scale;
 * t, q, z: the column's values at stride `stride` (q, z may be NULL); zsd: zs * zs_scale (0 when not given). */
static int orc_height_column(int converter, int target, int kind, const double* ap, const double* b, int nk, double ptop, double psd,
                             double z_scale, const float* t, const float* q, const float* z, long long stride, double zsd, double* p,
                             double* zc)
{
    const double H = orc_H(), cq = orc_M / orc_Mw - 1.0;
    const double zsub = (target == ORC_VZ_HEIGHT && converter != ORC_VZ_HYPSOMETRIC) ? zsd : 0.0;
    int k, m, s0;
    for (k = 0; k < nk && converter != ORC_VZ_FIELD; ++k) {
        if (kind == ORC_VCOORD_HYBRID)
            p[k] = ap[k] + b[k] * psd;
        else if (kind == ORC_VCOORD_SIGMA)
            p[k] = ptop + b[k] * (psd - ptop);
        else
            p[k] = ap[k];
    }
    if (converter == ORC_VZ_FIELD) {
        for (k = 0; k < nk; ++k)
            zc[k] = z_scale * (double)z[(long long)k * stride];
        if (!(zc[0] < zc[nk - 1]) && !(zc[0] > zc[nk - 1]))
            return -1;
        s0 = zc[0] < zc[nk - 1]; /* the surface end has the smaller z */
    } else {
        if (!(p[0] < p[nk - 1]) && !(p[0] > p[nk - 1]))
            return -1;
        s0 = p[0] > p[nk - 1]; /* the surface end has the larger p */
    }
    if (converter == ORC_VZ_STANDARD)
        for (k = 0; k < nk; ++k)
            zc[k] = orc_zstd(p[k]);
    if (converter == ORC_VZ_HYPSOMETRIC) { /* integrate upward from the surface: the trapezoid rule in ln p on Tv */
        double zprev = 0.0, tvprev = 0.0, pprev = 0.0;
        for (m = 0; m < nk; ++m) {
            const int kk = s0 ? m : nk - 1 - m;
            const double T = (double)t[(long long)kk * stride];
            const double tv = q ? T * (1.0 + cq * (double)q[(long long)kk * stride]) : T;
            if (m == 0)
                zprev = (target == ORC_VZ_ALTITUDE ? zsd : 0.0) + (H * tv) * orc_vlog(psd / p[kk]);
            else
                zprev = zprev + (H * (0.5 * (tv + tvprev))) * orc_vlog(pprev / p[kk]);
            tvprev = tv;
            pprev = p[kk];
            zc[kk] = zprev;
        }
    }
    for (k = 0; k < nk; ++k)
        zc[k] = zc[k] - zsub;
    return s0;
}

/* one column's coordinates for the tests: zc[nk] as above; returns the direction (1, 0) or -1 */
int orc_height_column_z(int converter, int target, int kind, const double* ap, const double* b, int nk, double ptop, double ps_scale,
                        double z_scale, double zs_scale, const float* ps, const float* t, const float* q, const float* z, const float* zs,
                        double* zc)
{
    double* p = (double*)malloc(sizeof(double) * nk);
    const int dir = orc_height_column(converter, target, kind, ap, b, nk, ptop, ps ? (double)ps[0] * ps_scale : 0.0, z_scale, t, q, z, 1,
                                      zs ? (double)zs[0] * zs_scale : 0.0, p, zc);
    free(p);
    return dir;
}

/* in, t, q, z [nt][nk][nxy]; ps [nt][nxy]; zs [nxy]; out [nt][np][nxy].  Inputs a converter does not use may be NULL. */
int orc_vinterp_height(int method, int converter, int target, int kind, const double* ap, const double* b, int nk, double ptop, double ps_scale,
                       double z_scale, double zs_scale, const double* levels, int np, int extrapolate, const float* in, const float* ps,
                       const float* t, const float* q, const float* z, const float* zs, long nxy, long nt, float* out)
{
    long long ncol = (long long)nxy * nt;
    if (nk < 2 || np < 1 || (method != ORC_VINT_LIN && method != ORC_VINT_NN) || converter < ORC_VZ_STANDARD || converter > ORC_VZ_FIELD)
        return ORC_ERROR;
#pragma omp parallel
    {
        double* p = (double*)malloc(sizeof(double) * nk);
        double* zc = (double*)malloc(sizeof(double) * nk);
        double* zw = (double*)malloc(sizeof(double) * nk);
        long long col;
#pragma omp for schedule(static)
        for (col = 0; col < ncol; ++col) {
            const long long tt = col / nxy, c = col % nxy, base = tt * nk * nxy + c;
            const float* v = in + base;
            float* o = out + tt * np * nxy + c;
            const double psd = ps ? (double)ps[tt * nxy + c] * ps_scale : 0.0;
            const double zsd = zs ? (double)zs[c] * zs_scale : 0.0;
            const int dir = orc_height_column(converter, target, kind, ap, b, nk, ptop, psd, z_scale, t ? t + base : NULL, q ? q + base : NULL,
                                              z ? z + base : NULL, nxy, zsd, p, zc);
            int m, i, mnan = nk;
            for (m = 0; m < nk && dir >= 0; ++m) { /* walk order: from the surface upward */
                zw[m] = zc[dir ? m : nk - 1 - m];
                if (isnan(zw[m]) && mnan == nk)
                    mnan = m;
            }
            for (i = 0; i < np; ++i) {
                const double Z = levels[i];
                float r = orc_undef_f();
                int mm = -1;
                if (dir >= 0 && mnan > 0) {
                    if (Z < zw[0]) {
                        if (extrapolate)
                            mm = 0;
                    } else {
                        for (m = 0; m + 1 < mnan; ++m) { /* the first pair with Z between its ends, endpoints included */
                            const double lo = zw[m] < zw[m + 1] ? zw[m] : zw[m + 1], hi = zw[m] < zw[m + 1] ? zw[m + 1] : zw[m];
                            if (lo <= Z && Z <= hi) {
                                mm = m;
                                break;
                            }
                        }
                        if (mm < 0 && mnan == nk && extrapolate) /* above the top level (a NaN level ends the column) */
                            mm = nk - 2;
                    }
                }
                if (mm >= 0) {
                    const int ka = dir ? mm : nk - 1 - mm, kb = dir ? mm + 1 : nk - 2 - mm;
                    const double za = zw[mm], zb = zw[mm + 1];
                    const float A = v[(long long)ka * nxy], B = v[(long long)kb * nxy];
                    if (isnan(za) || isnan(zb))
                        r = orc_undef_f();
                    else if (method == ORC_VINT_NN)
                        r = fabs(Z - zb) < fabs(Z - za) ? B : A; /* a tie takes the lower level */
                    else {
                        const double w = za == zb ? 0.0 : (Z - za) / (zb - za);
                        r = (float)((double)A + w * ((double)B - (double)A));
                    }
                }
                o[(long long)i * nxy] = r;
            }
        }
        free(p);
        free(zc);
        free(zw);
    }
    return ORC_OK;
}
