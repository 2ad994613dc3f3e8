/*
 * tests/vertical_convert_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement (plain C99) of the data conversions of the vertical
 * interpolator (--verticalInterpolate.dataConversion: theta2T, omega2vwind, add4Dpressure; the reference's CDMPressureConversions,
 * C++ and not compiled here), written out as DESIGN.md section 2 states it.  It includes tests/vertical_height_oracle.c (and through it
 * tests/vertical_oracle.c), so that ln() (orc_vlog), exp() (orc_vexp) and the constants R*, M and g0 are the very code the height
 * branch's restatement uses.  Only tests/ and profiles/tools/vertical_convert_time.py load the library built from this file
 * (tests/vertical_convert_oracle.py compiles it on demand); libfimex_b200.so never links, loads or calls it.
 *
 * Build: gcc -std=gnu99 -O2 -ffp-contract=off -fPIC -fopenmp (no FMA contraction), as tests/vertical_oracle.c.
 */
#include "vertical_height_oracle.c"

enum { ORC_VCONV_THETA2T = 0, ORC_VCONV_OMEGA2VWIND = 1, ORC_VCONV_PRESSURE = 2 };

/* p_k [hPa] of level k: pressure levels ap_k; hybrid ap_k + b_k psd; sigma ptop + sigma_k (psd - ptop), psd = ps * ps_scale */
static double orc_conv_pressure(int kind, const double* ap, const double* b, int k, double ptop, double psd)
{
    if (kind == ORC_VCOORD_HYBRID)
        return ap[k] + b[k] * psd;
    if (kind == ORC_VCOORD_SIGMA)
        return ptop + b[k] * (psd - ptop);
    return ap[k];
}

/* one value in fp64, before the rounding to float: x = theta or omega, T the air temperature (omega2vwind), p = p_k [hPa] */
double orc_vconv_value(int op, double x, double T, double p)
{
    const double kappa = 2.0 / 7.0, H = orc_H();
    if (op == ORC_VCONV_THETA2T)
        return x * orc_vexp(kappa * orc_vlog(p / 1000.0));
    if (op == ORC_VCONV_OMEGA2VWIND)
        return -(x * (H * T)) / (100.0 * p);
    return p;
}

/* in, t [nt][nk][nxy] (in unused for ORC_VCONV_PRESSURE, t for all but omega2vwind); ps [nt][nxy] (unused for pressure levels);
 * out [nt][nk][nxy] */
int orc_vconvert(int op, int kind, const double* ap, const double* b, int nk, double ptop, double ps_scale, const float* in, const float* ps,
                 const float* t, long nxy, long nt, float* out)
{
    long long ncol = (long long)nxy * nt, col;
    if (nk < 1 || op < ORC_VCONV_THETA2T || op > ORC_VCONV_PRESSURE || kind < ORC_VCOORD_PRESSURE || kind > ORC_VCOORD_SIGMA)
        return ORC_ERROR;
#pragma omp parallel for schedule(static)
    for (col = 0; col < ncol; ++col) {
        const long long tt = col / nxy, c = col % nxy;
        const double psd = kind != ORC_VCOORD_PRESSURE ? (double)ps[tt * nxy + c] * ps_scale : 0.0;
        int k;
        for (k = 0; k < nk; ++k) {
            const long long i = (tt * nk + k) * nxy + c;
            const double p = orc_conv_pressure(kind, ap, b, k, ptop, psd);
            const double x = op == ORC_VCONV_PRESSURE ? 0.0 : (double)in[i];
            const double T = op == ORC_VCONV_OMEGA2VWIND ? (double)t[i] : 0.0;
            out[i] = (float)orc_vconv_value(op, x, T, p);
        }
    }
    return ORC_OK;
}
