/*
 * tests/vertical_depth_oracle.c -- TEST INFRASTRUCTURE ONLY.  CPU restatement (plain C99) of vertical interpolation to depth levels, the
 * depth branch of the reference's CDMVerticalInterpolator, written out as DESIGN.md section 2 states it (the reference's converters,
 * OceanSG1 / OceanSG2 and mifi_ocean_s_g1_z / _g2_z, are not compiled here).  It includes tests/vertical_oracle.c for the undefined
 * value and the method numbers.  Only tests/ and profiles/tools/vertical_depth_time.py load the library built from this file
 * (tests/vertical_depth_oracle.py compiles it on demand); libfimex_b200.so never links, loads or calls it.
 *
 * Build: gcc -std=gnu99 -O2 -ffp-contract=off -fPIC -fopenmp (no FMA contraction), as tests/vertical_oracle.c.
 */
#include "vertical_oracle.c"

enum { ORC_VD_DEPTH = 3, ORC_VD_OCEAN_SIGMA = 4, ORC_VD_OCEAN_S_G1 = 5, ORC_VD_OCEAN_S_G2 = 6 }; /* FB200_VCOORD_* */

/* z[nk] of one column, in the operation order of the contract: h = the sea-floor depth, eta = the sea surface height (0 when not
 * given); depth levels: z_k = -s_k.  dcs_k = depth_c * s_k is one rounded product, as the library forms it on the host. */
static void orc_depth_z(int vcoord, const double* s, const double* Ck, int nk, double depth_c, double h, double eta, double* z)
{
    int k;
    for (k = 0; k < nk; ++k) {
        if (vcoord == ORC_VD_DEPTH) {
            z[k] = -s[k];
        } else if (vcoord == ORC_VD_OCEAN_SIGMA) {
            z[k] = eta + s[k] * (h + eta);
        } else if (vcoord == ORC_VD_OCEAN_S_G1) {
            const double S = depth_c * s[k] + (h - depth_c) * Ck[k];
            z[k] = S + eta * (1.0 + S / h);
        } else {
            const double S = (depth_c * s[k] + h * Ck[k]) / (depth_c + h);
            z[k] = eta + (eta + h) * S;
        }
    }
}

/* The coordinate x[k] = -z_k of every level of one column and the column's direction: 1 when level 0 is the surface end (the smaller
 * x), 0 when level nk - 1 is, -1 for a NaN column (land: h NaN or <= 0; a NaN eta; equal or NaN ends). */
static int orc_depth_column(int vcoord, const double* s, const double* Ck, int nk, double depth_c, double h, double eta, double* x)
{
    int k;
    if (vcoord != ORC_VD_DEPTH && (!(h > 0.0) || isnan(eta)))
        return -1;
    orc_depth_z(vcoord, s, Ck, nk, depth_c, h, eta, x);
    for (k = 0; k < nk; ++k)
        x[k] = -x[k];
    if (!(x[0] < x[nk - 1]) && !(x[0] > x[nk - 1]))
        return -1;
    return x[0] < x[nk - 1];
}

/* one column's z_k for the tests (no NaN-column rules): z[nk] */
void orc_depth_column_z(int vcoord, const double* s, const double* Ck, int nk, double depth_c, double h, double eta, double* z)
{
    orc_depth_z(vcoord, s, Ck, nk, depth_c, h, eta, z);
}

/* in [nt][nk][nxy]; eta [nt][nxy] (NULL: 0); depth [nxy] (NULL for depth levels); out [nt][np][nxy] */
int orc_vinterp_depth(int method, int vcoord, const double* s, const double* Ck, int nk, double depth_c, const double* levels, int np,
                      int extrapolate, const float* in, const float* eta, const float* depth, long nxy, long nt, float* out)
{
    long long ncol = (long long)nxy * nt;
    if (nk < 2 || np < 1 || (method != ORC_VINT_LIN && method != ORC_VINT_NN) || vcoord < ORC_VD_DEPTH || vcoord > ORC_VD_OCEAN_S_G2 ||
        (vcoord != ORC_VD_DEPTH && !depth))
        return ORC_ERROR;
#pragma omp parallel
    {
        double* x = (double*)malloc(sizeof(double) * nk);
        double* xw = (double*)malloc(sizeof(double) * nk);
        long long col;
#pragma omp for schedule(static)
        for (col = 0; col < ncol; ++col) {
            const long long tt = col / nxy, c = col % nxy;
            const float* v = in + tt * nk * nxy + c;
            float* o = out + tt * np * nxy + c;
            const double h = depth ? (double)depth[c] : 0.0;
            const double e = eta ? (double)eta[tt * nxy + c] : 0.0;
            const int dir = orc_depth_column(vcoord, s, Ck, nk, depth_c, h, e, x);
            int m, i, mnan = nk;
            for (m = 0; m < nk && dir >= 0; ++m) { /* walk order: from the surface down */
                xw[m] = x[dir ? m : nk - 1 - m];
                if (isnan(xw[m]) && mnan == nk)
                    mnan = m;
            }
            for (i = 0; i < np; ++i) {
                const double D = levels[i];
                float r = orc_undef_f();
                int mm = -1;
                if (dir >= 0 && mnan > 0) {
                    if (D < xw[0]) { /* above the top level */
                        if (extrapolate)
                            mm = 0;
                    } else {
                        for (m = 0; m + 1 < mnan; ++m) { /* the first pair with D between its ends, endpoints included */
                            const double lo = xw[m] < xw[m + 1] ? xw[m] : xw[m + 1], hi = xw[m] < xw[m + 1] ? xw[m + 1] : xw[m];
                            if (lo <= D && D <= hi) {
                                mm = m;
                                break;
                            }
                        }
                        if (mm < 0 && mnan == nk && extrapolate) /* below the bottom level */
                            mm = nk - 2;
                    }
                }
                if (mm >= 0) {
                    const int ka = dir ? mm : nk - 1 - mm, kb = dir ? mm + 1 : nk - 2 - mm;
                    const double xa = xw[mm], xb = xw[mm + 1];
                    const float A = v[(long long)ka * nxy], B = v[(long long)kb * nxy];
                    if (isnan(xa) || isnan(xb))
                        r = orc_undef_f();
                    else if (method == ORC_VINT_NN)
                        r = fabs(D - xb) < fabs(D - xa) ? B : A; /* a tie takes the upper level */
                    else {
                        const double w = xa == xb ? 0.0 : (D - xa) / (xb - xa);
                        r = (float)((double)A + w * ((double)B - (double)A));
                    }
                }
                o[(long long)i * nxy] = r;
            }
        }
        free(x);
        free(xw);
    }
    return ORC_OK;
}
