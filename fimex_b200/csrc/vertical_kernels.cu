// fimex_b200/csrc/vertical_kernels.cu -- vertical interpolation to pressure levels: the pressure branch of the reference's
// CDMVerticalInterpolator (linear / log / loglog / nearest neighbour between the two model levels that bracket each target
// pressure; the per-column step of mifi_get_values_linear_f / _log_f / _log_log_f, src/interpolation.c:1030-1156).
//
// One thread per column, consecutive lanes on consecutive columns, so every load of a level row and every store of a
// target row coalesces.  The column's pressures are never materialised: p_k = a_k + b_k * q is evaluated from the
// coefficients in shared memory where the walk needs it (q = ps * ps_scale for hybrid levels, ps * ps_scale - ptop for
// sigma levels, 0 for pressure levels).  The targets are sorted once on the host, so one forward walk over k finds every
// bracket; a bracket shared with the previous target (or shifted by one level) reuses the values held in registers, and
// only the levels a column actually brackets are read.
//
// Arithmetic (DESIGN.md section 2): fp64, every product through __dmul_rn so that nothing is contracted into an FMA, and
// ln() by vlog() below, the same sequence of IEEE operations as the oracle's orc_vlog (tests/vertical_oracle.c) -- results are bit-identical.
//
// k_vertical_height is the height branch (targets in metres above sea level or above ground): the same walk, in the column's
// altitude z_k, which it computes level by level as the walk goes up from the surface (standard atmosphere of p_k, the
// hypsometric sum over T and q, or a z field) and never stores.  The walk ends at the bracket of the highest target, so a column
// is read only up to there (DESIGN.md sections 2 and 4).
//
// k_vertical_depth is the depth branch (targets in metres below the sea surface datum, from depth levels or the CF ocean sigma and
// s-coordinates): the same walk, down from the surface end, in x_k = -z_k, which it computes from the terms in shared memory and the
// column's sea-floor depth and sea surface height as it goes and never stores.  Land columns read no field value.
#include "kernels.h"

namespace fb {
namespace {

constexpr int kThreads = 256;

// ln(x): fdlibm's __ieee754_log (e_log.c) -- argument reduction to [sqrt(2)/2, sqrt(2)) and a degree-14 odd polynomial in
// s = f / (2 + f); < 1 ulp.  Only +, -, *, / and bit operations, so it rounds identically on the GPU and in plain C.
__device__ double vlog(double x)
{
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, two54 = 1.80143985094819840000e+16;
    const double Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                 Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                 Lg7 = 1.479819860511658591e-01;
    int hx = __double2hiint(x);
    const unsigned lx = (unsigned)__double2loint(x);
    int k = 0;
    if (hx < 0x00100000) { // x < 2^-1022
        if (((hx & 0x7fffffff) | lx) == 0)
            return -__longlong_as_double(0x7ff0000000000000ll); // log(+-0) = -inf
        if (hx < 0)
            return __longlong_as_double(0x7ff8000000000000ll); // log(negative) = NaN
        k -= 54;
        x = __dmul_rn(x, two54); // subnormal: scale up
        hx = __double2hiint(x);
    }
    if (hx >= 0x7ff00000)
        return x + x; // inf, NaN
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    const int i0 = (hx + 0x95f64) & 0x100000;
    x = __hiloint2double(hx | (i0 ^ 0x3ff00000), __double2loint(x)); // normalise x or x / 2
    k += (i0 >> 20);
    const double f = x - 1.0;
    const double dk = (double)k;
    if ((0x000fffff & (2 + hx)) < 3) { // |f| < 2^-20
        if (f == 0.0)
            return k == 0 ? 0.0 : __dmul_rn(dk, ln2_hi) + __dmul_rn(dk, ln2_lo);
        const double R = __dmul_rn(__dmul_rn(f, f), 0.5 - __dmul_rn(0.33333333333333333, f));
        return k == 0 ? f - R : __dmul_rn(dk, ln2_hi) - ((R - __dmul_rn(dk, ln2_lo)) - f);
    }
    const double s = f / (2.0 + f);
    const double z = __dmul_rn(s, s);
    int i = hx - 0x6147a;
    const double w = __dmul_rn(z, z);
    const int j = 0x6b851 - hx;
    const double t1 = __dmul_rn(w, Lg2 + __dmul_rn(w, Lg4 + __dmul_rn(w, Lg6)));
    const double t2 = __dmul_rn(z, Lg1 + __dmul_rn(w, Lg3 + __dmul_rn(w, Lg5 + __dmul_rn(w, Lg7))));
    i |= j;
    const double R = t2 + t1;
    if (i > 0) {
        const double hfsq = __dmul_rn(__dmul_rn(0.5, f), f);
        if (k == 0)
            return f - (hfsq - __dmul_rn(s, hfsq + R));
        return __dmul_rn(dk, ln2_hi) - ((hfsq - (__dmul_rn(s, hfsq + R) + __dmul_rn(dk, ln2_lo))) - f);
    }
    if (k == 0)
        return f - __dmul_rn(s, f - R);
    return __dmul_rn(dk, ln2_hi) - ((__dmul_rn(s, f - R) - __dmul_rn(dk, ln2_lo)) - f);
}

// the coordinate the weights are linear in: p (linear, nearest neighbour), ln p (log), ln ln p (loglog)
template <int M>
__device__ __forceinline__ double vcoord(double p)
{
    if (M == FB_VINT_LOG)
        return vlog(p);
    if (M == FB_VINT_LOGLOG)
        return vlog(vlog(p));
    return p;
}

__global__ void k_vert_coords(int method, const double* __restrict__ lev, double* __restrict__ x, int np)
{
    for (int i = threadIdx.x; i < np; i += blockDim.x) {
        const double p = lev[i];
        x[i] = method == FB_VINT_LOG ? vcoord<FB_VINT_LOG>(p) : method == FB_VINT_LOGLOG ? vcoord<FB_VINT_LOGLOG>(p) : p;
    }
}

// in [nt][nk][nxy], ps [nt][nxy] (null for pressure levels), out [nt][np][nxy]; blockIdx.y = time step.
// tab: a[nk] | b[nk] | sorted target pressures[np] | their coordinates[np] | output row of each sorted target[np]
// (4 blocks per SM: 40-56 registers, no spills; without the minimum ptxas holds the kernel at 32 registers and spills)
template <int M>
__global__ void __launch_bounds__(kThreads, 4) k_vertical(const float* __restrict__ in, const float* __restrict__ ps, float* __restrict__ out,
                                                       const double* __restrict__ tab, int nk, int np, int extrapolate, double ps_scale,
                                                       double shift, long long nxy, long long t0)
{
    extern __shared__ double s_tab[];
    const int ntab = 2 * nk + 3 * np;
    for (int i = threadIdx.x; i < ntab; i += blockDim.x)
        s_tab[i] = tab[i];
    __syncthreads();
    const double* s_a = s_tab;
    const double* s_b = s_tab + nk;
    const double* s_lev = s_tab + 2 * nk;
    const double* s_x = s_lev + np;
    const double* s_row = s_x + np;

    const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (c >= nxy)
        return;
    const long long t = t0 + blockIdx.y;
    const float* col = in + t * nk * nxy + c;
    float* ocol = out + t * np * nxy + c;
    const double q = ps ? __dmul_rn((double)__ldg(ps + t * nxy + c), ps_scale) - shift : 0.0;
    auto pres = [&](int k) { return s_a[k] + __dmul_rn(s_b[k], q); };

    const double p0 = pres(0), pl = pres(nk - 1);
    const bool incr = p0 < pl;
    const bool flat = !(p0 < pl) && !(p0 > pl); // equal ends or NaN
    const double lo = incr ? p0 : pl, hi = incr ? pl : p0;
    // Targets in the column's direction: the bracket index j (first level at or beyond P) never moves back.
    int j = 1, kc = -2;
    double pa = 0., pb = 0., xa = 0., xb = 0.;
    float va = 0.f, vb = 0.f;
    for (int ii = 0; ii < np; ++ii) {
        const int i = incr ? ii : np - 1 - ii;
        const double P = s_lev[i];
        float r = undef_f();
        if (!flat && (extrapolate || (P >= lo && P <= hi))) {
            if (incr) {
                while (j < nk - 1 && pres(j) < P)
                    ++j;
            } else {
                while (j < nk - 1 && pres(j) > P)
                    ++j;
            }
            const int k = j - 1;
            if (k != kc) {
                if (k == kc + 1) { // the lower level of this bracket is the upper one of the last
                    pa = pb;
                    xa = xb;
                    va = vb;
                } else {
                    pa = pres(k);
                    xa = vcoord<M>(pa);
                    va = __ldg(col + (long long)k * nxy);
                }
                pb = pres(k + 1);
                xb = vcoord<M>(pb);
                vb = __ldg(col + (long long)(k + 1) * nxy);
                kc = k;
            }
            if (M == FB_VINT_NN) {
                r = fabs(P - pb) < fabs(P - pa) ? vb : va;
            } else {
                const double w = xa == xb ? 0.0 : (s_x[i] - xa) / (xb - xa);
                r = (float)((double)va + __dmul_rn(w, (double)vb - (double)va));
            }
        }
        __stcs(ocol + (long long)s_row[i] * nxy, r);
    }
}

// exp(x): fdlibm's __ieee754_exp (e_exp.c) -- x = k ln2 + r, |r| <= ln2 / 2, and a degree-5 rational approximation in r; < 1 ulp.
// Only +, -, *, / and bit operations, as vlog; the oracle's orc_vexp (tests/vertical_height_oracle.c) is the same sequence.
__device__ double vexp(double x)
{
    const double twom1000 = 9.33263618503218878990e-302, o_threshold = 7.09782712893383973096e+02,
                 u_threshold = -7.45133219101941108420e+02, ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10,
                 invln2 = 1.44269504088896338700e+00;
    const double P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03, P3 = 6.61375632143793436117e-05,
                 P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
    const unsigned hw = (unsigned)__double2hiint(x), lx = (unsigned)__double2loint(x);
    const int xsb = (int)(hw >> 31);
    const unsigned hx = hw & 0x7fffffffu;
    if (hx >= 0x40862E42u) { // |x| >= 709.78...
        if (hx >= 0x7ff00000u) {
            if (((hx & 0xfffffu) | lx) != 0)
                return x + x; // NaN
            return xsb == 0 ? x : 0.0;
        }
        if (x > o_threshold)
            return __longlong_as_double(0x7ff0000000000000ll); // overflow: huge * huge
        if (x < u_threshold)
            return 0.0; // underflow: twom1000 * twom1000
    }
    double hi = 0.0, lo = 0.0;
    int k = 0;
    if (hx > 0x3fd62e42u) {     // |x| > 0.5 ln2
        if (hx < 0x3FF0A2B2u) { // and |x| < 1.5 ln2
            hi = xsb ? x + ln2_hi : x - ln2_hi;
            lo = xsb ? -ln2_lo : ln2_lo;
            k = 1 - xsb - xsb;
        } else {
            k = (int)(__dmul_rn(invln2, x) + (xsb ? -0.5 : 0.5));
            const double t = (double)k;
            hi = x - __dmul_rn(t, ln2_hi); // t * ln2_hi is exact here
            lo = __dmul_rn(t, ln2_lo);
        }
        x = hi - lo;
    } else if (hx < 0x3e300000u) { // |x| < 2^-28
        return 1.0 + x;
    }
    const double t = __dmul_rn(x, x);
    const double c = x - __dmul_rn(t, P1 + __dmul_rn(t, P2 + __dmul_rn(t, P3 + __dmul_rn(t, P4 + __dmul_rn(t, P5)))));
    if (k == 0)
        return 1.0 - (__dmul_rn(x, c) / (c - 2.0) - x);
    const double y = 1.0 - ((lo - __dmul_rn(x, c) / (2.0 - c)) - hi);
    if (k >= -1021)
        return __hiloint2double(__double2hiint(y) + (k << 20), __double2loint(y)); // add k to y's exponent
    return __dmul_rn(__hiloint2double(__double2hiint(y) + ((k + 1000) << 20), __double2loint(y)), twom1000);
}

// standard-atmosphere altitude of p: the last layer b with p <= p_b; layer constants [h_b | p_b | c_b | e_b] x kStdLayers (api.cu)
__device__ __forceinline__ double zstd(const double* __restrict__ L, double p)
{
    int b = 0;
#pragma unroll
    for (int l = 1; l < kStdLayers; ++l)
        if (p <= L[kStdLayers + l])
            b = l;
    const double h = L[b], pb = L[kStdLayers + b], c = L[2 * kStdLayers + b], e = L[3 * kStdLayers + b];
    if (e != 0.0)
        return h + __dmul_rn(c, vexp(__dmul_rn(e, vlog(p / pb))) - 1.0);
    return h + __dmul_rn(c, vlog(pb / p));
}

// in, t, q, z [nt][nk][nxy]; ps [nt][nxy]; zs [nxy]; out [nt][np][nxy]; blockIdx.y = time step.  Inputs the converter does not use
// are null (q: optional for the hypsometric converter).
// tab: a[nk] | b[nk] | standard-atmosphere layers[4 * kStdLayers] | sorted target levels[np] | output row of each sorted target[np]
template <int CONV, int M>
__global__ void __launch_bounds__(kThreads, 3)
    k_vertical_height(const float* __restrict__ in, const float* __restrict__ ps, const float* __restrict__ tt, const float* __restrict__ qq,
                      const float* __restrict__ zf, const float* __restrict__ zs, float* __restrict__ out, const double* __restrict__ tab, int nk,
                      int np, int extrapolate, int target, double ps_scale, double shift, double z_scale, double zs_scale, double H, double cq,
                      long long nxy, long long t0)
{
    extern __shared__ double s_tab[];
    const int ntab = 2 * nk + 4 * kStdLayers + 2 * np;
    for (int i = threadIdx.x; i < ntab; i += blockDim.x)
        s_tab[i] = tab[i];
    __syncthreads();
    const double* s_a = s_tab;
    const double* s_b = s_tab + nk;
    const double* s_std = s_tab + 2 * nk;
    const double* s_lev = s_std + 4 * kStdLayers;
    const double* s_row = s_lev + np;

    const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (c >= nxy)
        return;
    const long long t = t0 + blockIdx.y;
    const long long base = t * nk * nxy + c;
    const float* col = in + base;
    float* ocol = out + t * np * nxy + c;
    const double psd = ps ? __dmul_rn((double)__ldg(ps + t * nxy + c), ps_scale) : 0.0;
    const double qs = psd - shift;
    const double zsd = zs ? __dmul_rn((double)__ldg(zs + c), zs_scale) : 0.0;
    // the hypsometric sum starts at the surface altitude for altitude targets, at 0 for heights; the other converters subtract
    // z_s from z for heights
    const double zsub = (target == FB_VZ_HEIGHT && CONV != FB_VZ_HYPSOMETRIC) ? zsd : 0.0;
    auto pres = [&](int k) { return s_a[k] + __dmul_rn(s_b[k], qs); };
    auto zfield = [&](int k) { return __dmul_rn(z_scale, (double)__ldg(zf + base + (long long)k * nxy)); };

    bool up, flat; // up: level 0 is the surface end
    if (CONV == FB_VZ_FIELD) {
        const double z0 = zfield(0), zl = zfield(nk - 1);
        up = z0 < zl;
        flat = !(z0 < zl) && !(z0 > zl);
    } else {
        const double p0 = pres(0), pl = pres(nk - 1);
        up = p0 > pl;
        flat = !(p0 < pl) && !(p0 > pl);
    }
    // The walk: level m counted from the surface; zj = the coordinate of level j, zjm = that of level j - 1.  The hypsometric
    // converter carries Tv and p of level j in registers and returns the increment of its sum over the layer below level m.
    double tvj = 0.0, pj = 0.0;
    auto level_z = [&](int m) -> double {
        const int k = up ? m : nk - 1 - m;
        if (CONV == FB_VZ_FIELD)
            return zfield(k) - zsub;
        const double p = pres(k);
        if (CONV == FB_VZ_STANDARD)
            return zstd(s_std, p) - zsub;
        const double T = (double)__ldg(tt + base + (long long)k * nxy);
        const double tv = qq ? __dmul_rn(T, 1.0 + __dmul_rn(cq, (double)__ldg(qq + base + (long long)k * nxy))) : T;
        const double hterm = m == 0 ? __dmul_rn(H, tv) : __dmul_rn(H, __dmul_rn(0.5, tv + tvj));
        const double dz = __dmul_rn(hterm, vlog((m == 0 ? psd : pj) / p));
        tvj = tv;
        pj = p;
        return dz;
    };
    double z0 = 0.0, zjm = 0.0, zj = 0.0;
    if (!flat) {
        z0 = CONV == FB_VZ_HYPSOMETRIC ? (target == FB_VZ_ALTITUDE ? zsd : 0.0) + level_z(0) : level_z(0);
        zj = CONV == FB_VZ_HYPSOMETRIC ? z0 + level_z(1) : level_z(1);
        zjm = z0;
        flat = isnan(z0);
    }
    int j = 1, kc = -2;
    float va = 0.f, vb = 0.f;
    for (int i = 0; i < np; ++i) {
        const double Z = s_lev[i];
        float r = undef_f();
        if (!flat) {
            while (j < nk - 1 && zj < Z) { // NaN stops the walk: every target above it gets NaN
                zjm = zj;
                ++j;
                zj = CONV == FB_VZ_HYPSOMETRIC ? zjm + level_z(j) : level_z(j);
            }
            if (extrapolate || (Z >= z0 && !(j == nk - 1 && zj < Z))) {
                const int k = j - 1;
                const int ka = up ? k : nk - 1 - k, kb = up ? k + 1 : nk - 2 - k;
                if (k != kc) {
                    va = k == kc + 1 ? vb : __ldg(col + (long long)ka * nxy); // the lower level of this bracket is the upper one of the last
                    vb = __ldg(col + (long long)kb * nxy);
                    kc = k;
                }
                if (isnan(zjm) || isnan(zj)) {
                    r = undef_f();
                } else if (M == FB_VINT_NN) {
                    r = fabs(Z - zj) < fabs(Z - zjm) ? vb : va;
                } else {
                    const double w = zjm == zj ? 0.0 : (Z - zjm) / (zj - zjm);
                    r = (float)((double)va + __dmul_rn(w, (double)vb - (double)va));
                }
            }
        }
        __stcs(ocol + (long long)s_row[i] * nxy, r);
    }
}

// in [nt][nk][nxy]; eta [nt][nxy] (null: 0); depth [nxy] (null for depth levels); out [nt][np][nxy]; blockIdx.y = time step.
// tab: levels, sigma_k or depth_c * s_k [nk] | C_k [nk] | sorted target depths[np] | output row of each sorted target[np]
template <int VC, int M>
__global__ void __launch_bounds__(kThreads, 3)
    k_vertical_depth(const float* __restrict__ in, const float* __restrict__ eta, const float* __restrict__ depth, float* __restrict__ out,
                     const double* __restrict__ tab, int nk, int np, int extrapolate, double depth_c, long long nxy, long long t0)
{
    extern __shared__ double s_tab[];
    const int ntab = 2 * nk + 2 * np;
    for (int i = threadIdx.x; i < ntab; i += blockDim.x)
        s_tab[i] = tab[i];
    __syncthreads();
    const double* s_a = s_tab;
    const double* s_c = s_tab + nk;
    const double* s_lev = s_tab + 2 * nk;
    const double* s_row = s_lev + np;

    const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (c >= nxy)
        return;
    const long long t = t0 + blockIdx.y;
    const float* col = in + t * nk * nxy + c;
    float* ocol = out + t * np * nxy + c;
    // the sea-floor depth h and the sea surface height e: land (h NaN or <= 0) and a NaN eta give a NaN column, which reads no field value
    double h = 0.0, e = 0.0;
    bool flat = false;
    if (VC != FB_VD_DEPTH) {
        h = (double)__ldg(depth + c);
        flat = !(h > 0.0);
        if (!flat && eta) {
            e = (double)__ldg(eta + t * nxy + c);
            flat = isnan(e);
        }
    }
    const double eh = e + h;                                                // sigma, g2
    const double hd = VC == FB_VD_OCEAN_S_G1 ? h - depth_c : depth_c + h; // g1: h - depth_c; g2: depth_c + h
    // x_k = -z_k, the depth of level k below the datum of eta (DESIGN.md section 2)
    auto level_x = [&](int k) -> double {
        if (VC == FB_VD_DEPTH)
            return s_a[k];
        if (VC == FB_VD_OCEAN_SIGMA)
            return -(e + __dmul_rn(s_a[k], eh));
        if (VC == FB_VD_OCEAN_S_G1) {
            const double S = s_a[k] + __dmul_rn(hd, s_c[k]);
            return -(S + __dmul_rn(e, 1.0 + S / h));
        }
        const double S = (s_a[k] + __dmul_rn(h, s_c[k])) / hd;
        return -(e + __dmul_rn(eh, S));
    };
    // The walk: level m counted from the surface end (the smaller x); xj = the coordinate of level j, xjm = that of level j - 1.
    bool up = true;
    double x0 = 0.0, xjm = 0.0, xj = 0.0;
    if (!flat) {
        const double xf = level_x(0), xl = level_x(nk - 1);
        up = xf < xl;
        flat = !(xf < xl) && !(xf > xl);
        x0 = up ? xf : xl;
        xj = up ? level_x(1) : level_x(nk - 2);
        xjm = x0;
    }
    int j = 1, kc = -2;
    float va = 0.f, vb = 0.f;
    for (int i = 0; i < np; ++i) {
        const double D = s_lev[i];
        float r = undef_f();
        if (!flat) {
            while (j < nk - 1 && xj < D) { // NaN stops the walk: every target below it gets NaN
                xjm = xj;
                ++j;
                xj = level_x(up ? j : nk - 1 - j);
            }
            if (extrapolate || (D >= x0 && !(j == nk - 1 && xj < D))) {
                const int k = j - 1;
                const int ka = up ? k : nk - 1 - k, kb = up ? k + 1 : nk - 2 - k;
                if (k != kc) {
                    va = k == kc + 1 ? vb : __ldg(col + (long long)ka * nxy); // the upper level of this bracket is the lower one of the last
                    vb = __ldg(col + (long long)kb * nxy);
                    kc = k;
                }
                if (isnan(xjm) || isnan(xj)) {
                    r = undef_f();
                } else if (M == FB_VINT_NN) {
                    r = fabs(D - xj) < fabs(D - xjm) ? vb : va;
                } else {
                    const double w = xjm == xj ? 0.0 : (D - xjm) / (xj - xjm);
                    r = (float)((double)va + __dmul_rn(w, (double)vb - (double)va));
                }
            }
        }
        __stcs(ocol + (long long)s_row[i] * nxy, r);
    }
}

// The data conversions of the vertical interpolator (CDMPressureConversions: theta2T, omega2vwind, add4Dpressure) on [nt][nk][nxy]
// fields, one thread per column and time step, level by level: every level row is a coalesced load and store.  p_k as the pressure
// handles form it (a, b and the shift of a VertTable), evaluated where it is needed and never stored except as add4Dpressure's output.
// in [nt][nk][nxy] (theta or omega; unused for FB_VCONV_PRESSURE), ps [nt][nxy] (null for pressure levels), tt [nt][nk][nxy]
// (omega2vwind), out [nt][nk][nxy].  in and out may be the same array, so neither is __restrict__ nor read through the texture path.
// tab: a[nk] | b[nk]; pressure levels: the factor (p_k / p0)^kappa of every level is formed once per block in s_tab[nk .. 2 nk)
template <int OP, int VC>
__global__ void __launch_bounds__(kThreads)
    k_vconvert(const float* in, const float* __restrict__ ps, const float* tt, float* out, const double* __restrict__ tab, int nk,
               double ps_scale, double shift, double kappa, double H, long long nxy, long long t0)
{
    extern __shared__ double s_tab[];
    for (int i = threadIdx.x; i < 2 * nk; i += blockDim.x)
        s_tab[i] = tab[i];
    __syncthreads();
    const double* s_a = s_tab;
    const double* s_b = s_tab + nk;
    if (OP == FB_VCONV_THETA2T && VC == FB_VCOORD_PRESSURE) {
        for (int k = threadIdx.x; k < nk; k += blockDim.x)
            s_tab[nk + k] = vexp(__dmul_rn(kappa, vlog(s_a[k] / 1000.0)));
        __syncthreads();
    }

    const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (c >= nxy)
        return;
    const long long t = t0 + blockIdx.y;
    const long long base = t * nk * nxy + c;
    const double q = VC == FB_VCOORD_PRESSURE ? 0.0 : __dmul_rn((double)__ldg(ps + t * nxy + c), ps_scale) - shift;
#pragma unroll 4
    for (int k = 0; k < nk; ++k) {
        const long long i = base + (long long)k * nxy;
        const double p = VC == FB_VCOORD_PRESSURE ? s_a[k] : s_a[k] + __dmul_rn(s_b[k], q);
        double r;
        if (OP == FB_VCONV_THETA2T) {
            const double f = VC == FB_VCOORD_PRESSURE ? s_b[k] : vexp(__dmul_rn(kappa, vlog(p / 1000.0)));
            r = __dmul_rn((double)in[i], f);
        } else if (OP == FB_VCONV_OMEGA2VWIND) {
            r = -__dmul_rn((double)in[i], __dmul_rn(H, (double)tt[i])) / __dmul_rn(100.0, p);
        } else {
            r = p;
        }
        __stcs(out + i, (float)r);
    }
}

} // namespace

int launch_vert_coords(int method, const double* d_lev, double* d_x, int np, cudaStream_t st)
{
    k_vert_coords<<<1, kThreads, 0, st>>>(method, d_lev, d_x, np);
    count_launch();
    FB_CUDA_CHECK(cudaGetLastError());
    return FB_OK;
}

int launch_vertical(const VertTable& vt, const float* d_in, const float* d_ps, long long nxy, long long nt, float* d_out, cudaStream_t st)
{
    if (nxy == 0 || nt == 0)
        return FB_OK;
    const size_t smem = sizeof(double) * (size_t)(2 * vt.nk + 3 * vt.np);
    const long long bx = (nxy + kThreads - 1) / kThreads;
    FB_REQUIRE(bx < 2147483647LL, "too many columns for one call");
    for (long long t0 = 0; t0 < nt; t0 += 65535) {
        const dim3 grid((unsigned)bx, (unsigned)std::min<long long>(nt - t0, 65535));
        switch (vt.method) {
#define FB_CASE(M)                                                                                                                         \
    case M:                                                                                                                                \
        k_vertical<M><<<grid, kThreads, smem, st>>>(d_in, d_ps, d_out, vt.d_tab, vt.nk, vt.np, vt.extrapolate ? 1 : 0, vt.ps_scale,       \
                                                    vt.shift, nxy, t0);                                                                    \
        break;
            FB_CASE(FB_VINT_LIN)
            FB_CASE(FB_VINT_LOG)
            FB_CASE(FB_VINT_LOGLOG)
            FB_CASE(FB_VINT_NN)
#undef FB_CASE
        default:
            FB_REQUIRE(false, "unknown vertical interpolation method " + std::to_string(vt.method));
        }
        count_launch();
        FB_CUDA_CHECK(cudaGetLastError());
    }
    return FB_OK;
}

int launch_vertical_height(const VertTable& vt, const float* d_in, const float* d_ps, const float* d_t, const float* d_q, const float* d_z,
                           const float* d_zs, long long nxy, long long nt, float* d_out, cudaStream_t st)
{
    if (nxy == 0 || nt == 0)
        return FB_OK;
    const size_t smem = sizeof(double) * (size_t)(2 * vt.nk + 4 * kStdLayers + 2 * vt.np);
    const long long bx = (nxy + kThreads - 1) / kThreads;
    FB_REQUIRE(bx < 2147483647LL, "too many columns for one call");
    const int key = vt.converter * 8 + vt.method;
    for (long long t0 = 0; t0 < nt; t0 += 65535) {
        const dim3 grid((unsigned)bx, (unsigned)std::min<long long>(nt - t0, 65535));
        switch (key) {
#define FB_CASE(C, M)                                                                                                                      \
    case C * 8 + M:                                                                                                                        \
        k_vertical_height<C, M><<<grid, kThreads, smem, st>>>(d_in, d_ps, d_t, d_q, d_z, d_zs, d_out,                 vt.d_tab, vt.nk, vt.np, \
                                                              vt.extrapolate ? 1 : 0, vt.target, vt.ps_scale, vt.shift, vt.z_scale,        \
                                                              vt.zs_scale, vt.H, vt.cq, nxy, t0);                                          \
        break;
            FB_CASE(FB_VZ_STANDARD, FB_VINT_LIN)
            FB_CASE(FB_VZ_STANDARD, FB_VINT_NN)
            FB_CASE(FB_VZ_HYPSOMETRIC, FB_VINT_LIN)
            FB_CASE(FB_VZ_HYPSOMETRIC, FB_VINT_NN)
            FB_CASE(FB_VZ_FIELD, FB_VINT_LIN)
            FB_CASE(FB_VZ_FIELD, FB_VINT_NN)
#undef FB_CASE
        default:
            FB_REQUIRE(false, "unknown height converter / method " + std::to_string(vt.converter) + " / " + std::to_string(vt.method));
        }
        count_launch();
        FB_CUDA_CHECK(cudaGetLastError());
    }
    return FB_OK;
}

int launch_vertical_depth(const VertTable& vt, const float* d_in, const float* d_eta, const float* d_depth, long long nxy, long long nt, float* d_out,
                          cudaStream_t st)
{
    if (nxy == 0 || nt == 0)
        return FB_OK;
    FB_REQUIRE(vt.depth_vcoord == FB_VD_DEPTH || d_depth != nullptr, "ocean s- and sigma coordinates need the sea-floor depth");
    const size_t smem = sizeof(double) * (size_t)(2 * vt.nk + 2 * vt.np);
    const long long bx = (nxy + kThreads - 1) / kThreads;
    FB_REQUIRE(bx < 2147483647LL, "too many columns for one call");
    const int key = vt.depth_vcoord * 8 + vt.method;
    for (long long t0 = 0; t0 < nt; t0 += 65535) {
        const dim3 grid((unsigned)bx, (unsigned)std::min<long long>(nt - t0, 65535));
        switch (key) {
#define FB_CASE(V, M)                                                                                                                      \
    case V * 8 + M:                                                                                                                        \
        k_vertical_depth<V, M><<<grid, kThreads, smem, st>>>(d_in, d_eta, d_depth, d_out, vt.d_tab, vt.nk, vt.np, vt.extrapolate ? 1 : 0,  \
                                                             vt.depth_c, nxy, t0);                                                         \
        break;
            FB_CASE(FB_VD_DEPTH, FB_VINT_LIN)
            FB_CASE(FB_VD_DEPTH, FB_VINT_NN)
            FB_CASE(FB_VD_OCEAN_SIGMA, FB_VINT_LIN)
            FB_CASE(FB_VD_OCEAN_SIGMA, FB_VINT_NN)
            FB_CASE(FB_VD_OCEAN_S_G1, FB_VINT_LIN)
            FB_CASE(FB_VD_OCEAN_S_G1, FB_VINT_NN)
            FB_CASE(FB_VD_OCEAN_S_G2, FB_VINT_LIN)
            FB_CASE(FB_VD_OCEAN_S_G2, FB_VINT_NN)
#undef FB_CASE
        default:
            FB_REQUIRE(false, "unknown depth coordinate / method " + std::to_string(vt.depth_vcoord) + " / " + std::to_string(vt.method));
        }
        count_launch();
        FB_CUDA_CHECK(cudaGetLastError());
    }
    return FB_OK;
}

int launch_vconvert(int op, int vcoord, const VertTable& vt, double kappa, const float* d_in, const float* d_ps, const float* d_t, long long nxy,
                    long long nt, float* d_out, cudaStream_t st)
{
    if (nxy == 0 || nt == 0)
        return FB_OK;
    const size_t smem = sizeof(double) * (size_t)(2 * vt.nk);
    const long long bx = (nxy + kThreads - 1) / kThreads;
    FB_REQUIRE(bx < 2147483647LL, "too many columns for one call");
    const int key = op * 8 + vcoord;
    for (long long t0 = 0; t0 < nt; t0 += 65535) {
        const dim3 grid((unsigned)bx, (unsigned)std::min<long long>(nt - t0, 65535));
        switch (key) {
#define FB_CASE(O, V)                                                                                                                      \
    case O * 8 + V:                                                                                                                        \
        k_vconvert<O, V><<<grid, kThreads, smem, st>>>(d_in, d_ps, d_t, d_out, vt.d_tab, vt.nk, vt.ps_scale, vt.shift, kappa, vt.H, nxy, t0); \
        break;
            FB_CASE(FB_VCONV_THETA2T, FB_VCOORD_PRESSURE)
            FB_CASE(FB_VCONV_THETA2T, FB_VCOORD_HYBRID)
            FB_CASE(FB_VCONV_THETA2T, FB_VCOORD_SIGMA)
            FB_CASE(FB_VCONV_OMEGA2VWIND, FB_VCOORD_PRESSURE)
            FB_CASE(FB_VCONV_OMEGA2VWIND, FB_VCOORD_HYBRID)
            FB_CASE(FB_VCONV_OMEGA2VWIND, FB_VCOORD_SIGMA)
            FB_CASE(FB_VCONV_PRESSURE, FB_VCOORD_PRESSURE)
            FB_CASE(FB_VCONV_PRESSURE, FB_VCOORD_HYBRID)
            FB_CASE(FB_VCONV_PRESSURE, FB_VCOORD_SIGMA)
#undef FB_CASE
        default:
            FB_REQUIRE(false, "unknown data conversion / source coordinate " + std::to_string(op) + " / " + std::to_string(vcoord));
        }
        count_launch();
        FB_CUDA_CHECK(cudaGetLastError());
    }
    return FB_OK;
}

} // namespace fb
