// fimex_b200/csrc/coordnn_kernels.cu -- K9: the coord_nearestneighbor index search.
//
// Replaces fastTranslatePointsToClosestInputCell + getGridDistance
// (/root/reference/src/CDMInterpolator.cc:1141-1220, :1064-1125).  The reference sorts the source points by
// latitude, and for every target scans up and down from lower_bound(latitude) while |dlat| <= the best
// distance so far, keeping the candidate with the strictly largest
//     cos_d = cos(lat_s) cos(lat_t) cos(lon_s - lon_t) + sin(lat_s) sin(lat_t).
// Because a great-circle distance is never smaller than the latitude difference, that pruned scan finds the
// global maximum of cos_d over the candidates inside the initial window |dlat| <= ROI (cos_d > cos ROI),
// ties going to the candidate met first (upwards from lower_bound, then downwards).  Here one WARP owns a
// target: its lanes stride over the window, and a shuffle reduction keeps (max cos_d, min scan rank).
// The latitude sort is a stable radix sort on the device (cub), so ties among equal latitudes follow the
// reference's insertion order (ix outer, iy inner); std::sort in the reference is unstable, so that order
// is unspecified there (SURVEY.md 8a trap 12).
#include "kernels.h"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cmath>
#include <vector>

namespace fb {

namespace {

constexpr int kThreads = 256;

struct SrcPoint {
    double lat, lon, coslat, sinlat;
    int x, y;
};

// order-preserving map double -> uint64 for the radix sort
__device__ __forceinline__ unsigned long long orderable(double v)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}

// insertion order of the reference: for ix, for iy: pos = ix + iy*nx, skipping NaN coordinates
__global__ void k_nn_keys(const double* __restrict__ lon, const double* __restrict__ lat, int nx, int ny, unsigned long long* __restrict__ keys,
                          int* __restrict__ vals)
{
    const long long n = (long long)nx * ny;
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < n; s += (long long)gridDim.x * blockDim.x) {
        const int ix = (int)(s / ny), iy = (int)(s % ny);
        const long long pos = ix + (long long)iy * nx;
        const bool bad = isnan(lon[pos]) || isnan(lat[pos]);
        // invalid points sort last and are cut off; -0 + 0 is +0, so -0 and +0 are one key and keep insertion order
        keys[s] = bad ? 0xffffffffffffffffull : orderable(lat[pos] + 0.);
        vals[s] = (int)s;
    }
}

__global__ void k_nn_points(const double* __restrict__ lon, const double* __restrict__ lat, int nx, int ny, const int* __restrict__ order,
                            long long m, SrcPoint* __restrict__ pts, double* __restrict__ sorted_lat)
{
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < m; k += (long long)gridDim.x * blockDim.x) {
        const int s = order[k];
        const int ix = s / ny, iy = s % ny;
        const long long pos = ix + (long long)iy * nx;
        SrcPoint p;
        p.lat = lat[pos];
        p.lon = lon[pos];
        sincos(p.lat, &p.sinlat, &p.coslat);
        p.x = ix;
        p.y = iy;
        pts[k] = p;
        sorted_lat[k] = p.lat;
    }
}

__global__ void k_count_valid(const double* __restrict__ lon, const double* __restrict__ lat, long long n, unsigned long long* count)
{
    unsigned long long c = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        c += !(isnan(lon[i]) || isnan(lat[i]));
    for (int o = 16; o > 0; o >>= 1)
        c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c)
        atomicAdd(count, c);
}

// getGridDistance: one block per sample; max cos_d to any other valid source point
__global__ void k_grid_distance(const double* __restrict__ lon, const double* __restrict__ lat, long long n, long long step,
                                double* __restrict__ best_out)
{
    __shared__ double sbest[kThreads / 32];
    const long long sp = blockIdx.x * step;
    const double lon0 = lon[sp], lat0 = lat[sp];
    double best = -2.;
    if (!(isnan(lon0) || isnan(lat0))) {
        double s0, c0;
        sincos(lat0, &s0, &c0);
        for (long long i = threadIdx.x; i < n; i += blockDim.x) {
            if (i == sp)
                continue;
            const double lo = lon[i], la = lat[i];
            if (isnan(lo) || isnan(la))
                continue;
            double s1, c1;
            sincos(la, &s1, &c1);
            const double cd = c0 * c1 * cos(lon0 - lo) + s0 * s1;
            if (cd > best)
                best = cd;
        }
    } else {
        best = 3.; // marks "sample skipped" (the reference does not push it)
    }
    for (int o = 16; o > 0; o >>= 1) {
        const double b2 = __shfl_xor_sync(0xffffffffu, best, o);
        if (b2 > best)
            best = b2;
    }
    if ((threadIdx.x & 31) == 0)
        sbest[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < kThreads / 32; ++k)
            if (sbest[k] > best)
                best = sbest[k];
        best_out[blockIdx.x] = best;
    }
}

__global__ void __launch_bounds__(kThreads) k_nn_search(double* __restrict__ px, double* __restrict__ py, long long n,
                                                      const SrcPoint* __restrict__ pts, const double* __restrict__ sorted_lat, long long m,
                                                      double min_grid_cos, double roi, unsigned long long* ties)
{
    const int lane = threadIdx.x & 31;
    const long long warp = (blockIdx.x * (long long)kThreads + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * kThreads) >> 5;
    for (long long t = warp; t < n; t += nwarps) {
        const double plat = py[t], plon = px[t];
        double sp, cp;
        sincos(plat, &sp, &cp);
        // lower_bound(latitude) and the window |dlat| <= roi (one cell of slack each side, predicate re-checked)
        long long lb, a, b;
        {
            long long lo = 0, hi = m;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (sorted_lat[mid] < plat)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            lb = lo;
            lo = 0;
            hi = lb;
            const double lowlat = plat - roi;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (sorted_lat[mid] < lowlat)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            a = lo > 0 ? lo - 1 : 0;
            lo = lb;
            hi = m;
            const double highlat = plat + roi;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (sorted_lat[mid] <= highlat)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            b = lo < m ? lo + 1 : m;
        }
        double best = min_grid_cos;
        long long best_rank = 0x7fffffffffffffffLL;
        int bx = -1, by = -1;
        int tie = 0;
        for (long long k = a + lane; k < b; k += 32) {
            const SrcPoint s = pts[k];
            if (fabs(s.lat - plat) > roi)
                continue;
            const double dlon = s.lon - plon;
            const double cd = s.coslat * cp * cos(dlon) + s.sinlat * sp;
            const long long rank = (k >= lb) ? (k - lb) : (m - lb) + (lb - 1 - k);
            if (cd > best || (cd == best && bx >= 0 && rank < best_rank)) {
                tie = (cd == best && bx >= 0);
                best = cd;
                best_rank = rank;
                bx = s.x;
                by = s.y;
            } else if (cd == best && bx >= 0) {
                tie = 1;
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double b2 = __shfl_xor_sync(0xffffffffu, best, o);
            const long long r2 = __shfl_xor_sync(0xffffffffu, best_rank, o);
            const int x2 = __shfl_xor_sync(0xffffffffu, bx, o);
            const int y2 = __shfl_xor_sync(0xffffffffu, by, o);
            const int t2 = __shfl_xor_sync(0xffffffffu, tie, o);
            if (x2 >= 0) {
                if (bx < 0 || b2 > best || (b2 == best && r2 < best_rank)) {
                    tie = (bx >= 0 && b2 == best) ? 1 : t2;
                    best = b2;
                    best_rank = r2;
                    bx = x2;
                    by = y2;
                } else if (b2 == best) {
                    tie = 1;
                }
            }
        }
        if (lane == 0) {
            px[t] = (double)bx; // (-1,-1) when nothing is closer than the ROI (LL_POINT default, :1134)
            py[t] = (double)by;
            if (tie)
                atomicAdd(ties, 1ull);
        }
    }
}

// ---- coord_kdtree (MIFI_INTERPOL_COORD_NN_KD): flannTranslatePointsToClosestInputCell, CDMInterpolator.cc:991-1062 --------
// The reference puts every source point on the unit sphere (cos lat cos lon, cos lat sin lon, sin lat), builds a nanoflann
// kd-tree and, per target, takes the first match of radiusSearch(sorted): the source point with the smallest squared
// chord distance d0*d0 + d1*d1 + d2*d2 (PointCloud::kdtree_distance, :967-973) that is < (maxDist / R)^2, or (-1000, -1000).
// A kd-tree only prunes; the answer is the exact nearest neighbour inside the radius.  Here: the latitude-sorted array of K9,
// a window |dlat| <= the angle of the chord radius, one warp per target, the same distance expression.
struct KdPoint {
    double lat, x, y, z;
    int ix, iy;
};

__global__ void k_kd_points(const double* __restrict__ lon, const double* __restrict__ lat, int nx, int ny, const int* __restrict__ order,
                            long long m, KdPoint* __restrict__ pts, double* __restrict__ sorted_lat)
{
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < m; k += (long long)gridDim.x * blockDim.x) {
        const int s = order[k];
        const int ix = s / ny, iy = s % ny;
        const long long pos = ix + (long long)iy * nx;
        KdPoint p;
        p.lat = lat[pos];
        double sla, cla, slo, clo;
        sincos(p.lat, &sla, &cla);
        sincos(lon[pos], &slo, &clo);
        p.x = __dmul_rn(cla, clo); // :1013-1015
        p.y = __dmul_rn(cla, slo);
        p.z = sla;
        p.ix = ix;
        p.iy = iy;
        pts[k] = p;
        sorted_lat[k] = p.lat;
    }
}

__global__ void __launch_bounds__(kThreads) k_kd_search(double* __restrict__ px, double* __restrict__ py, long long n,
                                                      const KdPoint* __restrict__ pts, const double* __restrict__ sorted_lat, long long m,
                                                      double radius2, double window, int nx, unsigned long long* ties)
{
    const int lane = threadIdx.x & 31;
    const long long warp = (blockIdx.x * (long long)kThreads + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * kThreads) >> 5;
    for (long long t = warp; t < n; t += nwarps) {
        const double plat = py[t], plon = px[t];
        double sla, cla, slo, clo;
        sincos(plat, &sla, &cla);
        sincos(plon, &slo, &clo);
        const double qx = __dmul_rn(cla, clo), qy = __dmul_rn(cla, slo), qz = sla; // :1045-1047
        // the window is centred on the latitude of the point q, which a target beyond a pole (|plat| > pi/2) is not
        double wlat = remainder(plat, 2. * FB_PI);
        if (wlat > 0.5 * FB_PI)
            wlat = FB_PI - wlat;
        else if (wlat < -0.5 * FB_PI)
            wlat = -FB_PI - wlat;
        long long a, b;
        {
            long long lo = 0, hi = m;
            const double lowlat = wlat - window;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (sorted_lat[mid] < lowlat)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            a = lo;
            hi = m;
            const double highlat = wlat + window;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (sorted_lat[mid] <= highlat)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            b = lo;
        }
        double best = radius2; // RadiusResultSet::addPoint: dist < radius
        long long best_pos = 0x7fffffffffffffffLL;
        int tie = 0;
        for (long long k = a + lane; k < b; k += 32) {
            const KdPoint s = pts[k];
            const double d0 = __dsub_rn(qx, s.x), d1 = __dsub_rn(qy, s.y), d2 = __dsub_rn(qz, s.z);
            const double dist = __dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2));
            const long long pos = s.ix + (long long)s.iy * nx;
            if (dist < best) {
                best = dist;
                best_pos = pos;
                tie = 0;
            } else if (dist == best && best_pos != 0x7fffffffffffffffLL) { // equal distances: std::sort's order is unspecified
                tie = 1;
                if (pos < best_pos)
                    best_pos = pos;
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double b2 = __shfl_xor_sync(0xffffffffu, best, o);
            const long long p2 = __shfl_xor_sync(0xffffffffu, best_pos, o);
            const int t2 = __shfl_xor_sync(0xffffffffu, tie, o);
            if (p2 != 0x7fffffffffffffffLL) {
                if (best_pos == 0x7fffffffffffffffLL || b2 < best) {
                    best = b2;
                    best_pos = p2;
                    tie = t2;
                } else if (b2 == best) {
                    tie = 1;
                    if (p2 < best_pos)
                        best_pos = p2;
                }
            }
        }
        if (lane == 0) {
            if (best_pos != 0x7fffffffffffffffLL) {
                px[t] = (double)(best_pos % nx); // :1052-1056
                py[t] = (double)(best_pos / nx);
            } else {
                px[t] = -1000.; // :1059-1060
                py[t] = -1000.;
            }
            if (tie)
                atomicAdd(ties, 1ull);
        }
    }
}

} // namespace

int coordnn_search(double* d_px, double* d_py, long long n, const double* h_lon, const double* h_lat, size_t nx, size_t ny,
                   long long* ties_out, cudaStream_t st)
{
    const long long ns = (long long)nx * (long long)ny;
    FB_REQUIRE(ns > 0 && ns < 2147483647LL, "coord_nearestneighbor: empty or too large source grid");
    double *d_lon = nullptr, *d_lat = nullptr, *d_sorted_lat = nullptr, *d_best = nullptr;
    unsigned long long *d_keys = nullptr, *d_keys2 = nullptr, *d_count = nullptr;
    int *d_vals = nullptr, *d_order = nullptr;
    SrcPoint* d_pts = nullptr;
    void* d_tmp = nullptr;
    FB_CUDA_CHECK(cudaMallocAsync(&d_lon, sizeof(double) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_lat, sizeof(double) * ns, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(d_lon, h_lon, sizeof(double) * ns, cudaMemcpyHostToDevice, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(d_lat, h_lat, sizeof(double) * ns, cudaMemcpyHostToDevice, st));

    // ---- ROI: getGridDistance (:1064-1125)
    int steps;
    long long step;
    if (ns > 1000) {
        steps = 53;
        step = ns / steps;
    } else {
        step = 1;
        steps = (int)ns;
    }
    FB_CUDA_CHECK(cudaMallocAsync(&d_best, sizeof(double) * steps, st));
    k_grid_distance<<<steps, kThreads, 0, st>>>(d_lon, d_lat, ns, step, d_best);
    count_launch();
    std::vector<double> h_best((size_t)steps);
    FB_CUDA_CHECK(cudaMemcpyAsync(h_best.data(), d_best, sizeof(double) * steps, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    double worst = 2.;
    for (double b : h_best)
        if (b < worst) // a skipped sample is 3
            worst = b;
    // no valid sample leaves worst = 2 and, as in the reference, roi = acos(2) = NaN: every target gets (-1, -1)
    double roi = std::acos(worst);
    roi *= 1.414;
    if (roi > FB_PI)
        roi = FB_PI;
    const double min_grid_cos = std::cos(roi);
    // the reference compares |dlat| with acos(min_grid_cos), not with roi itself (:1166-1167)
    const double window = std::acos(min_grid_cos);

    // ---- latitude-sorted source points
    FB_CUDA_CHECK(cudaMallocAsync(&d_keys, sizeof(unsigned long long) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_keys2, sizeof(unsigned long long) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_vals, sizeof(int) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_order, sizeof(int) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_count, sizeof(unsigned long long), st));
    FB_CUDA_CHECK(cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), st));
    const int blocks = (int)std::min<long long>((ns + kThreads - 1) / kThreads, (long long)sm_count() * 32);
    k_nn_keys<<<blocks, kThreads, 0, st>>>(d_lon, d_lat, (int)nx, (int)ny, d_keys, d_vals);
    k_count_valid<<<blocks, kThreads, 0, st>>>(d_lon, d_lat, ns, d_count);
    count_launch(2);
    size_t tmp_bytes = 0;
    FB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys2, d_vals, d_order, (int)ns, 0, 64, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_tmp, tmp_bytes ? tmp_bytes : 16, st));
    FB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys2, d_vals, d_order, (int)ns, 0, 64, st));
    count_launch(8);
    unsigned long long m = 0;
    FB_CUDA_CHECK(cudaMemcpyAsync(&m, d_count, sizeof(m), cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_pts, sizeof(SrcPoint) * (m ? m : 1), st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_sorted_lat, sizeof(double) * (m ? m : 1), st));
    if (m > 0) {
        k_nn_points<<<blocks, kThreads, 0, st>>>(d_lon, d_lat, (int)nx, (int)ny, d_order, (long long)m, d_pts, d_sorted_lat);
        count_launch();
    }

    // ---- search
    unsigned long long* d_ties = d_count;
    FB_CUDA_CHECK(cudaMemsetAsync(d_ties, 0, sizeof(unsigned long long), st));
    if (n > 0) {
        const long long warps_needed = n;
        long long nb = (warps_needed * 32 + kThreads - 1) / kThreads;
        nb = std::min<long long>(nb, (long long)sm_count() * 64);
        k_nn_search<<<(int)nb, kThreads, 0, st>>>(d_px, d_py, n, d_pts, d_sorted_lat, (long long)m, min_grid_cos, window, d_ties);
        count_launch();
    }
    FB_CUDA_CHECK(cudaGetLastError());
    unsigned long long ties = 0;
    FB_CUDA_CHECK(cudaMemcpyAsync(&ties, d_ties, sizeof(ties), cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    if (ties_out)
        *ties_out = (long long)ties;
    cudaFreeAsync(d_lon, st);
    cudaFreeAsync(d_lat, st);
    cudaFreeAsync(d_best, st);
    cudaFreeAsync(d_keys, st);
    cudaFreeAsync(d_keys2, st);
    cudaFreeAsync(d_vals, st);
    cudaFreeAsync(d_order, st);
    cudaFreeAsync(d_count, st);
    cudaFreeAsync(d_tmp, st);
    cudaFreeAsync(d_pts, st);
    cudaFreeAsync(d_sorted_lat, st);
    return FB_OK;
}

// coord_kdtree: d_px / d_py hold target lon / lat in radians on entry and source (ix, iy) or (-1000, -1000) on return.
// max_dist_m: the reference's getMaxDistanceOfInterest (metres); *ties_out counts targets with two equally near sources.
int coordkd_search(double* d_px, double* d_py, long long n, const double* h_lon, const double* h_lat, size_t nx, size_t ny, double max_dist_m,
                   long long* ties_out, cudaStream_t st)
{
    const long long ns = (long long)nx * (long long)ny;
    FB_REQUIRE(ns > 0 && ns < 2147483647LL, "coord_kdtree: empty or too large source grid");
    FB_REQUIRE(max_dist_m > 0., "coord_kdtree: the distance of interest must be positive");
    const double r = max_dist_m / 6371000.; // MIFI_EARTH_RADIUS_M, CDMInterpolator.cc:1001
    const double radius2 = r * r;           // :1033
    // points whose chord is shorter than r lie within the angle 2 asin(r / 2) (plus rounding slack) in latitude
    const double window = (r >= 2. ? FB_PI : 2. * std::asin(r / 2.)) * (1. + 1e-9) + 1e-12;
    double *d_lon = nullptr, *d_lat = nullptr, *d_sorted_lat = nullptr;
    unsigned long long *d_keys = nullptr, *d_keys2 = nullptr, *d_count = nullptr;
    int *d_vals = nullptr, *d_order = nullptr;
    KdPoint* d_pts = nullptr;
    void* d_tmp = nullptr;
    FB_CUDA_CHECK(cudaMallocAsync(&d_lon, sizeof(double) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_lat, sizeof(double) * ns, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(d_lon, h_lon, sizeof(double) * ns, cudaMemcpyHostToDevice, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(d_lat, h_lat, sizeof(double) * ns, cudaMemcpyHostToDevice, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_keys, sizeof(unsigned long long) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_keys2, sizeof(unsigned long long) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_vals, sizeof(int) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_order, sizeof(int) * ns, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_count, sizeof(unsigned long long), st));
    FB_CUDA_CHECK(cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), st));
    const int blocks = (int)std::min<long long>((ns + kThreads - 1) / kThreads, (long long)sm_count() * 32);
    k_nn_keys<<<blocks, kThreads, 0, st>>>(d_lon, d_lat, (int)nx, (int)ny, d_keys, d_vals);
    k_count_valid<<<blocks, kThreads, 0, st>>>(d_lon, d_lat, ns, d_count);
    count_launch(2);
    size_t tmp_bytes = 0;
    FB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys2, d_vals, d_order, (int)ns, 0, 64, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_tmp, tmp_bytes ? tmp_bytes : 16, st));
    FB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys2, d_vals, d_order, (int)ns, 0, 64, st));
    count_launch(8);
    unsigned long long m = 0;
    FB_CUDA_CHECK(cudaMemcpyAsync(&m, d_count, sizeof(m), cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_pts, sizeof(KdPoint) * (m ? m : 1), st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_sorted_lat, sizeof(double) * (m ? m : 1), st));
    if (m > 0) {
        k_kd_points<<<blocks, kThreads, 0, st>>>(d_lon, d_lat, (int)nx, (int)ny, d_order, (long long)m, d_pts, d_sorted_lat);
        count_launch();
    }
    unsigned long long* d_ties = d_count;
    FB_CUDA_CHECK(cudaMemsetAsync(d_ties, 0, sizeof(unsigned long long), st));
    if (n > 0) {
        long long nb = (n * 32 + kThreads - 1) / kThreads;
        nb = std::min<long long>(nb, (long long)sm_count() * 64);
        k_kd_search<<<(int)nb, kThreads, 0, st>>>(d_px, d_py, n, d_pts, d_sorted_lat, (long long)m, radius2, window, (int)nx, d_ties);
        count_launch();
    }
    FB_CUDA_CHECK(cudaGetLastError());
    unsigned long long ties = 0;
    FB_CUDA_CHECK(cudaMemcpyAsync(&ties, d_ties, sizeof(ties), cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    if (ties_out)
        *ties_out = (long long)ties;
    cudaFreeAsync(d_lon, st);
    cudaFreeAsync(d_lat, st);
    cudaFreeAsync(d_keys, st);
    cudaFreeAsync(d_keys2, st);
    cudaFreeAsync(d_vals, st);
    cudaFreeAsync(d_order, st);
    cudaFreeAsync(d_count, st);
    cudaFreeAsync(d_tmp, st);
    cudaFreeAsync(d_pts, st);
    cudaFreeAsync(d_sorted_lat, st);
    return FB_OK;
}

} // namespace fb
