// fimex_b200/csrc/merge_kernels.cu -- the per-value parts of CDMMerger around its three gathers: the crop of a source slab to a
// handle's reduced domain (fused with the type adapter of the gather's input), the linear border smoothing of the inner grid
// (CDMBorderSmoothing::getDataSlice + CDMBorderSmoothing_Linear) and the overlay on the target grid (CDMOverlay::getDataSlice).
//
// Arithmetic (DESIGN.md section 2): for cell (x, y) of the nx x ny inner grid, transition width t, border width b,
//   xmin1 = b, xmax1 = b + t, xmax2 = nx - b, xmin2 = xmax2 - t (same for y)
//   dx = x < xmax1 ? xmax1 - x : (x >= xmin2 ? x - xmin2 : 0) (same for dy)
//   alpha = min(max(sqrt(dx dx + dy dy) / t, 0), 1) in fp64
//   outside the border: the outer value; inside the interior: the inner value; between: vi + alpha (vo - vi) in fp64 with the
//   product never contracted into an FMA (vo where vo - vi == 0); vo undefined: vi; vi undefined: vo or NaN.
// The inner value enters in fp64 (not rounded to float first), the result is rounded to float once: the inner -> target gather
// would round it there anyway.  All three kernels are bound by HBM bandwidth; none of them does more than a few flops a byte.
#include "kernels.h"

namespace fb {
namespace {

constexpr int kThreads = 256;

// [nz][ny][nx] of IN -> the window [x0, x0 + w) x [y0, y0 + h) of every level as float, badValue -> NaN (data2InterpolationArray)
template <class IN>
__global__ void __launch_bounds__(kThreads) k_crop_as_float(const IN* __restrict__ in, long long nx, long long ny, long long x0, long long y0, long long w,
                                                            long long h, long long n, int has_bad, float bad, float* __restrict__ out)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long x = i % w, r = i / w;
        const long long y = r % h, z = r / h;
        out[i] = load_as_float<IN>(__ldg(in + (z * ny + y0 + y) * nx + x0 + x), has_bad != 0, bad);
    }
}

// One thread per cell (x, y) of the window [x0, x0 + w) x [y0, y0 + h) of the inner grid that the inner -> target gather reads:
// alpha and the zone once, then the levels [blockIdx.y * zseg, +zseg).  inner [nz][ny][nx] of IN (bad: the fill value in IN),
// outer [nz][ny][nx] float (the outer -> inner gather), out [nz][h][w] float.
template <class IN>
__global__ void __launch_bounds__(kThreads) k_border_smooth_linear(const IN* __restrict__ inner, int has_bad, IN bad, const float* __restrict__ outer,
                                                                   long long nx, long long ny, long long t, long long b, int use_outer, long long x0,
                                                                   long long y0, long long w, long long h, long long nz, long long zseg,
                                                                   float* __restrict__ out)
{
    const long long cell = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (cell >= w * h)
        return;
    const long long wx = cell % w, wy = cell / w;
    const long long x = x0 + wx, y = y0 + wy;
    const long long xmin1 = b, xmax1 = b + t, xmax2 = nx - b, xmin2 = xmax2 - t;
    const long long ymin1 = b, ymax1 = b + t, ymax2 = ny - b, ymin2 = ymax2 - t;
    const double dx = x < xmax1 ? (double)(xmax1 - x) : (x >= xmin2 ? (double)(x - xmin2) : 0.);
    const double dy = y < ymax1 ? (double)(ymax1 - y) : (y >= ymin2 ? (double)(y - ymin2) : 0.);
    const double alpha = fmin(fmax(__ddiv_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))), (double)t), 0.), 1.);
    const bool outside = x < xmin1 || x >= xmax2 || y < ymin1 || y >= ymax2;
    const bool inside = x >= xmax1 && x < xmin2 && y >= ymax1 && y < ymin2;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    const long long z0 = blockIdx.y * zseg, z1 = min(nz, z0 + zseg);
    for (long long z = z0; z < z1; ++z) {
        const long long src = (z * ny + y) * nx + x;
        const IN raw = __ldg(inner + src);
        const double vi = (has_bad && raw == bad) ? qnan : (double)raw;
        const double vo = (double)__ldg(outer + src);
        double m;
        if (outside) {
            m = vo;
        } else if (inside) {
            m = vi;
        } else {
            const double d = __dsub_rn(vo, vi);
            m = d == 0. ? vo : __dadd_rn(vi, __dmul_rn(alpha, d));
        }
        if (isnan(vo))
            m = vi;
        if (isnan(vi))
            m = use_outer ? vo : qnan;
        __stcs(out + (z * h + wy) * w + wx, (float)m);
    }
}

// out = top where it is defined, else base; NaN -> fill, round + cast (interpolationArray2Data).  Four values per thread, with
// one 16-byte load per input and one store when vec (n % 4 == 0, out aligned to four elements; the inputs are scratch buffers).
template <class OUT>
__global__ void __launch_bounds__(kThreads) k_merge_overlay(const float* __restrict__ top, const float* __restrict__ base, long long n, bool vec,
                                                            StoreAs<OUT> conv, OUT* __restrict__ out)
{
    const long long e0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * 4;
    if (e0 >= n)
        return;
    if (vec) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(top + e0));
        const float4 c = __ldcs(reinterpret_cast<const float4*>(base + e0));
        store_vec4<OUT>(out + e0, conv(isnan(a.x) ? c.x : a.x), conv(isnan(a.y) ? c.y : a.y), conv(isnan(a.z) ? c.z : a.z),
                        conv(isnan(a.w) ? c.w : a.w));
        return;
    }
    const int m = (int)min(4LL, n - e0);
    for (int i = 0; i < m; ++i) {
        const float a = top[e0 + i];
        __stcs(out + e0 + i, conv(isnan(a) ? base[e0 + i] : a));
    }
}

unsigned blocks_for(long long n)
{
    const long long b = (n + kThreads - 1) / kThreads;
    const long long cap = (long long)sm_count() * 32;
    return (unsigned)(b < cap ? (b < 1 ? 1 : b) : cap);
}

template <class IN>
int crop_typed(const void* d_in, long long nx, long long ny, long long x0, long long y0, long long w, long long h, long long nz, bool has_bad, float bad,
               float* d_out, cudaStream_t st)
{
    const long long n = w * h * nz;
    k_crop_as_float<IN><<<blocks_for(n), kThreads, 0, st>>>(static_cast<const IN*>(d_in), nx, ny, x0, y0, w, h, n, has_bad ? 1 : 0, bad, d_out);
    count_launch();
    FB_CUDA_CHECK(cudaGetLastError());
    return FB_OK;
}

template <class IN>
int smooth_typed(const void* d_inner, bool has_bad, double bad, const float* d_outer, long long nx, long long ny, int t, int b, bool use_outer, long long x0,
                 long long y0, long long w, long long h, long long nz, float* d_out, cudaStream_t st)
{
    const long long bx = (w * h + kThreads - 1) / kThreads;
    FB_REQUIRE(bx <= 0x7fffffffLL, "border smoothing: inner grid too large");
    // few cells: split the levels over gridDim.y until about eight blocks per multiprocessor are in flight
    const long long want = (long long)sm_count() * 8;
    long long segs = bx >= want ? 1 : (want + bx - 1) / bx;
    if (segs > nz)
        segs = nz;
    const long long zseg = (nz + segs - 1) / segs;
    const long long gy = (nz + zseg - 1) / zseg;
    k_border_smooth_linear<IN><<<dim3((unsigned)bx, (unsigned)gy), kThreads, 0, st>>>(static_cast<const IN*>(d_inner), has_bad ? 1 : 0,
                                                                                      has_bad ? cast_fill<IN>(bad) : IN(0), d_outer, nx, ny, t, b,
                                                                                      use_outer ? 1 : 0, x0, y0, w, h, nz, zseg, d_out);
    count_launch();
    FB_CUDA_CHECK(cudaGetLastError());
    return FB_OK;
}

template <class OUT>
int overlay_typed(const float* d_top, const float* d_base, long long n, double fill, void* d_out, cudaStream_t st)
{
    const bool vec = n % 4 == 0 && reinterpret_cast<uintptr_t>(d_out) % (4 * sizeof(OUT)) == 0 && reinterpret_cast<uintptr_t>(d_top) % 16 == 0 &&
                     reinterpret_cast<uintptr_t>(d_base) % 16 == 0;
    const long long threads = (n + 3) / 4;
    const long long bx = (threads + kThreads - 1) / kThreads;
    FB_REQUIRE(bx <= 0x7fffffffLL, "merge overlay: too many values");
    k_merge_overlay<OUT><<<(unsigned)bx, kThreads, 0, st>>>(d_top, d_base, n, vec, StoreAs<OUT>{cast_fill<OUT>(fill)}, static_cast<OUT*>(d_out));
    count_launch();
    FB_CUDA_CHECK(cudaGetLastError());
    return FB_OK;
}

} // namespace

#define FB_ALL_TYPES(MACRO)                                                                                                                \
    MACRO(FB_T_CHAR, signed char)                                                                                                          \
    MACRO(FB_T_SHORT, short)                                                                                                               \
    MACRO(FB_T_INT, int)                                                                                                                   \
    MACRO(FB_T_FLOAT, float)                                                                                                               \
    MACRO(FB_T_DOUBLE, double)                                                                                                             \
    MACRO(FB_T_UCHAR, unsigned char)                                                                                                       \
    MACRO(FB_T_USHORT, unsigned short)                                                                                                     \
    MACRO(FB_T_UINT, unsigned int)                                                                                                         \
    MACRO(FB_T_INT64, long long)                                                                                                           \
    MACRO(FB_T_UINT64, unsigned long long)

int launch_crop_as_float(int in_type, const void* d_in, long long nx, long long ny, long long x0, long long y0, long long w, long long h, long long nz,
                         bool has_bad, float bad, float* d_out, cudaStream_t st)
{
    if (w * h * nz == 0)
        return FB_OK;
    switch (in_type) {
#define FB_CASE(TAG, T)                                                                                                                    \
    case TAG:                                                                                                                              \
        return crop_typed<T>(d_in, nx, ny, x0, y0, w, h, nz, has_bad, bad, d_out, st);
        FB_ALL_TYPES(FB_CASE)
#undef FB_CASE
    default:
        FB_REQUIRE(false, "unsupported input data type " + std::to_string(in_type));
    }
}

int launch_border_smooth_linear(int in_type, const void* d_inner, bool has_bad, double bad, const float* d_outer, long long nx, long long ny, int t, int b,
                                bool use_outer, long long x0, long long y0, long long w, long long h, long long nz, float* d_out, cudaStream_t st)
{
    if (w * h * nz == 0)
        return FB_OK;
    switch (in_type) {
#define FB_CASE(TAG, T)                                                                                                                    \
    case TAG:                                                                                                                              \
        return smooth_typed<T>(d_inner, has_bad, bad, d_outer, nx, ny, t, b, use_outer, x0, y0, w, h, nz, d_out, st);
        FB_ALL_TYPES(FB_CASE)
#undef FB_CASE
    default:
        FB_REQUIRE(false, "unsupported input data type " + std::to_string(in_type));
    }
}

int launch_merge_overlay(const float* d_top, const float* d_base, long long n, int out_type, double fill, void* d_out, cudaStream_t st)
{
    if (n == 0)
        return FB_OK;
    switch (out_type) {
#define FB_CASE(TAG, T)                                                                                                                    \
    case TAG:                                                                                                                              \
        return overlay_typed<T>(d_top, d_base, n, fill, d_out, st);
        FB_ALL_TYPES(FB_CASE)
#undef FB_CASE
    default:
        FB_REQUIRE(false, "unsupported output data type " + std::to_string(out_type));
    }
}

#undef FB_ALL_TYPES

} // namespace fb
