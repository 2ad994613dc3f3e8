// fimex_b200/csrc/time_kernels.cu -- time interpolation (the linear change of the time axis of CDMTimeInterpolator): a device
// stack of source steps in [T][n] -> out [J][n], every source step the targets need read from HBM once per call.
//
// The handle keeps the targets sorted by their bracket (TimeStep: lower source step, output row, weight), so the brackets a thread
// walks never go down.  A thread owns four consecutive elements and keeps the current bracket's A and B in registers; when the
// bracket moves up by one, the old B becomes the new A, and only a jump loads both.  Arithmetic (DESIGN.md section 2):
// r = (float)((double)A + w * ((double)B - (double)A)) with the product through __dmul_rn, so that it is never contracted into
// an FMA (the two-level step of the vertical kernels and of orc_vint_value).  The type adapters of (1c) are fused into the loads
// (any CDM type -> float, badValue -> NaN) and the stores (NaN -> fill, round + cast), so no float copy of the stack is written.
#include "kernels.h"

namespace fb {
namespace {

constexpr int kThreads = 256;
constexpr int kVec = 4; // elements per thread

// four consecutive values from p (aligned to 4 * sizeof(T)) with one non-coherent load (two for 8-byte types)
template <class T>
__device__ __forceinline__ void load_vec4(const T* p, T v[kVec])
{
    if constexpr (sizeof(T) == 1) {
        union {
            unsigned u;
            T t[4];
        } w;
        w.u = __ldg(reinterpret_cast<const unsigned*>(p));
        for (int i = 0; i < kVec; ++i)
            v[i] = w.t[i];
    } else if constexpr (sizeof(T) == 2) {
        union {
            uint2 u;
            T t[4];
        } w;
        w.u = __ldg(reinterpret_cast<const uint2*>(p));
        for (int i = 0; i < kVec; ++i)
            v[i] = w.t[i];
    } else if constexpr (sizeof(T) == 4) {
        union {
            uint4 u;
            T t[4];
        } w;
        w.u = __ldg(reinterpret_cast<const uint4*>(p));
        for (int i = 0; i < kVec; ++i)
            v[i] = w.t[i];
    } else {
        union {
            uint4 u[2];
            T t[4];
        } w;
        w.u[0] = __ldg(reinterpret_cast<const uint4*>(p));
        w.u[1] = __ldg(reinterpret_cast<const uint4*>(p) + 1);
        for (int i = 0; i < kVec; ++i)
            v[i] = w.t[i];
    }
}

// blockIdx.y: a contiguous segment of the sorted targets [s0, s1); every segment starts with its own first bracket.
// in_b != nullptr: a two-step call, step 0 at `in` and step 1 at `in_b` (the step pointers of fb200_tinterp_get_step_device);
// otherwise step k is at in + k * n.  vec: n % 4 == 0 and every pointer aligned to four elements; else scalar loads and stores.
template <class IN, class OUT>
__global__ void __launch_bounds__(kThreads, 4) k_tinterp(const IN* __restrict__ in, const IN* __restrict__ in_b, long long n, int has_bad, float bad,
                                                      const TimeStep* __restrict__ tab, int nj, int seg, bool vec, StoreAs<OUT> conv,
                                                      OUT* __restrict__ out)
{
    const long long e0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * kVec;
    if (e0 >= n)
        return;
    const int s0 = blockIdx.y * seg;
    const int s1 = min(nj, s0 + seg);
    const int m = (int)min((long long)kVec, n - e0);
    auto step = [&](int k) { return (k == 1 && in_b) ? in_b : in + (long long)k * n; };
    auto load = [&](int k, float f[kVec]) {
        const IN* p = step(k) + e0;
        IN v[kVec];
        if (vec) {
            load_vec4<IN>(p, v);
        } else {
            for (int i = 0; i < kVec; ++i)
                v[i] = i < m ? __ldg(p + i) : IN(0);
        }
        for (int i = 0; i < kVec; ++i)
            f[i] = load_as_float<IN>(v[i], has_bad != 0, bad);
    };
    float A[kVec], B[kVec];
    int cur = -2; // the lower source step of the bracket held in A, B (none yet)
    for (int s = s0; s < s1; ++s) {
        const TimeStep ts = tab[s];
        OUT r[kVec];
        if (ts.ia < 0) { // no bracket: NaN, stored as the fill value
            for (int i = 0; i < kVec; ++i)
                r[i] = conv(undef_f());
        } else {
            if (ts.ia == cur + 1) {
                for (int i = 0; i < kVec; ++i)
                    A[i] = B[i];
                load(ts.ia + 1, B);
            } else if (ts.ia != cur) {
                load(ts.ia, A);
                load(ts.ia + 1, B);
            }
            cur = ts.ia;
            for (int i = 0; i < kVec; ++i)
                r[i] = conv((float)((double)A[i] + __dmul_rn(ts.w, (double)B[i] - (double)A[i])));
        }
        OUT* o = out + (long long)ts.row * n + e0;
        if (vec) {
            store_vec4<OUT>(o, r[0], r[1], r[2], r[3]);
        } else {
#pragma unroll
            for (int i = 0; i < kVec; ++i)
                if (i < m)
                    __stcs(o + i, r[i]);
        }
    }
}

template <class T>
bool aligned4(const void* p)
{
    return p == nullptr || reinterpret_cast<uintptr_t>(p) % (kVec * sizeof(T)) == 0;
}

template <class IN, class OUT>
int launch_typed(const void* d_in, const void* d_in_b, long long n, bool has_bad, float bad, const TimeStep* d_tab, int nj, double fill, void* d_out,
                 cudaStream_t st)
{
    const bool vec = n % kVec == 0 && aligned4<IN>(d_in) && aligned4<IN>(d_in_b) && aligned4<OUT>(d_out);
    const long long threads = (n + kVec - 1) / kVec;
    const long long bx = (threads + kThreads - 1) / kThreads;
    FB_REQUIRE(bx <= 0x7fffffffLL, "time interpolation: too many elements per step");
    // small n: split the sorted targets over gridDim.y until about eight blocks per multiprocessor are in flight
    const long long want = (long long)sm_count() * 8;
    long long segs = bx >= want ? 1 : (want + bx - 1) / bx;
    if (segs > nj)
        segs = nj;
    const int seg = (int)((nj + segs - 1) / segs);
    const int gy = (nj + seg - 1) / seg;
    k_tinterp<IN, OUT><<<dim3((unsigned)bx, (unsigned)gy), kThreads, 0, st>>>(static_cast<const IN*>(d_in), static_cast<const IN*>(d_in_b), n,
                                                                              has_bad ? 1 : 0, bad, d_tab, nj, seg, vec,
                                                                              StoreAs<OUT>{cast_fill<OUT>(fill)}, static_cast<OUT*>(d_out));
    count_launch();
    FB_CUDA_CHECK(cudaGetLastError());
    return FB_OK;
}

template <class IN>
int launch_out(int out_type, const void* d_in, const void* d_in_b, long long n, bool has_bad, float bad, const TimeStep* d_tab, int nj, double fill,
               void* d_out, cudaStream_t st)
{
    switch (out_type) {
#define FB_CASE(TAG, T)                                                                                                                    \
    case TAG:                                                                                                                              \
        return launch_typed<IN, T>(d_in, d_in_b, n, has_bad, bad, d_tab, nj, fill, d_out, st);
        FB_CASE(FB_T_CHAR, signed char)
        FB_CASE(FB_T_SHORT, short)
        FB_CASE(FB_T_INT, int)
        FB_CASE(FB_T_FLOAT, float)
        FB_CASE(FB_T_DOUBLE, double)
        FB_CASE(FB_T_UCHAR, unsigned char)
        FB_CASE(FB_T_USHORT, unsigned short)
        FB_CASE(FB_T_UINT, unsigned int)
        FB_CASE(FB_T_INT64, long long)
        FB_CASE(FB_T_UINT64, unsigned long long)
#undef FB_CASE
    default:
        FB_REQUIRE(false, "unsupported output data type " + std::to_string(out_type));
    }
}

} // namespace

int launch_tinterp(int in_type, const void* d_in, const void* d_in_b, long long n, bool has_bad, float bad, const TimeStep* d_tab, int nj, int out_type,
                   double fill, void* d_out, cudaStream_t st)
{
    if (n == 0 || nj == 0)
        return FB_OK;
    switch (in_type) {
#define FB_CASE(TAG, T)                                                                                                                    \
    case TAG:                                                                                                                              \
        return launch_out<T>(out_type, d_in, d_in_b, n, has_bad, bad, d_tab, nj, fill, d_out, st);
        FB_CASE(FB_T_CHAR, signed char)
        FB_CASE(FB_T_SHORT, short)
        FB_CASE(FB_T_INT, int)
        FB_CASE(FB_T_FLOAT, float)
        FB_CASE(FB_T_DOUBLE, double)
        FB_CASE(FB_T_UCHAR, unsigned char)
        FB_CASE(FB_T_USHORT, unsigned short)
        FB_CASE(FB_T_UINT, unsigned int)
        FB_CASE(FB_T_INT64, long long)
        FB_CASE(FB_T_UINT64, unsigned long long)
#undef FB_CASE
    default:
        FB_REQUIRE(false, "unsupported input data type " + std::to_string(in_type));
    }
}

} // namespace fb
