// fimex_b200/csrc/forward_kernels.cu -- K8: forward ("scatter") interpolation as sort-then-segment.
//
// Replaces CachedForwardInterpolation::interpolateValues
// (/root/reference/src/CachedForwardInterpolation.cc:92-131, aggregators :38-59).  The reference pushes
// every defined input value into a std::vector per target cell, in input (row-major) order, then
// aggregates each vector.  Here the bucketing is done ONCE per grid: input indices are stably sorted by
// target cell (CSR: `perm` + `offsets`), and each slice runs one segmented-reduce kernel in which a thread
// walks its cell's segment in ascending input order -- the same order as the reference's vectors, so the
// sequential fp32 sum of forward_mean/forward_sum is bit-identical; max/min are order-free.
//
// Per level: reads 4 B per input value + 4 B per perm entry + 4 B per cell offset, writes 4 B per cell.
// The one-time stable sort uses cub::DeviceRadixSort (CUDA toolkit); the per-slice kernel is hand-written.
#include "kernels.h"

#include <cub/device/device_radix_sort.cuh>

namespace fb {

namespace {
constexpr int kThreads = 256;

__global__ void k_forward_keys(const int* __restrict__ cell, long long n, unsigned n_cells, unsigned* __restrict__ keys,
                               int* __restrict__ vals)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int c = cell[i];
        keys[i] = c >= 0 ? (unsigned)c : n_cells; // unmapped points sort behind every cell
        vals[i] = (int)i;
    }
}

// offsets[c] = first position in the sorted keys whose key >= c  (c in [0, n_cells])
__global__ void k_forward_offsets(const unsigned* __restrict__ sorted_keys, long long n, long long n_cells, int* __restrict__ offsets)
{
    for (long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x; c <= n_cells; c += (long long)gridDim.x * blockDim.x) {
        long long lo = 0, hi = n;
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (sorted_keys[mid] < (unsigned)c)
                lo = mid + 1;
            else
                hi = mid;
        }
        offsets[c] = (int)lo;
    }
}

enum { AG_SUM = 0, AG_MEAN = 1, AG_MEDIAN = 2, AG_MAX = 3, AG_MIN = 4 };

#ifndef FB_FWD_CELLS
#define FB_FWD_CELLS 4
#endif
constexpr int kCells = FB_FWD_CELLS; // target cells per thread: their first gathers are issued together (the kernel is bound by the
                          // dependent chain offsets -> permutation -> value, not by bandwidth).  Measured and rejected (round 2, config 5):
                          // a second table with the first input index of every cell, read next to the offsets, shortens the chain to
                          // two loads but adds 72 MB of table traffic per slice: 0.093 ms instead of 0.081 (mean), 0.090 / 0.078 (max)

// std::nth_element(first, first + nth, first + n) with operator<, restated from libstdc++ (bits/stl_algo.h __introselect and its
// helpers, bits/stl_heap.h); the same comparisons and moves as oracle/mifi_oracle.c's orc_nth_element.  Only segments whose result
// depends on the algorithm come here (NaN, or both signs of zero): one thread works through its own copy of the segment.
namespace nth {
__device__ __forceinline__ void swapf(float* a, float* b)
{
    const float t = *a;
    *a = *b;
    *b = t;
}

__device__ void push_heap(float* v, long long hole, long long top, float value)
{
    long long parent = (hole - 1) / 2;
    while (hole > top && v[parent] < value) {
        v[hole] = v[parent];
        hole = parent;
        parent = (hole - 1) / 2;
    }
    v[hole] = value;
}

__device__ void adjust_heap(float* v, long long hole, long long len, float value)
{
    const long long top = hole;
    long long child = hole;
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
    push_heap(v, hole, top, value);
}

__device__ void heap_select(float* first, float* middle, float* last)
{
    const long long len = middle - first;
    if (len >= 2) {
        for (long long parent = (len - 2) / 2;; parent--) {
            adjust_heap(first, parent, len, first[parent]);
            if (parent == 0)
                break;
        }
    }
    for (float* i = middle; i < last; ++i)
        if (*i < *first) {
            const float value = *i;
            *i = *first;
            adjust_heap(first, 0, len, value);
        }
}

__device__ void insertion_sort(float* first, float* last)
{
    if (first == last)
        return;
    for (float* i = first + 1; i != last; ++i) {
        const float val = *i;
        if (val < *first) {
            for (float* p = i; p != first; --p)
                *p = *(p - 1);
            *first = val;
        } else {
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

__device__ void move_median_to_first(float* result, float* a, float* b, float* c)
{
    if (*a < *b) {
        if (*b < *c)
            swapf(result, b);
        else if (*a < *c)
            swapf(result, c);
        else
            swapf(result, a);
    } else if (*a < *c)
        swapf(result, a);
    else if (*b < *c)
        swapf(result, c);
    else
        swapf(result, b);
}

__device__ float* unguarded_partition_pivot(float* first, float* last)
{
    float* mid = first + (last - first) / 2;
    move_median_to_first(first, first + 1, mid, last - 1);
    float* lo = first + 1;
    float* hi = last;
    for (;;) {
        while (*lo < *first)
            ++lo;
        --hi;
        while (*first < *hi)
            --hi;
        if (!(lo < hi))
            return lo;
        swapf(lo, hi);
        ++lo;
    }
}

__device__ void nth_element(float* first, long long nth_index, long long n)
{
    float* last = first + n;
    float* nth = first + nth_index;
    if (first == last || nth == last)
        return;
    int depth_limit = 0; // std::__lg(n) * 2
    for (long long m = n; m > 1; m >>= 1)
        depth_limit += 2;
    while (last - first > 3) {
        if (depth_limit == 0) {
            heap_select(first, nth + 1, last);
            swapf(first, nth);
            return;
        }
        --depth_limit;
        float* cut = unguarded_partition_pivot(first, last);
        if (cut <= nth)
            first = cut;
        else
            last = cut;
    }
    insertion_sort(first, last);
}
} // namespace nth

// one target cell: aggregate its CSR segment [beg, end) in ascending input order; v0 = value of the first entry (prefetched).
// scr (median only): this level's scratch, one float per mapped point; the cell may use scr[beg, end).
template <int AGG, bool UNDEF>
__device__ __forceinline__ float aggregate_cell(const float* __restrict__ lv, const int* __restrict__ perm, int beg, int end, float v0,
                                                float* __restrict__ scr)
{
    float res = undef_f();
    if (beg >= end)
        return res;
    if (AGG == AG_SUM || AGG == AG_MEAN) {
        float s = 0.f; // std::accumulate(begin, end, 0.f): sequential, input order
        long long cnt = 0;
        if (UNDEF || !isnan(v0)) {
            s = __fadd_rn(s, v0);
            ++cnt;
        }
        for (int k = beg + 1; k < end; ++k) {
            const float v = __ldg(lv + __ldg(perm + k));
            if (UNDEF || !isnan(v)) {
                s = __fadd_rn(s, v);
                ++cnt;
            }
        }
        if (cnt > 0)
            res = (AGG == AG_MEAN) ? __fdiv_rn(s, __ll2float_rn(cnt)) : s;
    } else if (AGG == AG_MAX || AGG == AG_MIN) {
        bool have = false;
        float best = 0.f;
        if (UNDEF || !isnan(v0)) {
            best = v0;
            have = true;
        }
        for (int k = beg + 1; k < end; ++k) {
            const float v = __ldg(lv + __ldg(perm + k));
            if (UNDEF || !isnan(v)) {
                if (!have) {
                    best = v;
                    have = true;
                } else if (AGG == AG_MAX ? (best < v) : (v < best)) { // std::max_element / min_element
                    best = v;
                }
            }
        }
        if (have)
            res = best;
    } else { // median = v[n/2] after nth_element(v.begin(), v.begin() + n/2, v.end()) (:49-53)
        long long cnt = 0;
        bool has_nan = false, has_pz = false, has_nz = false;
        for (int k = beg; k < end; ++k) {
            const float v = __ldg(lv + __ldg(perm + k));
            if (UNDEF || !isnan(v)) {
                ++cnt;
                has_nan |= isnan(v);
                has_pz |= (v == 0.f && !signbit(v));
                has_nz |= (v == 0.f && signbit(v));
            }
        }
        if (has_nan || (has_pz && has_nz)) { // < is no strict weak order here, or equal elements differ in their bits
            long long m = 0;
            for (int k = beg; k < end; ++k) {
                const float v = __ldg(lv + __ldg(perm + k));
                if (UNDEF || !isnan(v))
                    scr[beg + m++] = v;
            }
            nth::nth_element(scr + beg, cnt / 2, cnt);
            res = scr[beg + cnt / 2];
        } else if (cnt > 0) { // every element equal to the median has the same bits: rank selection, O(n^2) but segments are short
            const long long want = cnt / 2;
            for (int k = beg; k < end; ++k) {
                const float v = __ldg(lv + __ldg(perm + k));
                if (!(UNDEF || !isnan(v)))
                    continue;
                long long less = 0, eq = 0;
                for (int j = beg; j < end; ++j) {
                    const float w = __ldg(lv + __ldg(perm + j));
                    if (!(UNDEF || !isnan(w)))
                        continue;
                    less += (w < v);
                    eq += (w == v);
                }
                if (less <= want && want < less + eq) {
                    res = v;
                    break;
                }
            }
        }
    }
    return res;
}

// ZL levels of one target cell at a time (sum / mean / max / min): the permutation entry of every segment element is read ONCE
// and its ZL values -- independent gathers, one per level -- are in flight together; every level keeps its own sequential
// accumulator, so each level's result is exactly what aggregate_cell gives for it.
template <int AGG, bool UNDEF, int ZL>
__device__ __forceinline__ void aggregate_cell_levels(const float* __restrict__ lv, long long n_in, const int* __restrict__ perm, int beg, int end,
                                                      const float (&v0)[ZL], float (&res)[ZL])
{
    static_assert(AGG != AG_MEDIAN, "median goes level by level");
    float acc[ZL];
    long long cnt[ZL];
    bool have[ZL];
#pragma unroll
    for (int l = 0; l < ZL; ++l) {
        res[l] = undef_f();
        acc[l] = 0.f;
        cnt[l] = 0;
        have[l] = false;
    }
    if (beg >= end)
        return;
    auto feed = [&](int l, float v) {
        if (!(UNDEF || !isnan(v)))
            return;
        if (AGG == AG_SUM || AGG == AG_MEAN) {
            acc[l] = __fadd_rn(acc[l], v); // std::accumulate(begin, end, 0.f): sequential, input order
            ++cnt[l];
        } else if (!have[l]) {
            acc[l] = v;
            have[l] = true;
        } else if (AGG == AG_MAX ? (acc[l] < v) : (v < acc[l])) { // std::max_element / min_element
            acc[l] = v;
        }
    };
#pragma unroll
    for (int l = 0; l < ZL; ++l)
        feed(l, v0[l]);
    for (int k = beg + 1; k < end; ++k) {
        const float* p = lv + __ldg(perm + k);
        float v[ZL];
#pragma unroll
        for (int l = 0; l < ZL; ++l)
            v[l] = __ldg(p + l * n_in);
#pragma unroll
        for (int l = 0; l < ZL; ++l)
            feed(l, v[l]);
    }
#pragma unroll
    for (int l = 0; l < ZL; ++l) {
        if (AGG == AG_SUM || AGG == AG_MEAN) {
            if (cnt[l] > 0)
                res[l] = (AGG == AG_MEAN) ? __fdiv_rn(acc[l], __ll2float_rn(cnt[l])) : acc[l];
        } else if (have[l]) {
            res[l] = acc[l];
        }
    }
}

// ZL = levels per thread and pass (1 for single-level slices, 4 otherwise; the median always works level by level)
template <int AGG, bool UNDEF, int ZL>
__global__ void __launch_bounds__(kThreads) k_forward(const int* __restrict__ perm, const int* __restrict__ offsets,
                                                    const float* __restrict__ in, float* __restrict__ out, long long n_in,
                                                    long long n_cells, long long nz, int vec_ok, float* __restrict__ scratch,
                                                    long long scratch_stride)
{
    const long long c0 = (blockIdx.x * (long long)kThreads + threadIdx.x) * kCells;
    if (c0 >= n_cells)
        return;
    int off[kCells + 1], first[kCells];
    if (c0 + kCells <= n_cells) { // offsets[c0 .. c0+3] in one 128-bit load (c0 is a multiple of 4, cudaMalloc aligns the array)
#pragma unroll
        for (int q = 0; q < kCells / 4; ++q) {
            const int4 o4 = __ldg(reinterpret_cast<const int4*>(offsets + c0) + q);
            off[4 * q] = o4.x, off[4 * q + 1] = o4.y, off[4 * q + 2] = o4.z, off[4 * q + 3] = o4.w;
        }
        off[kCells] = __ldg(offsets + c0 + kCells);
    } else {
#pragma unroll
        for (int j = 0; j <= kCells; ++j)
            off[j] = __ldg(offsets + (c0 + j <= n_cells ? c0 + j : n_cells));
    }
#pragma unroll
    for (int j = 0; j < kCells; ++j)
        first[j] = off[j] < off[j + 1] ? __ldg(perm + off[j]) : -1; // the same for every level
    // the median's scratch: one slot of n_mapped floats per blockIdx.y, which works through its levels one after another
    float* scr = AGG == AG_MEDIAN ? scratch + (long long)blockIdx.y * scratch_stride : nullptr;
    const long long valid = n_cells - c0;
    auto store = [&](long long z, const float (&res)[kCells]) {
        float* o = out + z * n_cells + c0;
        if (vec_ok && valid >= kCells) {
#pragma unroll
            for (int q = 0; q < kCells / 4; ++q)
                __stcs(reinterpret_cast<float4*>(o) + q, make_float4(res[4 * q], res[4 * q + 1], res[4 * q + 2], res[4 * q + 3]));
        } else {
#pragma unroll
            for (int j = 0; j < kCells; ++j)
                if (j < valid)
                    __stcs(o + j, res[j]);
        }
    };
    for (long long z = (long long)blockIdx.y * ZL; z < nz; z += (long long)gridDim.y * ZL) {
        const float* lv = in + z * n_in;
        if (ZL > 1 && AGG != AG_MEDIAN && z + ZL <= nz) {
            float v0[kCells][ZL], res[kCells][ZL];
#pragma unroll
            for (int j = 0; j < kCells; ++j)
#pragma unroll
                for (int l = 0; l < ZL; ++l)
                    v0[j][l] = first[j] >= 0 ? __ldg(lv + l * n_in + first[j]) : 0.f; // kCells * ZL independent gathers in flight
            if (AGG != AG_MEDIAN) {
#pragma unroll
                for (int j = 0; j < kCells; ++j)
                    aggregate_cell_levels<(AGG == AG_MEDIAN ? AG_SUM : AGG), UNDEF, ZL>(lv, n_in, perm, off[j], off[j + 1], v0[j], res[j]);
            }
#pragma unroll
            for (int l = 0; l < ZL; ++l) {
                float r[kCells];
#pragma unroll
                for (int j = 0; j < kCells; ++j)
                    r[j] = res[j][l];
                store(z + l, r);
            }
            continue;
        }
        for (long long zz = z; zz < nz && zz < z + ZL; ++zz, lv += n_in) { // single levels: ZL == 1, the tail of the stack, the median
            float v0[kCells], res[kCells];
#pragma unroll
            for (int j = 0; j < kCells; ++j)
                v0[j] = first[j] >= 0 ? __ldg(lv + first[j]) : 0.f; // kCells independent gathers in flight
#pragma unroll
            for (int j = 0; j < kCells; ++j)
                res[j] = aggregate_cell<AGG, UNDEF>(lv, perm, off[j], off[j + 1], v0[j], scr);
            store(zz, res);
        }
    }
}

// the median's scratch is at most this many bytes: config 5 (10 M points) would need 2.5 GB for 64 levels at once
constexpr size_t kMedianScratchBytes = 256u << 20;

template <int AGG>
int launch_agg(bool undef, int gx, cudaStream_t st, const ForwardPlan& p, const float* in, float* out, long long nz)
{
    const int vec_ok = ((p.n_cells % 4) == 0 && (reinterpret_cast<uintptr_t>(out) & 15u) == 0) ? 1 : 0;
    if (nz >= 4 && AGG != AG_MEDIAN) { // several levels: four per thread and pass
        const long long passes = (nz + 3) / 4;
        dim3 grid(gx, (unsigned)(passes < 64 ? passes : 64));
        if (undef)
            k_forward<AGG, true, 4><<<grid, kThreads, 0, st>>>(p.d_perm, p.d_offsets, in, out, p.n_in, p.n_cells, nz, vec_ok, nullptr, 0);
        else
            k_forward<AGG, false, 4><<<grid, kThreads, 0, st>>>(p.d_perm, p.d_offsets, in, out, p.n_in, p.n_cells, nz, vec_ok, nullptr, 0);
    } else {
        long long gy = nz < 64 ? nz : 64;
        float* scratch = nullptr;
        const long long stride = p.n_mapped > 0 ? p.n_mapped : 1;
        if (AGG == AG_MEDIAN) { // one scratch slot per blockIdx.y: fewer levels at once when the slots would not fit
            const long long fit = (long long)(kMedianScratchBytes / (sizeof(float) * (size_t)stride));
            gy = gy < fit ? gy : (fit > 1 ? fit : 1);
            FB_CUDA_CHECK(cudaMallocAsync(&scratch, sizeof(float) * (size_t)(stride * gy), st));
        }
        dim3 grid(gx, (unsigned)gy);
        if (undef)
            k_forward<AGG, true, 1><<<grid, kThreads, 0, st>>>(p.d_perm, p.d_offsets, in, out, p.n_in, p.n_cells, nz, vec_ok, scratch, stride);
        else
            k_forward<AGG, false, 1><<<grid, kThreads, 0, st>>>(p.d_perm, p.d_offsets, in, out, p.n_in, p.n_cells, nz, vec_ok, scratch, stride);
        if (scratch) {
            const cudaError_t e = cudaGetLastError();
            cudaFreeAsync(scratch, st);
            FB_CUDA_CHECK(e);
        }
    }
    count_launch();
    FB_CUDA_CHECK(cudaGetLastError());
    return FB_OK;
}

} // namespace

int forward_build_plan(const int* d_cell, long long n_in, long long n_cells, ForwardPlan* plan, cudaStream_t st)
{
    FB_REQUIRE(n_in < 2147483647LL && n_cells < 2147483647LL, "forward interpolation: more than 2^31 points or cells");
    plan->n_in = n_in;
    plan->n_cells = n_cells;
    FB_CUDA_CHECK(cudaMalloc(&plan->d_perm, sizeof(int) * (size_t)(n_in > 0 ? n_in : 1)));
    FB_CUDA_CHECK(cudaMalloc(&plan->d_offsets, sizeof(int) * (size_t)(n_cells + 1)));
    if (n_in == 0) {
        FB_CUDA_CHECK(cudaMemsetAsync(plan->d_offsets, 0, sizeof(int) * (size_t)(n_cells + 1), st));
        return FB_OK;
    }
    unsigned *d_keys = nullptr, *d_keys_sorted = nullptr;
    int* d_vals = nullptr;
    void* d_tmp = nullptr;
    FB_CUDA_CHECK(cudaMallocAsync(&d_keys, sizeof(unsigned) * (size_t)n_in, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_keys_sorted, sizeof(unsigned) * (size_t)n_in, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_vals, sizeof(int) * (size_t)n_in, st));
    const int blocks = (int)((n_in + kThreads - 1) / kThreads < 65535 * 16 ? (n_in + kThreads - 1) / kThreads : 65535 * 16);
    k_forward_keys<<<blocks, kThreads, 0, st>>>(d_cell, n_in, (unsigned)n_cells, d_keys, d_vals);
    count_launch();
    int end_bit = 1;
    while (end_bit < 32 && (1ull << end_bit) <= (unsigned long long)n_cells)
        ++end_bit;
    size_t tmp_bytes = 0;
    FB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys_sorted, d_vals, plan->d_perm, (int)n_in, 0, end_bit, st));
    FB_CUDA_CHECK(cudaMallocAsync(&d_tmp, tmp_bytes ? tmp_bytes : 16, st));
    // LSD radix sort is stable: inside a cell the input indices stay ascending
    FB_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys_sorted, d_vals, plan->d_perm, (int)n_in, 0, end_bit, st));
    count_launch(4);
    const long long nb = (n_cells + 1 + kThreads - 1) / kThreads;
    k_forward_offsets<<<(int)(nb < 65535 * 16 ? nb : 65535 * 16), kThreads, 0, st>>>(d_keys_sorted, n_in, n_cells, plan->d_offsets);
    count_launch();
    FB_CUDA_CHECK(cudaGetLastError());
    int last = 0;
    FB_CUDA_CHECK(cudaMemcpyAsync(&last, plan->d_offsets + n_cells, sizeof(int), cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaFreeAsync(d_keys, st));
    FB_CUDA_CHECK(cudaFreeAsync(d_keys_sorted, st));
    FB_CUDA_CHECK(cudaFreeAsync(d_vals, st));
    FB_CUDA_CHECK(cudaFreeAsync(d_tmp, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    plan->n_mapped = last;
    return FB_OK;
}

void forward_free_plan(ForwardPlan* plan)
{
    if (plan->d_perm)
        cudaFree(plan->d_perm);
    if (plan->d_offsets)
        cudaFree(plan->d_offsets);
    plan->d_perm = nullptr;
    plan->d_offsets = nullptr;
}

int launch_forward(int method, const ForwardPlan& plan, const float* d_in, float* d_out, long long nz, cudaStream_t st)
{
    if (plan.n_cells == 0 || nz == 0)
        return FB_OK;
    const bool undef = method >= FB_FWD_UNDEF_SUM;
    const int gx = ceil_div(ceil_div(plan.n_cells, kCells), kThreads);
    const int grid = gx;
    switch (method) {
    case FB_FWD_SUM:
    case FB_FWD_UNDEF_SUM:
        return launch_agg<AG_SUM>(undef, grid, st, plan, d_in, d_out, nz);
    case FB_FWD_MEAN:
    case FB_FWD_UNDEF_MEAN:
        return launch_agg<AG_MEAN>(undef, grid, st, plan, d_in, d_out, nz);
    case FB_FWD_MEDIAN:
    case FB_FWD_UNDEF_MEDIAN:
        return launch_agg<AG_MEDIAN>(undef, grid, st, plan, d_in, d_out, nz);
    case FB_FWD_MAX:
    case FB_FWD_UNDEF_MAX:
        return launch_agg<AG_MAX>(undef, grid, st, plan, d_in, d_out, nz);
    case FB_FWD_MIN:
    case FB_FWD_UNDEF_MIN:
        return launch_agg<AG_MIN>(undef, grid, st, plan, d_in, d_out, nz);
    default:
        set_error("unknown forward interpolation method");
        return FB_ERROR;
    }
}

} // namespace fb
