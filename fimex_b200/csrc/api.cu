// fimex_b200/csrc/api.cu -- the C ABI of include/fimex_b200.h: handle lifetime, device selection, host<->device
// staging, error mapping (MIFI_OK / MIFI_ERROR).  No arithmetic of the path is done on the host here: the host
// only parses proj strings, converts axis units (a few hundred doubles) and orchestrates launches.
#include "../../include/fimex_b200.h"

#include "kernels.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <map>
#include <unordered_map>
#include <iterator>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include <unistd.h>

// ======================================================================================================
// library state
// ======================================================================================================
namespace fb {

static thread_local std::string t_error;
static thread_local int t_device = -2; // -2: not chosen yet
static std::atomic<unsigned long long> g_launches{0};

void set_error(const std::string& msg)
{
    t_error = msg;
    if (!std::getenv("FIMEX_B200_QUIET"))
        fprintf(stderr, "fimex_b200: %s\n", msg.c_str());
}
const char* last_error()
{
    return t_error.c_str();
}
void count_launch(int n)
{
    g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed);
}
unsigned long long launches()
{
    return g_launches.load(std::memory_order_relaxed);
}

int sm_count()
{
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess)
        return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
        cached = n;
        cached_dev = dev;
    }
    return cached;
}

namespace {

std::once_flag g_pool_once[64];

// make `dev` current; keep freed stream-ordered scratch in the pool instead of returning it to the driver
int use_device(int dev)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error(std::string("no usable CUDA device (this library has no CPU fallback): ") + cudaGetErrorString(e));
        return FB_ERROR;
    }
    FB_REQUIRE(dev >= 0 && dev < count, "CUDA device index out of range");
    FB_CUDA_CHECK(cudaSetDevice(dev));
    if (dev < 64) {
        std::call_once(g_pool_once[dev], [dev]() {
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
                unsigned long long keep = ~0ull;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            }
        });
    }
    return FB_OK;
}

int default_device()
{
    if (t_device == -2) {
        const char* env = std::getenv("FIMEX_B200_DEVICE");
        if (env && *env) {
            t_device = std::atoi(env);
        } else {
            int cur = 0;
            t_device = (cudaGetDevice(&cur) == cudaSuccess) ? cur : 0;
        }
    }
    return t_device;
}

// Switch the calling thread's current device for a scope and put it back: destructors and helpers must not leak a
// cudaSetDevice into the caller (a thread may alternate between handles that live on different GPUs).
struct DeviceGuard {
    int saved = -1;
    bool switched = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&saved) != cudaSuccess)
            saved = -1;
        if (dev >= 0 && dev != saved)
            switched = cudaSetDevice(dev) == cudaSuccess;
    }
    bool ok(int dev) const { return switched || saved == dev; }
    ~DeviceGuard()
    {
        if (switched && saved >= 0)
            cudaSetDevice(saved);
    }
};

cudaStream_t as_stream(void* s)
{
    return s ? reinterpret_cast<cudaStream_t>(s) : cudaStreamPerThread;
}

template <typename T>
int dev_alloc(T** p, size_t count)
{
    FB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(p), sizeof(T) * (count ? count : 1)));
    return FB_OK;
}

// RAII for stream-ordered scratch
struct Scratch {
    cudaStream_t st;
    std::vector<void*> ptrs;
    explicit Scratch(cudaStream_t s) : st(s) {}
    ~Scratch()
    {
        for (void* p : ptrs)
            cudaFreeAsync(p, st);
    }
    template <typename T>
    int get(T** p, size_t count)
    {
        void* q = nullptr;
        FB_CUDA_CHECK(cudaMallocAsync(&q, sizeof(T) * (count ? count : 1), st));
        ptrs.push_back(q);
        *p = static_cast<T*>(q);
        return FB_OK;
    }
    template <typename T>
    int upload(T** p, const T* host, size_t count)
    {
        if (get(p, count) != FB_OK)
            return FB_ERROR;
        if (count)
            FB_CUDA_CHECK(cudaMemcpyAsync(*p, host, sizeof(T) * count, cudaMemcpyHostToDevice, st));
        return FB_OK;
    }
};

int check_status(int* d_status, cudaStream_t st, const char* what)
{
    int h = 0;
    FB_CUDA_CHECK(cudaMemcpyAsync(&h, d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    if (h != 0) {
        set_error(std::string(what) + ": projection failed with proj error " + std::to_string(h));
        return FB_ERROR;
    }
    return FB_OK;
}

int parse_pair(const char* a, const char* b, ProjDef* pa, ProjDef* pb)
{
    char msg[256];
    FB_REQUIRE(a && b, "null projection string");
    if (parse_proj(a, pa, msg, sizeof(msg)) != 0) {
        set_error(std::string("Proj error: ") + msg + " in '" + a + "'");
        return FB_ERROR;
    }
    if (parse_proj(b, pb, msg, sizeof(msg)) != 0) {
        set_error(std::string("Proj error: ") + msg + " in '" + b + "'");
        return FB_ERROR;
    }
    return FB_OK;
}

// convertAxis (interpolation.c:221-229) / the DEG_TO_RAD transforms of CDMInterpolator.cc:1446-1451,1468-1473
std::vector<double> axis_in_radians(const double* axis, size_t n, bool degree)
{
    std::vector<double> out(n);
    for (size_t i = 0; i < n; ++i) {
        volatile double v = degree ? FB_DEG_TO_RAD * axis[i] : axis[i];
        out[i] = v;
    }
    return out;
}

bool is_backward(int m)
{
    return m == FB_NN || m == FB_BILINEAR || m == FB_BICUBIC || m == FB_COORD_NN || m == FB_COORD_NN_KD;
}
bool is_forward(int m)
{
    return m >= FB_FWD_SUM && m <= FB_FWD_UNDEF_MIN;
}

} // namespace
} // namespace fb

using namespace fb;

// ======================================================================================================
// handles
// ======================================================================================================
struct fb200_interp {
    int method = -1;
    bool forward = false;
    int device = 0;
    size_t inX = 0, inY = 0, outX = 0, outY = 0;
    size_t srcX = 0, srcY = 0; // the source grid as created: inX, inY before createReducedDomain cropped them
    size_t npts = 0; // outX*outY (backward) or inX*inY (forward)
    double* d_px = nullptr;
    double* d_py = nullptr;
    // compiled tables (exactly one family is non-null)
    int* d_nn = nullptr;
    int4* d_bil = nullptr;
    int* d_bic_off = nullptr;
    double2* d_bic_frac = nullptr;
    ForwardPlan fwd;
    TileTable tiles;       // staged fast path of the bilinear / nearest-neighbour gather
    BicubicTiles bic_tiles; // staged fast path of the bicubic gather
    bool reduced = false;
    bool invalid = false; // a table rebuild failed half-way (createReducedDomain out of memory): every later call is refused
    long long xMin = 0, yMin = 0;
    long long coordnn_ties = 0;
    // 2-D pre/post-processes of getDataSlice (CDMInterpolator::addPreprocess / addPostprocess, src/CDMInterpolator.cc:1886-1896)
    struct Process {
        int kind = 0; // 0 fill2d, 1 creepfill2d, 2 creepfillval2d
        float relaxCrit = 0.f, corrEff = 0.f, defVal = 0.f;
        size_t maxLoop = 0;
        unsigned short repeat = 0;
        signed char weight = 0;
    };
    std::vector<Process> preprocesses, postprocesses;

    ~fb200_interp()
    {
        fb::DeviceGuard on(device); // restored on return: destroying a handle does not change the caller's current device
        free_tables();
        if (d_px)
            cudaFree(d_px);
        if (d_py)
            cudaFree(d_py);
    }
    void free_tables()
    {
        if (d_nn)
            cudaFree(d_nn);
        if (d_bil)
            cudaFree(d_bil);
        if (d_bic_off)
            cudaFree(d_bic_off);
        if (d_bic_frac)
            cudaFree(d_bic_frac);
        d_nn = nullptr;
        d_bil = nullptr;
        d_bic_off = nullptr;
        d_bic_frac = nullptr;
        forward_free_plan(&fwd);
        tile_table_free(&tiles);
        bicubic_tiles_free(&bic_tiles);
    }
};

struct fb200_vector {
    int method = 0;
    int ox = 0, oy = 0;
    int device = 0;
    double* d_matrix = nullptr; // [oy][ox][4]
    double2* d_cs = nullptr;    // compact (cos, sin)
    ~fb200_vector()
    {
        fb::DeviceGuard on(device);
        if (d_matrix)
            cudaFree(d_matrix);
        if (d_cs)
            cudaFree(d_cs);
    }
};

namespace {

// positions -> gather tables (or forward CSR plan); synchronises
int compile_tables(fb200_interp* h, cudaStream_t st)
{
    h->free_tables();
    const long long n = (long long)h->npts;
    if (h->forward) {
        Scratch tmp(st);
        int* d_cell = nullptr;
        if (tmp.get(&d_cell, h->npts) != FB_OK)
            return FB_ERROR;
        if (launch_compile_forward_cells(h->d_px, h->d_py, n, (int)h->outX, (int)h->outY, d_cell, st) != FB_OK)
            return FB_ERROR;
        return forward_build_plan(d_cell, n, (long long)h->outX * (long long)h->outY, &h->fwd, st);
    }
    FB_REQUIRE((long long)h->inX * (long long)h->inY < 2147483647LL, "source grid larger than 2^31 cells");
    switch (h->method) {
    case FB_BILINEAR:
        if (dev_alloc(&h->d_bil, h->npts) != FB_OK)
            return FB_ERROR;
        if (launch_compile_bilinear(h->d_px, h->d_py, n, (int)h->inX, (int)h->inY, h->d_bil, st) != FB_OK)
            return FB_ERROR;
        if (tile_table_supported((int)h->inX, (int)h->inY, (int)h->outX, (int)h->outY) && !std::getenv("FIMEX_B200_DIRECT_GATHER")) {
            if (tile_table_build(false, h->d_px, h->d_py, (int)h->inX, (int)h->inY, (int)h->outX, (int)h->outY, &h->tiles, st) != FB_OK)
                return FB_ERROR;
        }
        break;
    case FB_BICUBIC:
        if (dev_alloc(&h->d_bic_off, h->npts) != FB_OK || dev_alloc(&h->d_bic_frac, h->npts) != FB_OK)
            return FB_ERROR;
        if (launch_compile_bicubic(h->d_px, h->d_py, n, (int)h->inX, (int)h->inY, h->d_bic_off, h->d_bic_frac, st) != FB_OK)
            return FB_ERROR;
        if (bicubic_tiles_supported((int)h->inX, (int)h->inY, (int)h->outX, (int)h->outY) && !std::getenv("FIMEX_B200_DIRECT_GATHER")) {
            if (bicubic_tiles_build(h->d_bic_off, h->d_bic_frac, (int)h->inX, (int)h->inY, (int)h->outX, (int)h->outY, &h->bic_tiles, st) !=
                FB_OK)
                return FB_ERROR;
        }
        break;
    default:
        if (dev_alloc(&h->d_nn, h->npts) != FB_OK)
            return FB_ERROR;
        if (launch_compile_nn(h->d_px, h->d_py, n, (int)h->inX, (int)h->inY, h->d_nn, st) != FB_OK)
            return FB_ERROR;
        if (tile_table_supported((int)h->inX, (int)h->inY, (int)h->outX, (int)h->outY) && !std::getenv("FIMEX_B200_DIRECT_GATHER")) {
            if (tile_table_build(true, h->d_px, h->d_py, (int)h->inX, (int)h->inY, (int)h->outX, (int)h->outY, &h->tiles, st) != FB_OK)
                return FB_ERROR;
        }
        break;
    }
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return FB_OK;
}

int new_interp(int funcType, bool forward, size_t inX, size_t inY, size_t outX, size_t outY, std::unique_ptr<fb200_interp>* out)
{
    if (forward)
        FB_REQUIRE(is_forward(funcType), "unknown forward interpolation method: " + std::to_string(funcType));
    else
        FB_REQUIRE(is_backward(funcType), "unknown interpolation function: " + std::to_string(funcType));
    FB_REQUIRE(inX < 2147483647u && inY < 2147483647u && outX < 2147483647u && outY < 2147483647u, "grid dimension too large");
    if (use_device(default_device()) != FB_OK)
        return FB_ERROR;
    std::unique_ptr<fb200_interp> h(new fb200_interp());
    h->method = funcType;
    h->forward = forward;
    h->device = default_device();
    h->inX = inX;
    h->inY = inY;
    h->srcX = inX;
    h->srcY = inY;
    h->outX = outX;
    h->outY = outY;
    h->npts = forward ? inX * inY : outX * outY;
    if (dev_alloc(&h->d_px, h->npts) != FB_OK || dev_alloc(&h->d_py, h->npts) != FB_OK)
        return FB_ERROR;
    *out = std::move(h);
    return FB_OK;
}

int create_from_points(int funcType, bool forward, const double* px, const double* py, bool on_device, size_t inX, size_t inY, size_t outX,
                       size_t outY, fb200_interp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    std::unique_ptr<fb200_interp> h;
    if (new_interp(funcType, forward, inX, inY, outX, outY, &h) != FB_OK)
        return FB_ERROR;
    FB_REQUIRE(h->npts == 0 || (px && py), "null position table");
    cudaStream_t st = cudaStreamPerThread;
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (h->npts) {
        FB_CUDA_CHECK(cudaMemcpyAsync(h->d_px, px, sizeof(double) * h->npts, kind, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(h->d_py, py, sizeof(double) * h->npts, kind, st));
    }
    if (compile_tables(h.get(), st) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = h.release();
    return FB_OK;
}

GatherGeom geom_of(const fb200_interp* h, size_t nz)
{
    GatherGeom g;
    g.ix = (int)h->inX;
    g.iy = (int)h->inY;
    g.ox = (int)h->outX;
    g.oy = (int)h->outY;
    g.in_level = (long long)h->inX * (long long)h->inY;
    g.out_level = (long long)h->outX * (long long)h->outY;
    g.nz = (long long)nz;
    return g;
}

// types and fill values either side of the gather for one slice call (CDMInterpolator::getDataSlice, :250-285)
struct SliceIO {
    bool typed = false; // false: CachedInterpolationInterface::interpolateValues itself (float in, float out, NaN = undefined)
    int in_type = FB_T_FLOAT, out_type = FB_T_FLOAT;
    double bad[2] = {0., 0.}; // CDM::getFillValue of each field: fill -> NaN on the way in, NaN -> fill on the way out
};

// the gather itself: float slabs in, plain floats out -- or, where the kernel can, converted while storing (sc)
int run_gather(const fb200_interp* h, const float* d_in, size_t nz, void* d_out, const SliceConv& sc, cudaStream_t st)
{
    if (h->forward)
        return launch_forward(h->method, h->fwd, d_in, static_cast<float*>(d_out), (long long)nz, st);
    const GatherGeom g = geom_of(h, nz);
    switch (h->method) {
    case FB_BILINEAR:
        if (h->tiles.ready())
            return launch_gather_bilinear_staged(g, h->tiles, d_in, d_out, sc, st);
        return launch_gather_bilinear(g, h->d_bil, d_in, static_cast<float*>(d_out), st);
    case FB_BICUBIC:
        if (h->bic_tiles.ready())
            return launch_gather_bicubic_staged(g, h->bic_tiles, h->d_bic_off, h->d_bic_frac, nullptr, d_in, nullptr, d_out, nullptr, sc, st);
        return launch_gather_bicubic(g, h->d_bic_off, h->d_bic_frac, d_in, static_cast<float*>(d_out), st);
    default:
        if (h->tiles.ready())
            return launch_gather_bilinear_staged(g, h->tiles, d_in, d_out, sc, st);
        return launch_gather_nn(g, h->d_nn, d_in, static_cast<float*>(d_out), st);
    }
}

int run_gather_vector(const fb200_interp* h, const fb200_vector* v, const float* d_u, const float* d_v, size_t nz, float* d_uo, float* d_vo,
                      const SliceConv& sc, cudaStream_t st)
{
    const GatherGeom g = geom_of(h, nz);
    const double2* cs = v ? v->d_cs : nullptr;
    switch (h->method) {
    case FB_BILINEAR:
        if (h->tiles.ready())
            return launch_gather_staged_vector(g, h->tiles, cs, d_u, d_v, d_uo, d_vo, sc, st);
        return launch_gather_vector(FB_BILINEAR, g, h->d_bil, nullptr, cs, d_u, d_v, d_uo, d_vo, st);
    case FB_BICUBIC:
        if (h->bic_tiles.ready())
            return launch_gather_bicubic_staged(g, h->bic_tiles, h->d_bic_off, h->d_bic_frac, cs, d_u, d_v, d_uo, d_vo, sc, st);
        return launch_gather_vector(FB_BICUBIC, g, h->d_bic_off, h->d_bic_frac, cs, d_u, d_v, d_uo, d_vo, st);
    default:
        if (h->tiles.ready())
            return launch_gather_staged_vector(g, h->tiles, cs, d_u, d_v, d_uo, d_vo, sc, st);
        return launch_gather_vector(FB_NN, g, h->d_nn, nullptr, cs, d_u, d_v, d_uo, d_vo, st);
    }
}

// processArray_ (src/CDMInterpolator.cc:136-159): every process on every level of a float slab, in place
int process_array(const std::vector<fb200_interp::Process>& procs, float* d_array, size_t nx, size_t ny, size_t nz, cudaStream_t st)
{
    for (const fb200_interp::Process& p : procs) {
        int rc;
        if (p.kind == 0)
            rc = launch_fill2d(d_array, nx, ny, nz, p.relaxCrit, p.corrEff, p.maxLoop, nullptr, st);
        else
            rc = launch_creepfill2d(d_array, nx, ny, nz, p.kind == 1, p.defVal, p.repeat, p.weight, nullptr, st);
        if (rc != FB_OK)
            return rc;
    }
    return FB_OK;
}

// One slice on the device: nfields = 1 (scalar) or 2 (u/v with optional rotation).  With io.typed this is
// data2InterpolationArray -> interpolateValues [-> reprojectValues] -> interpolationArray2Data; the staged gathers do the
// first and last step inside the gather kernel, everything else goes through a float slab and a conversion pass.
int run_slice_device(const fb200_interp* h, const fb200_vector* v, int nfields, const void* const* d_in, size_t nz, void* const* d_out,
                     const SliceIO& io, cudaStream_t st)
{
    const size_t in_n = nz * h->inX * h->inY, out_n = nz * h->outX * h->outY;
    if (nz == 0 || out_n == 0)
        return FB_OK;
    const bool staged_scalar = nfields == 1 && !h->forward && (h->method == FB_BICUBIC ? h->bic_tiles.ready() : h->tiles.ready());
    const bool staged_vector = nfields == 2 && !h->forward && (h->method == FB_BICUBIC ? h->bic_tiles.ready() : h->tiles.ready());
    const bool kernel_fills = staged_scalar || staged_vector;
    const bool pre = io.typed && !h->preprocesses.empty(), post = io.typed && !h->postprocesses.empty();
    Scratch tmp(st);
    SliceConv sc;
    const float* fin[2] = {nullptr, nullptr};
    for (int f = 0; f < nfields; ++f) {
        const float bad = (float)io.bad[f]; // mifi_bad2nanf takes a float (interpolation.c:1775)
        const bool has_bad = io.typed && !std::isnan(bad);
        sc.bad_in[f] = std::numeric_limits<float>::quiet_NaN();
        if (pre) { // the preprocesses work in place on the float + NaN array (:254-256): a private copy of the input
            float* conv = nullptr;
            if (tmp.get(&conv, in_n) != FB_OK || launch_as_float(io.in_type, d_in[f], (long long)in_n, has_bad, bad, conv, st) != FB_OK ||
                process_array(h->preprocesses, conv, h->inX, h->inY, nz, st) != FB_OK)
                return FB_ERROR;
            fin[f] = conv;
        } else if (!io.typed || (io.in_type == FB_T_FLOAT && (!has_bad || kernel_fills))) {
            fin[f] = static_cast<const float*>(d_in[f]);
            if (has_bad) {
                sc.fill_in = true;
                sc.bad_in[f] = bad;
            }
        } else {
            float* conv = nullptr;
            if (tmp.get(&conv, in_n) != FB_OK || launch_as_float(io.in_type, d_in[f], (long long)in_n, has_bad, bad, conv, st) != FB_OK)
                return FB_ERROR;
            fin[f] = conv;
        }
    }
    if (!io.typed) {
        if (nfields == 1)
            return run_gather(h, fin[0], nz, d_out[0], sc, st);
        return run_gather_vector(h, v, fin[0], fin[1], nz, static_cast<float*>(d_out[0]), static_cast<float*>(d_out[1]), sc, st);
    }
    if (!post && staged_scalar && staged_store_supports(io.out_type)) { // the fused form: one pass over the output
        sc.convert_out = true;
        sc.out_type = io.out_type;
        sc.fill_out = io.bad[0];
        return run_gather(h, fin[0], nz, d_out[0], sc, st);
    }
    float* fout[2] = {nullptr, nullptr};
    for (int f = 0; f < nfields; ++f) {
        if (io.out_type == FB_T_FLOAT)
            fout[f] = static_cast<float*>(d_out[f]); // converted in place afterwards
        else if (tmp.get(&fout[f], out_n) != FB_OK)
            return FB_ERROR;
    }
    const int rc = nfields == 1 ? run_gather(h, fin[0], nz, fout[0], sc, st) : run_gather_vector(h, v, fin[0], fin[1], nz, fout[0], fout[1], sc, st);
    if (rc != FB_OK)
        return rc;
    for (int f = 0; f < nfields; ++f) {
        if (post && process_array(h->postprocesses, fout[f], h->outX, h->outY, nz, st) != FB_OK) // :284
            return FB_ERROR;
        if (launch_from_float(fout[f], (long long)out_n, io.out_type, io.bad[f], d_out[f], st) != FB_OK)
            return FB_ERROR;
    }
    return FB_OK;
}

// Per host thread and device: the three streams of the host-buffer pipeline and its events, created once.  A call owns them
// for its duration (a thread runs one call at a time), so concurrent calls from several threads never share a stream.
struct HostPipe {
    int device = -1;
    cudaStream_t up = nullptr, run = nullptr, down = nullptr;
    cudaEvent_t ev[3][3] = {};
    cudaEvent_t ready = nullptr;
    void destroy()
    {
        if (device < 0)
            return;
        DeviceGuard on(device); // the caller's current device is put back afterwards
        if (on.ok(device)) {    // fails harmlessly when the runtime is already shutting down
            for (auto& row : ev)
                for (cudaEvent_t& e : row)
                    if (e)
                        cudaEventDestroy(e);
            if (ready)
                cudaEventDestroy(ready);
            if (up)
                cudaStreamDestroy(up);
            if (run)
                cudaStreamDestroy(run);
            if (down)
                cudaStreamDestroy(down);
        }
        *this = HostPipe();
    }
    ~HostPipe() { destroy(); }
};

HostPipe* host_pipe(int device)
{
    // one pipe per (host thread, device): a thread that alternates between handles on two GPUs keeps both sets of streams
    static thread_local std::map<int, std::unique_ptr<HostPipe>> pipes;
    auto it = pipes.find(device);
    if (it != pipes.end())
        return it->second.get();
    // streams and events belong to the device that is current when they are created: make that the handle's device for the
    // duration, whatever the thread used last, and put the caller's device back
    DeviceGuard on(device);
    if (!on.ok(device))
        return nullptr;
    std::unique_ptr<HostPipe> pipe(new HostPipe());
    bool ok = cudaStreamCreateWithFlags(&pipe->up, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&pipe->run, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&pipe->down, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&pipe->ready, cudaEventDisableTiming) == cudaSuccess;
    for (auto& row : pipe->ev)
        for (cudaEvent_t& e : row)
            ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    pipe->device = device; // so that destroy() releases whatever was created
    if (!ok)
        return nullptr; // ~HostPipe releases the partial set
    HostPipe* raw = pipe.get();
    pipes.emplace(device, std::move(pipe));
    return raw;
}

// ---- pageable host buffers ------------------------------------------------------------------------------------------------
// The reference hands `new float[]` arrays in and expects one back (boost::shared_array).  cudaMemcpyAsync to or from such
// pageable memory goes through the driver's own staging at ~15 GB/s (measured: a 137-level call takes 146 ms instead of
// 43 ms), slower than the reference's CPU loop; staged here with 16 host threads it takes 79 ms.  run_slice_host therefore detects pageable buffers and stages them itself:
// page-locked bounce buffers from the pinned cache, filled / drained by a few host threads while the next chunks are in flight.
bool host_pageable(const void* p)
{
    if (!p)
        return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError(); // older drivers report plain malloc memory as an error
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

int copy_threads()
{
    static const int n = []() {
        int want = 16; // measured (one 2.19 GB pageable output, 16-core host): 1 / 4 / 8 / 16 threads -> 167 / 105 / 93 / 79 ms
        if (const char* env = std::getenv("FIMEX_B200_COPY_THREADS"))
            want = std::atoi(env);
        const int hw = (int)std::thread::hardware_concurrency();
        if (hw > 0 && want > hw)
            want = hw;
        return want < 1 ? 1 : want;
    }();
    return n;
}

void parallel_memcpy(void* dst, const void* src, size_t bytes)
{
    const int nt = copy_threads();
    if (nt <= 1 || bytes < (size_t)(8u << 20)) {
        std::memcpy(dst, src, bytes);
        return;
    }
    const size_t per = ((bytes + nt - 1) / nt + 4095) & ~(size_t)4095;
    std::vector<std::thread> workers;
    size_t done_by_workers_from = bytes; // everything below this offset that no worker took is copied here
    for (int t = nt - 1; t >= 1; --t) {
        const size_t off = per * (size_t)t;
        if (off >= bytes)
            continue;
        const size_t len = done_by_workers_from - off;
        try {
            workers.emplace_back([=]() { std::memcpy(static_cast<char*>(dst) + off, static_cast<const char*>(src) + off, len); });
        } catch (...) { // no more threads to be had: the calling thread copies the rest
            break;
        }
        done_by_workers_from = off;
    }
    std::memcpy(dst, src, done_by_workers_from);
    for (auto& w : workers)
        w.join();
}

// Host arrays of a call that the device works through in chunks of `units` (levels, time steps): up to four inputs and two
// outputs, each `bytes per unit` long per unit (0: that array is absent and its device pointer is null).
constexpr int kHostIn = 4, kHostOut = 2;
struct HostArrays {
    int device = 0;
    const void* in[kHostIn] = {nullptr, nullptr, nullptr, nullptr};
    size_t in_unit[kHostIn] = {0, 0, 0, 0};
    void* out[kHostOut] = {nullptr, nullptr};
    size_t out_unit[kHostOut] = {0, 0};
};
// the device work of one chunk: `n` units of every array, already on the device
using ChunkRun = std::function<int(const void* const* d_in, size_t n, void* const* d_out, cudaStream_t st)>;

// Host-buffer execution: units are cut into chunks that rotate through three (stream, scratch) slots, so that
// the H2D copy of chunk k+1, the kernel of chunk k and the D2H copy of chunk k-1 overlap.  Every call owns its
// streams and scratch => re-entrant on a shared handle.
int stage_host(const HostArrays& io, size_t nz, const ChunkRun& run)
{
    size_t bytes_per_level = 0;
    for (int f = 0; f < kHostIn; ++f)
        bytes_per_level += io.in_unit[f];
    for (int f = 0; f < kHostOut; ++f)
        bytes_per_level += io.out_unit[f];
    size_t chunk_bytes = 192ull << 20;
    if (const char* env = std::getenv("FIMEX_B200_HOST_CHUNK_MB")) // experiments: bytes of (input + output) per pipeline chunk
        if (std::atoll(env) > 0)
            chunk_bytes = (size_t)std::atoll(env) << 20;
    size_t zc = chunk_bytes / (bytes_per_level ? bytes_per_level : 1);
    if (zc < 1)
        zc = 1;
    if (zc > nz)
        zc = nz;
    // Three streams by ROLE: uploads, kernels and downloads each form one back-to-back queue, so both copy engines stay busy in
    // both PCIe directions.  Slots rotate through three sets of device buffers; events order upload -> kernel -> download per
    // chunk and guard the reuse of a slot's buffers.  Measured on B200 (PCIe Gen5 x16): a 137-level call (0.16 GB up, 2.19 GB
    // down) takes 41.7 ms = 52 GB/s; one monolithic 2.19 GB download takes 38.3-40.3 ms, the same bytes as 13 back-to-back
    // copies 42.5 ms, so the call runs at the rate chunked copies allow and the kernels are invisible.
    bool bounce_in = false, bounce_out = false; // pageable host arrays: staged through page-locked bounce buffers, see above
    // (with fewer than 4 host threads the driver's own staging, one thread at ~15 GB/s, is as fast; small calls are latency-bound)
    if (copy_threads() >= 4 && nz * bytes_per_level >= (size_t)(8u << 20)) {
        for (int f = 0; f < kHostIn; ++f)
            bounce_in = bounce_in || (io.in_unit[f] && host_pageable(io.in[f]));
        for (int f = 0; f < kHostOut; ++f)
            bounce_out = bounce_out || (io.out_unit[f] && host_pageable(io.out[f]));
    }
    if ((bounce_in || bounce_out) && zc * bytes_per_level > (64ull << 20)) { // smaller chunks: the host copy of chunk k runs while k+1, k+2 are in flight
        zc = (64ull << 20) / bytes_per_level;
        if (zc < 1)
            zc = 1;
    }
    const int nslots = (nz > zc) ? 3 : 1;
    struct Slot {
        void* d_in[kHostIn] = {nullptr, nullptr, nullptr, nullptr};
        void* d_out[kHostOut] = {nullptr, nullptr};
        void* h_in[kHostIn] = {nullptr, nullptr, nullptr, nullptr}; // bounce buffers (page-locked, from the pinned cache)
        void* h_out[kHostOut] = {nullptr, nullptr};
        cudaEvent_t uploaded = nullptr, computed = nullptr, downloaded = nullptr;
    } slots[3];
    HostPipe* pipe = host_pipe(io.device);
    FB_REQUIRE(pipe != nullptr, std::string("cannot create the copy / compute streams: ") + cudaGetErrorString(cudaGetLastError()));
    const cudaStream_t s_up = pipe->up, s_run = pipe->run, s_down = pipe->down;
    for (int s = 0; s < nslots; ++s) {
        slots[s].uploaded = pipe->ev[s][0];
        slots[s].computed = pipe->ev[s][1];
        slots[s].downloaded = pipe->ev[s][2];
    }
    int rc = FB_OK;
    const bool trace = std::getenv("FIMEX_B200_TRACE") != nullptr;
    auto now = []() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t0 = now(), t1 = 0, t2 = 0, t3 = 0;
    auto body = [&]() -> int {
        for (int s = 0; s < nslots; ++s) {
            for (int f = 0; f < kHostIn; ++f)
                if (io.in_unit[f])
                    FB_CUDA_CHECK(cudaMallocAsync(&slots[s].d_in[f], zc * io.in_unit[f], s_run));
            for (int f = 0; f < kHostOut; ++f)
                if (io.out_unit[f])
                    FB_CUDA_CHECK(cudaMallocAsync(&slots[s].d_out[f], zc * io.out_unit[f], s_run));
        }
        // the buffers were allocated in s_run's order: the copy streams must not touch them earlier
        cudaEvent_t ready = pipe->ready;
        FB_CUDA_CHECK(cudaEventRecord(ready, s_run));
        FB_CUDA_CHECK(cudaStreamWaitEvent(s_up, ready, 0));
        FB_CUDA_CHECK(cudaStreamWaitEvent(s_down, ready, 0));
        if (bounce_in || bounce_out) {
            for (int s = 0; s < nslots; ++s) {
                for (int f = 0; f < kHostIn; ++f) {
                    if (bounce_in && io.in_unit[f]) {
                        slots[s].h_in[f] = fb200_host_alloc(zc * io.in_unit[f]);
                        FB_REQUIRE(slots[s].h_in[f] != nullptr, "cannot allocate a page-locked staging buffer");
                    }
                }
                for (int f = 0; f < kHostOut; ++f) {
                    if (bounce_out && io.out_unit[f]) {
                        slots[s].h_out[f] = fb200_host_alloc(zc * io.out_unit[f]);
                        FB_REQUIRE(slots[s].h_out[f] != nullptr, "cannot allocate a page-locked staging buffer");
                    }
                }
            }
        }
        t1 = now();
        const size_t nchunks = (nz + zc - 1) / zc;
        auto enqueue = [&](size_t chunk) -> int {
            Slot& sl = slots[chunk % nslots];
            const bool reused = chunk >= (size_t)nslots;
            const size_t z0 = chunk * zc;
            const size_t zn = (z0 + zc <= nz) ? zc : nz - z0;
            if (reused) // the kernel that read this slot's input three chunks ago is done
                FB_CUDA_CHECK(cudaStreamWaitEvent(s_up, sl.computed, 0));
            for (int f = 0; f < kHostIn; ++f) {
                if (!io.in_unit[f])
                    continue;
                const char* src = static_cast<const char*>(io.in[f]) + z0 * io.in_unit[f];
                if (bounce_in) { // the upload that last read this bounce buffer finished before its chunk's download was waited for
                    parallel_memcpy(sl.h_in[f], src, zn * io.in_unit[f]);
                    src = static_cast<const char*>(sl.h_in[f]);
                }
                FB_CUDA_CHECK(cudaMemcpyAsync(sl.d_in[f], src, zn * io.in_unit[f], cudaMemcpyHostToDevice, s_up));
            }
            FB_CUDA_CHECK(cudaEventRecord(sl.uploaded, s_up));
            FB_CUDA_CHECK(cudaStreamWaitEvent(s_run, sl.uploaded, 0));
            if (reused) // ... and the download of its previous output
                FB_CUDA_CHECK(cudaStreamWaitEvent(s_run, sl.downloaded, 0));
            if (run(sl.d_in, zn, sl.d_out, s_run) != FB_OK)
                return FB_ERROR;
            FB_CUDA_CHECK(cudaEventRecord(sl.computed, s_run));
            FB_CUDA_CHECK(cudaStreamWaitEvent(s_down, sl.computed, 0));
            for (int f = 0; f < kHostOut; ++f) {
                if (!io.out_unit[f])
                    continue;
                char* dst = bounce_out ? static_cast<char*>(sl.h_out[f]) : static_cast<char*>(io.out[f]) + z0 * io.out_unit[f];
                FB_CUDA_CHECK(cudaMemcpyAsync(dst, sl.d_out[f], zn * io.out_unit[f], cudaMemcpyDeviceToHost, s_down));
            }
            FB_CUDA_CHECK(cudaEventRecord(sl.downloaded, s_down));
            return FB_OK;
        };
        if (!bounce_in && !bounce_out) { // page-locked host arrays: everything is enqueued at once
            for (size_t chunk = 0; chunk < nchunks; ++chunk)
                if (enqueue(chunk) != FB_OK)
                    return FB_ERROR;
            t2 = now();
            FB_CUDA_CHECK(cudaStreamSynchronize(s_down)); // every download waited for its kernel, every kernel for its upload
            t3 = now();
            return FB_OK;
        }
        // pageable host arrays: nslots chunks in flight; the host drains chunk k (and fills chunk k + nslots) meanwhile
        for (size_t chunk = 0; chunk < nchunks && chunk < (size_t)nslots; ++chunk)
            if (enqueue(chunk) != FB_OK)
                return FB_ERROR;
        for (size_t chunk = 0; chunk < nchunks; ++chunk) {
            Slot& sl = slots[chunk % nslots];
            const size_t z0 = chunk * zc;
            const size_t zn = (z0 + zc <= nz) ? zc : nz - z0;
            FB_CUDA_CHECK(cudaEventSynchronize(sl.downloaded));
            if (bounce_out)
                for (int f = 0; f < kHostOut; ++f)
                    if (io.out_unit[f])
                        parallel_memcpy(static_cast<char*>(io.out[f]) + z0 * io.out_unit[f], sl.h_out[f], zn * io.out_unit[f]);
            if (chunk + nslots < nchunks && enqueue(chunk + nslots) != FB_OK)
                return FB_ERROR;
        }
        t2 = now();
        FB_CUDA_CHECK(cudaStreamSynchronize(s_down));
        t3 = now();
        return FB_OK;
    };
    rc = body();
    if (rc != FB_OK) { // drain whatever was enqueued before the buffers go away
        cudaStreamSynchronize(s_up);
        cudaStreamSynchronize(s_run);
        cudaStreamSynchronize(s_down);
    }
    // all work that touches the buffers is complete: hand them back in s_run's order (no further synchronisation needed)
    for (int s = 0; s < nslots; ++s) {
        for (int f = 0; f < kHostIn; ++f) {
            if (slots[s].d_in[f])
                cudaFreeAsync(slots[s].d_in[f], s_run);
            if (slots[s].h_in[f])
                fb200_host_free(slots[s].h_in[f]);
        }
        for (int f = 0; f < kHostOut; ++f) {
            if (slots[s].d_out[f])
                cudaFreeAsync(slots[s].d_out[f], s_run);
            if (slots[s].h_out[f])
                fb200_host_free(slots[s].h_out[f]);
        }
    }
    if (trace)
        fprintf(stderr, "[fb200 trace] host slice: setup %.3f ms, enqueue %.3f ms, wait %.3f ms, cleanup %.3f ms\n", t1 - t0, t2 - t1, t3 - t2,
                now() - t3);
    return rc;
}

// `nfields` is 1 (scalar) or 2 (u/v); the levels are the units of the pipeline
int run_slice_host(const fb200_interp* h, const fb200_vector* v, int nfields, const void* const* in, void* const* out, size_t nz,
                   const SliceIO& io)
{
    const size_t in_level = h->inX * h->inY, out_level = h->outX * h->outY;
    if (nz == 0 || out_level == 0)
        return FB_OK;
    const size_t in_elem = io.typed ? type_size(io.in_type) : sizeof(float), out_elem = io.typed ? type_size(io.out_type) : sizeof(float);
    FB_REQUIRE(in_elem > 0 && out_elem > 0, "unsupported data type");
    HostArrays arrays;
    arrays.device = h->device;
    for (int f = 0; f < nfields; ++f) {
        arrays.in[f] = in[f];
        arrays.in_unit[f] = in_level * in_elem;
        arrays.out[f] = out[f];
        arrays.out_unit[f] = out_level * out_elem;
    }
    return stage_host(arrays, nz, [&](const void* const* d_in, size_t zn, void* const* d_out, cudaStream_t st) {
        return run_slice_device(h, v, nfields, d_in, zn, d_out, io, st);
    });
}

// plain interpolateValues forms of the above
int run_device(const fb200_interp* h, const float* d_in, size_t nz, float* d_out, cudaStream_t st)
{
    const void* in[1] = {d_in};
    void* out[1] = {d_out};
    return run_slice_device(h, nullptr, 1, in, nz, out, SliceIO(), st);
}

int run_vector_device(const fb200_interp* h, const fb200_vector* v, const float* d_u, const float* d_v, size_t nz, float* d_uo, float* d_vo,
                      cudaStream_t st)
{
    const void* in[2] = {d_u, d_v};
    void* out[2] = {d_uo, d_vo};
    return run_slice_device(h, v, 2, in, nz, out, SliceIO(), st);
}

int run_host(const fb200_interp* h, const fb200_vector* v, int nfields, const float* const* in, float* const* out, size_t nz)
{
    const void* vin[2] = {in[0], nfields > 1 ? in[1] : nullptr};
    void* vout[2] = {out[0], nfields > 1 ? out[1] : nullptr};
    return run_slice_host(h, v, nfields, vin, vout, nz, SliceIO());
}

bool known_type(int t)
{
    return type_size(t) > 0;
}

int check_interp_call(const fb200_interp* h, size_t size, size_t* nz)
{
    FB_REQUIRE(h != nullptr, "null interpolation handle");
    FB_REQUIRE(!h->invalid, "interpolation handle is unusable: createReducedDomain failed while rebuilding its tables");
    const size_t in_level = h->inX * h->inY;
    FB_REQUIRE(in_level > 0, "interpolation with an empty source grid");
    *nz = size / in_level; // CachedInterpolation.cc:121: inZ = size / (inX*inY), remainder ignored
    return use_device(h->device);
}

// deltas of mifi_get_vector_reproject_matrix_proj (interpolation.c:458-513); both derive from the x field
int pick_deltas(const double* d_in_x, int ox, int oy, cudaStream_t st, double* dx, double* dy)
{
    auto fetch = [&](size_t idx, double* v) -> int {
        FB_CUDA_CHECK(cudaMemcpyAsync(v, d_in_x + idx, sizeof(double), cudaMemcpyDeviceToHost, st));
        return FB_OK;
    };
    const double eps = 1e-3;
    double a = 0, b = 0, c = 0, e = 0;
    volatile double d;
    if (ox > 1 && oy > 1) {
        const size_t hx = (size_t)ox / 2, hy = (size_t)oy / 2;
        if (fetch(0, &a) != FB_OK || fetch((size_t)ox + 1, &b) != FB_OK || fetch(hy * ox + hx, &c) != FB_OK ||
            fetch((hy + 1) * ox + (hx + 1), &e) != FB_OK)
            return FB_ERROR;
        FB_CUDA_CHECK(cudaStreamSynchronize(st));
        d = eps * (b - a);
        volatile double d2 = eps * (e - c);
        d = d + d2;
        d = d / 2;
    } else if (ox > 1) {
        if (fetch(0, &a) != FB_OK || fetch(1, &b) != FB_OK)
            return FB_ERROR;
        FB_CUDA_CHECK(cudaStreamSynchronize(st));
        d = eps * (b - a);
    } else if (oy > 1) {
        if (fetch(0, &a) != FB_OK || fetch((size_t)ox, &b) != FB_OK)
            return FB_ERROR;
        FB_CUDA_CHECK(cudaStreamSynchronize(st));
        d = eps * (b - a);
    } else {
        if (fetch(0, &a) != FB_OK)
            return FB_ERROR;
        FB_CUDA_CHECK(cudaStreamSynchronize(st));
        d = (a > 1) ? (a * eps) : eps;
    }
    *dx = d;
    *dy = d;
    if (std::fabs(*dx) < 1e-9 || std::fabs(*dy) < 1e-9) {
        fprintf(stderr, "WARNING, tiny deltaX/Y: %f %f possible singularity in vector-reprojection. Using default: %f\n", *dx, *dy, eps);
        *dx = eps;
        *dy = eps;
    }
    return FB_OK;
}

// the three matrix builders share this: d_matrix (device, 4*on) from axes/fields
enum MatrixInput { MI_AXES, MI_FIELD, MI_POINTS };
int build_matrix_device(MatrixInput kind, const char* proj_input, const char* proj_output, const double* a, const double* b, int xt, int yt,
                        int ox, int oy, int input_is_metric, double* d_matrix, cudaStream_t st)
{
    ProjDef pin, pout;
    if (parse_pair(proj_input, proj_output, &pin, &pout) != FB_OK)
        return FB_ERROR;
    const long long on = (kind == MI_POINTS) ? (long long)ox : (long long)ox * oy;
    if (on == 0)
        return FB_OK;
    Scratch tmp(st);
    int* d_status = nullptr;
    double *d_inx = nullptr, *d_iny = nullptr, *d_outx = nullptr, *d_outy = nullptr;
    if (tmp.get(&d_status, 1) != FB_OK || tmp.get(&d_inx, on) != FB_OK || tmp.get(&d_iny, on) != FB_OK || tmp.get(&d_outx, on) != FB_OK ||
        tmp.get(&d_outy, on) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    double dx, dy;
    if (kind == MI_AXES) {
        // interpolation.c:744-779: axes (deg->rad where typed so) -> mesh in the OUTPUT crs; in = out -> input crs
        const std::vector<double> xa = axis_in_radians(a, (size_t)ox, xt == FB_AXIS_LONGITUDE || xt == FB_AXIS_LATITUDE);
        const std::vector<double> ya = axis_in_radians(b, (size_t)oy, yt == FB_AXIS_LONGITUDE || yt == FB_AXIS_LATITUDE);
        double *d_xa = nullptr, *d_ya = nullptr;
        if (tmp.upload(&d_xa, xa.data(), xa.size()) != FB_OK || tmp.upload(&d_ya, ya.data(), ya.size()) != FB_OK)
            return FB_ERROR;
        ProjDef ident = pout; // identity "projection": mesh only
        ident.is_latlong = 1;
        ProjDef ident2 = ident;
        if (launch_project_mesh(ident, ident2, d_xa, d_ya, ox, oy, d_outx, d_outy, d_status, st) != FB_OK)
            return FB_ERROR;
        if (launch_project_mesh(pout, pin, d_xa, d_ya, ox, oy, d_inx, d_iny, d_status, st) != FB_OK)
            return FB_ERROR;
        if (check_status(d_status, st, "mifi_get_vector_reproject_matrix") != FB_OK)
            return FB_ERROR;
        if (pick_deltas(d_inx, ox, oy, st, &dx, &dy) != FB_OK)
            return FB_ERROR;
    } else if (kind == MI_FIELD) {
        // :697-708: in fields given (input crs); out = in -> output crs
        FB_CUDA_CHECK(cudaMemcpyAsync(d_inx, a, sizeof(double) * on, cudaMemcpyHostToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(d_iny, b, sizeof(double) * on, cudaMemcpyHostToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(d_outx, d_inx, sizeof(double) * on, cudaMemcpyDeviceToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(d_outy, d_iny, sizeof(double) * on, cudaMemcpyDeviceToDevice, st));
        if (launch_project_values(pin, pout, d_outx, d_outy, on, d_status, st) != FB_OK)
            return FB_ERROR;
        if (check_status(d_status, st, "mifi_get_vector_reproject_matrix_field") != FB_OK)
            return FB_ERROR;
        if (pick_deltas(d_inx, ox, oy, st, &dx, &dy) != FB_OK)
            return FB_ERROR;
    } else {
        // :641-656: out points given (output crs); in = out -> input crs; fixed delta
        FB_CUDA_CHECK(cudaMemcpyAsync(d_outx, a, sizeof(double) * on, cudaMemcpyHostToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(d_outy, b, sizeof(double) * on, cudaMemcpyHostToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(d_inx, d_outx, sizeof(double) * on, cudaMemcpyDeviceToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(d_iny, d_outy, sizeof(double) * on, cudaMemcpyDeviceToDevice, st));
        if (launch_project_values(pout, pin, d_inx, d_iny, on, d_status, st) != FB_OK)
            return FB_ERROR;
        if (check_status(d_status, st, "mifi_get_vector_reproject_matrix_points") != FB_OK)
            return FB_ERROR;
        dx = dy = input_is_metric ? 100 : 0.00001;
    }
    if (launch_vector_matrix(pin, pout, d_inx, d_iny, d_outx, d_outy, dx, dy, on, d_matrix, d_status, st) != FB_OK)
        return FB_ERROR;
    return check_status(d_status, st, "vector reprojection matrix");
}

int matrix_to_host(MatrixInput kind, const char* proj_input, const char* proj_output, const double* a, const double* b, int xt, int yt, int ox,
                   int oy, int metric, double* matrix)
{
    if (use_device(default_device()) != FB_OK)
        return FB_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    const long long on = (kind == MI_POINTS) ? (long long)ox : (long long)ox * oy;
    FB_REQUIRE(on >= 0 && (on == 0 || (a && b && matrix)), "null argument");
    Scratch tmp(st);
    double* d_m = nullptr;
    if (tmp.get(&d_m, 4 * (size_t)on) != FB_OK)
        return FB_ERROR;
    if (build_matrix_device(kind, proj_input, proj_output, a, b, xt, yt, ox, oy, metric, d_m, st) != FB_OK)
        return FB_ERROR;
    if (on) {
        FB_CUDA_CHECK(cudaMemcpyAsync(matrix, d_m, sizeof(double) * 4 * on, cudaMemcpyDeviceToHost, st));
        FB_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    return FB_OK;
}

// target axes -> (x, y) in `pdst` on the device: the mesh projection of mifi_project_axes
int project_axes_device(const ProjDef& psrc, const ProjDef& pdst, const std::vector<double>& xa, const std::vector<double>& ya, double* d_x,
                        double* d_y, cudaStream_t st, const char* what)
{
    Scratch tmp(st);
    int* d_status = nullptr;
    double *d_xa = nullptr, *d_ya = nullptr;
    if (tmp.get(&d_status, 1) != FB_OK || tmp.upload(&d_xa, xa.data(), xa.size()) != FB_OK || tmp.upload(&d_ya, ya.data(), ya.size()) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (launch_project_mesh(psrc, pdst, d_xa, d_ya, (int)xa.size(), (int)ya.size(), d_x, d_y, d_status, st) != FB_OK)
        return FB_ERROR;
    return check_status(d_status, st, what);
}

int points2position_device(double* d_pts, long long n, const std::vector<double>& axis, int type, cudaStream_t st)
{
    Scratch tmp(st);
    double* d_axis = nullptr;
    if (tmp.upload(&d_axis, axis.data(), axis.size()) != FB_OK)
        return FB_ERROR;
    if (launch_points2position(d_pts, n, d_axis, axis.data(), (int)axis.size(), type, st) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return FB_OK;
}

const char* kWgs84LatLon = "+proj=latlong +datum=WGS84 +towgs84=0,0,0 +no_defs"; // MIFI_WGS84_LATLON_PROJ4, CDMconstants.h:118

} // namespace

// ======================================================================================================
// extern "C"
// ======================================================================================================
extern "C" {

const char* fb200_version(void)
{
    return "fimex_b200 0.1 (path of fimex 0.67.2; sm_100a)";
}
const char* fb200_last_error(void)
{
    return last_error();
}
int fb200_set_device(int device)
{
    if (use_device(device) != FB_OK)
        return MIFI_ERROR;
    t_device = device;
    return MIFI_OK;
}
int fb200_get_device(void)
{
    return default_device();
}
unsigned long long fb200_kernel_launches(void)
{
    return launches();
}
} // extern "C"
namespace {
// Page-locked host buffers with a size-keyed free list.  Page-locking costs about as much as copying the buffer, so the
// buffers a host allocates per slice (interpolateValues returns a NEW array per call, src/CachedInterpolation.cc:123) are
// recycled instead of being unpinned: up to FIMEX_B200_PINNED_CACHE_MB stay cached (default: RAM / 8, at most 8192;
// fb200_host_trim() releases them).
struct PinnedCache {
    std::mutex mu;
    std::multimap<size_t, void*> free_blocks;      // capacity -> block
    std::unordered_map<void*, size_t> capacity_of; // every live block, cached or handed out
    size_t cached_bytes = 0;
    // FIMEX_B200_PINNED_CACHE_MB (parsed once, clamped to [0, physical RAM / 2]); default: an eighth of the physical RAM, at
    // most 8 GiB -- with 8 ranks per node the caches together stay within the RAM whatever the host has
    static size_t limit()
    {
        static const size_t value = []() {
            size_t phys = (size_t)64 << 30;
            const long pages = sysconf(_SC_PHYS_PAGES), page = sysconf(_SC_PAGE_SIZE);
            if (pages > 0 && page > 0)
                phys = (size_t)pages * (size_t)page;
            size_t lim = std::min<size_t>((size_t)8 << 30, phys / 8);
            if (const char* env = std::getenv("FIMEX_B200_PINNED_CACHE_MB")) {
                char* end = nullptr;
                const long long mb = std::strtoll(env, &end, 10);
                if (end != env && mb >= 0)
                    lim = std::min<size_t>((size_t)mb << 20, phys / 2);
            }
            return lim;
        }();
        return value;
    }
    void* get(size_t bytes)
    {
        const size_t want = ((bytes ? bytes : 1) + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1); // 2 MB granules
        {
            std::lock_guard<std::mutex> lock(mu);
            auto it = free_blocks.lower_bound(want);
            if (it != free_blocks.end() && it->first <= want + want / 4) { // do not burn a much larger block
                void* p = it->second;
                cached_bytes -= it->first;
                free_blocks.erase(it);
                return p;
            }
        }
        void* p = nullptr;
        if (cudaHostAlloc(&p, want, cudaHostAllocPortable) != cudaSuccess) {
            trim(0); // make room and retry once
            if (cudaHostAlloc(&p, want, cudaHostAllocPortable) != cudaSuccess)
                return nullptr;
        }
        std::lock_guard<std::mutex> lock(mu);
        capacity_of[p] = want;
        return p;
    }
    void put(void* p)
    {
        size_t cap = 0;
        {
            std::lock_guard<std::mutex> lock(mu);
            auto it = capacity_of.find(p);
            if (it == capacity_of.end()) { // not ours (or already released)
                // page-locked memory from elsewhere (cudaHostAlloc / cudaMallocHost) is released as such; anything else -- malloc,
                // new[], a device pointer, a pointer freed twice -- is left alone and reported instead of being handed to cudaFreeHost
                cudaPointerAttributes a;
                if (cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeHost) {
                    cudaFreeHost(p);
                } else {
                    cudaGetLastError();
                    set_error("fb200_host_free: pointer was not allocated by fb200_host_alloc (ignored)");
                }
                return;
            }
            cap = it->second;
            if (cached_bytes + cap <= limit()) {
                free_blocks.emplace(cap, p);
                cached_bytes += cap;
                return;
            }
            capacity_of.erase(it);
        }
        cudaFreeHost(p);
    }
    void trim(size_t keep_bytes)
    {
        std::vector<void*> victims;
        {
            std::lock_guard<std::mutex> lock(mu);
            while (cached_bytes > keep_bytes && !free_blocks.empty()) {
                auto it = std::prev(free_blocks.end());
                cached_bytes -= it->first;
                capacity_of.erase(it->second);
                victims.push_back(it->second);
                free_blocks.erase(it);
            }
        }
        for (void* p : victims)
            cudaFreeHost(p);
    }
};
PinnedCache& pinned_cache()
{
    static PinnedCache* c = new PinnedCache(); // leaked on purpose: no CUDA calls during static destruction
    return *c;
}
} // namespace
extern "C" {

void* fb200_host_alloc(size_t bytes)
{
    // Portable page-locked memory is usable from every device, so the calling thread's current device is left alone (a slice
    // call on a handle of another GPU asks for its bounce buffers from here, mid-call).  Only a thread that has never touched
    // CUDA gets the library's default device, because cudaHostAlloc needs some context.
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        set_error("no usable CUDA device (this library has no CPU fallback)");
        return nullptr;
    }
    void* p = pinned_cache().get(bytes);
    if (!p)
        set_error("cudaHostAlloc failed");
    return p;
}
void fb200_host_free(void* p)
{
    if (p)
        pinned_cache().put(p);
}
void fb200_host_trim(void)
{
    pinned_cache().trim(0);
}

// ---------------------------------------------------------------------------------------- CachedInterpolation
int fb200_cached_interpolation_create(int funcType, const double* px, const double* py, size_t inX, size_t inY, size_t outX, size_t outY,
                                      fb200_interp** handle)
{
    return create_from_points(funcType, false, px, py, false, inX, inY, outX, outY, handle);
}

int fb200_cached_interpolation_create_device(int funcType, const double* d_px, const double* d_py, size_t inX, size_t inY, size_t outX,
                                             size_t outY, fb200_interp** handle)
{
    return create_from_points(funcType, false, d_px, d_py, true, inX, inY, outX, outY, handle);
}

int fb200_cached_forward_interpolation_create(int funcType, const double* px, const double* py, size_t inX, size_t inY, size_t outX,
                                              size_t outY, fb200_interp** handle)
{
    return create_from_points(funcType, true, px, py, false, inX, inY, outX, outY, handle);
}

int fb200_cached_interpolation_create_from_projection(int funcType, const char* proj_target, const double* out_x_axis,
                                                      const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                      int out_y_is_degree, const char* proj_source, const double* in_x_axis,
                                                      const double* in_y_axis, size_t inX, size_t inY, int in_is_degree, fb200_interp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(funcType == FB_NN || funcType == FB_BILINEAR || funcType == FB_BICUBIC,
               "changeProjectionByProjectionParameters: method must be nearestneighbor, bilinear or bicubic");
    FB_REQUIRE(out_x_axis && out_y_axis && in_x_axis && in_y_axis, "null axis");
    ProjDef ptgt, psrc;
    if (parse_pair(proj_target, proj_source, &ptgt, &psrc) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_interp> h;
    if (new_interp(funcType, false, inX, inY, outX, outY, &h) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    const std::vector<double> oxa = axis_in_radians(out_x_axis, outX, out_x_is_degree != 0);
    const std::vector<double> oya = axis_in_radians(out_y_axis, outY, out_y_is_degree != 0);
    const std::vector<double> ixa = axis_in_radians(in_x_axis, inX, in_is_degree != 0);
    const std::vector<double> iya = axis_in_radians(in_y_axis, inY, in_is_degree != 0);
    if (h->npts) {
        if (project_axes_device(ptgt, psrc, oxa, oya, h->d_px, h->d_py, st, "mifi_project_axes") != FB_OK)
            return MIFI_ERROR;
        if (points2position_device(h->d_px, (long long)h->npts, ixa, in_is_degree ? FB_AXIS_LONGITUDE : FB_AXIS_PROJ, st) != FB_OK)
            return MIFI_ERROR;
        if (points2position_device(h->d_py, (long long)h->npts, iya, in_is_degree ? FB_AXIS_LATITUDE : FB_AXIS_PROJ, st) != FB_OK)
            return MIFI_ERROR;
    }
    if (compile_tables(h.get(), st) != FB_OK)
        return MIFI_ERROR;
    *handle = h.release();
    return MIFI_OK;
}

int fb200_cached_interpolation_create_from_template(int funcType, const char* proj_template, const double* tmplLon, const double* tmplLat,
                                                    size_t outX, size_t outY, const char* proj_source, const double* in_x_axis,
                                                    const double* in_y_axis, size_t inX, size_t inY, int in_is_degree, fb200_interp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(funcType == FB_NN || funcType == FB_BILINEAR || funcType == FB_BICUBIC,
               "changeProjectionByProjectionParametersToLatLonTemplate: method must be nearestneighbor, bilinear or bicubic");
    FB_REQUIRE(tmplLon && tmplLat && in_x_axis && in_y_axis, "null argument");
    ProjDef ptmpl, psrc;
    if (parse_pair(proj_template, proj_source, &ptmpl, &psrc) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_interp> h;
    if (new_interp(funcType, false, inX, inY, outX, outY, &h) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    const std::vector<double> lon = axis_in_radians(tmplLon, h->npts, true); // template data is in degrees (:1760-1763)
    const std::vector<double> lat = axis_in_radians(tmplLat, h->npts, true);
    const std::vector<double> ixa = axis_in_radians(in_x_axis, inX, in_is_degree != 0); // :1781-1786
    const std::vector<double> iya = axis_in_radians(in_y_axis, inY, in_is_degree != 0);
    if (h->npts) {
        Scratch tmp(st);
        int* d_status = nullptr;
        if (tmp.get(&d_status, 1) != FB_OK)
            return MIFI_ERROR;
        FB_CUDA_CHECK(cudaMemsetAsync(d_status, 0, sizeof(int), st));
        FB_CUDA_CHECK(cudaMemcpyAsync(h->d_px, lon.data(), sizeof(double) * h->npts, cudaMemcpyHostToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(h->d_py, lat.data(), sizeof(double) * h->npts, cudaMemcpyHostToDevice, st));
        if (launch_project_values(ptmpl, psrc, h->d_px, h->d_py, (long long)h->npts, d_status, st) != FB_OK) // :1770
            return MIFI_ERROR;
        if (check_status(d_status, st, "mifi_project_values") != FB_OK)
            return MIFI_ERROR;
        if (points2position_device(h->d_py, (long long)h->npts, iya, in_is_degree ? FB_AXIS_LATITUDE : FB_AXIS_PROJ, st) != FB_OK) // :1789
            return MIFI_ERROR;
        if (points2position_device(h->d_px, (long long)h->npts, ixa, in_is_degree ? FB_AXIS_LONGITUDE : FB_AXIS_PROJ, st) != FB_OK) // :1790
            return MIFI_ERROR;
    }
    if (compile_tables(h.get(), st) != FB_OK)
        return MIFI_ERROR;
    *handle = h.release();
    return MIFI_OK;
}

// getMaxDistanceOfInterest (src/CDMInterpolator.cc:304-326): the largest step of either output axis, in metres; axes whose
// unit is a degree are multiplied by the earth radius AS GIVEN (the reference passes the unconverted axis values)
static double max_distance_of_interest(const double* xa, size_t nx, const double* ya, size_t ny, bool is_metric)
{
    const double factor = is_metric ? 1. : 6371000.;
    double mx = 0., my = 0.;
    for (size_t i = 0; i + 1 < nx; ++i)
        mx = std::max(factor * std::fabs(xa[i + 1] - xa[i]), mx);
    for (size_t j = 0; j + 1 < ny; ++j)
        my = std::max(factor * std::fabs(ya[j + 1] - ya[j]), my);
    return std::max(mx, my);
}

int fb200_cached_interpolation_create_from_coordinates_kd(int funcType, const char* proj_target, const double* out_x_axis,
                                                          const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                          int out_y_is_degree, const double* lon2d, const double* lat2d, size_t inX,
                                                          size_t inY, double maxDistance, fb200_interp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(funcType == FB_COORD_NN || funcType == FB_COORD_NN_KD,
               "unkown interpolation method for coordinates: " + std::to_string(funcType)); // CDMInterpolator.cc:1410
    FB_REQUIRE(out_x_axis && out_y_axis && lon2d && lat2d, "null argument");
    ProjDef ptgt, pll;
    if (parse_pair(proj_target, kWgs84LatLon, &ptgt, &pll) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_interp> h;
    if (new_interp(funcType, false, inX, inY, outX, outY, &h) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    const std::vector<double> oxa = axis_in_radians(out_x_axis, outX, out_x_is_degree != 0);
    const std::vector<double> oya = axis_in_radians(out_y_axis, outY, out_y_is_degree != 0);
    const std::vector<double> lon = axis_in_radians(lon2d, inX * inY, true); // CDMInterpolator.cc:1358-1359
    const std::vector<double> lat = axis_in_radians(lat2d, inX * inY, true);
    if (h->npts) {
        if (project_axes_device(ptgt, pll, oxa, oya, h->d_px, h->d_py, st, "mifi_project_axes") != FB_OK)
            return MIFI_ERROR;
        if (funcType == FB_COORD_NN) {
            if (coordnn_search(h->d_px, h->d_py, (long long)h->npts, lon.data(), lat.data(), inX, inY, &h->coordnn_ties, st) != FB_OK)
                return MIFI_ERROR;
        } else {
            // isMetric follows the x axis' unit only (:1389-1393); p_->maxDistance > 0 overrides (:306)
            const double dist = maxDistance > 0. ? maxDistance : max_distance_of_interest(out_x_axis, outX, out_y_axis, outY, out_x_is_degree == 0);
            FB_REQUIRE(dist > 0., "coord_kdtree: maximum distance of interest is 0 (single-point axes); set one explicitly");
            if (coordkd_search(h->d_px, h->d_py, (long long)h->npts, lon.data(), lat.data(), inX, inY, dist, &h->coordnn_ties, st) != FB_OK)
                return MIFI_ERROR;
        }
    }
    if (compile_tables(h.get(), st) != FB_OK)
        return MIFI_ERROR;
    *handle = h.release();
    return MIFI_OK;
}

int fb200_cached_interpolation_create_from_coordinates(int funcType, const char* proj_target, const double* out_x_axis,
                                                       const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                       int out_y_is_degree, const double* lon2d, const double* lat2d, size_t inX, size_t inY,
                                                       fb200_interp** handle)
{
    return fb200_cached_interpolation_create_from_coordinates_kd(funcType, proj_target, out_x_axis, out_y_axis, outX, outY, out_x_is_degree,
                                                                 out_y_is_degree, lon2d, lat2d, inX, inY, 0., handle);
}

int fb200_cached_forward_interpolation_create_from_coordinates(int funcType, const char* proj_target, const double* out_x_axis,
                                                               const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                               int out_y_is_degree, const double* lon2d, const double* lat2d, size_t inX,
                                                               size_t inY, fb200_interp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(out_x_axis && out_y_axis && lon2d && lat2d, "null argument");
    ProjDef pll, ptgt;
    if (parse_pair(kWgs84LatLon, proj_target, &pll, &ptgt) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_interp> h;
    if (new_interp(funcType, true, inX, inY, outX, outY, &h) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    const std::vector<double> oxa = axis_in_radians(out_x_axis, outX, out_x_is_degree != 0);
    const std::vector<double> oya = axis_in_radians(out_y_axis, outY, out_y_is_degree != 0);
    const std::vector<double> lon = axis_in_radians(lon2d, inX * inY, true); // CDMInterpolator.cc:1265-1266
    const std::vector<double> lat = axis_in_radians(lat2d, inX * inY, true);
    if (h->npts) {
        Scratch tmp(st);
        int* d_status = nullptr;
        if (tmp.get(&d_status, 1) != FB_OK)
            return MIFI_ERROR;
        FB_CUDA_CHECK(cudaMemsetAsync(d_status, 0, sizeof(int), st));
        FB_CUDA_CHECK(cudaMemcpyAsync(h->d_px, lon.data(), sizeof(double) * h->npts, cudaMemcpyHostToDevice, st));
        FB_CUDA_CHECK(cudaMemcpyAsync(h->d_py, lat.data(), sizeof(double) * h->npts, cudaMemcpyHostToDevice, st));
        if (launch_project_values(pll, ptgt, h->d_px, h->d_py, (long long)h->npts, d_status, st) != FB_OK)
            return MIFI_ERROR;
        if (check_status(d_status, st, "mifi_project_values") != FB_OK)
            return MIFI_ERROR;
        if (points2position_device(h->d_px, (long long)h->npts, oxa, out_x_is_degree ? FB_AXIS_LONGITUDE : FB_AXIS_PROJ, st) != FB_OK)
            return MIFI_ERROR;
        if (points2position_device(h->d_py, (long long)h->npts, oya, out_y_is_degree ? FB_AXIS_LATITUDE : FB_AXIS_PROJ, st) != FB_OK)
            return MIFI_ERROR;
    }
    if (compile_tables(h.get(), st) != FB_OK)
        return MIFI_ERROR;
    *handle = h.release();
    return MIFI_OK;
}

int fb200_interp_create_reduced_domain(fb200_interp* h, int* reduced, long long* xMin, long long* yMin)
{
    FB_REQUIRE(h != nullptr, "null interpolation handle");
    if (reduced)
        *reduced = 0;
    FB_REQUIRE(!h->forward, "createReducedDomain is defined for CachedInterpolation only");
    FB_REQUIRE(!h->invalid, "interpolation handle is unusable: an earlier createReducedDomain failed");
    if (use_device(h->device) != FB_OK)
        return MIFI_ERROR;
    if (h->reduced) { // "don't set twice", CachedInterpolation.cc:161-163
        if (reduced)
            *reduced = 1;
        if (xMin)
            *xMin = h->xMin;
        if (yMin)
            *yMin = h->yMin;
        return MIFI_OK;
    }
    if (h->npts == 0)
        return MIFI_OK;
    cudaStream_t st = cudaStreamPerThread;
    double lox, hix, loy, hiy;
    if (device_minmax(h->d_px, (long long)h->npts, &lox, &hix, st) != FB_OK || device_minmax(h->d_py, (long long)h->npts, &loy, &hiy, st) != FB_OK)
        return MIFI_ERROR;
    auto clamp = [](long long lo, double dv, long long hi) { // CachedInterpolation.cc:149-157
        const long long v = static_cast<long long>(dv);
        if (v < lo)
            return lo;
        if (v < hi)
            return v;
        return hi;
    };
    const long long EXT = 2;
    const long long x0 = clamp(0, std::floor(lox) - EXT, (long long)h->inX - 1);
    const long long y0 = clamp(0, std::floor(loy) - EXT, (long long)h->inY - 1);
    const long long x1 = clamp(0, std::ceil(hix) + EXT, (long long)h->inX - 1);
    const long long y1 = clamp(0, std::ceil(hiy) + EXT, (long long)h->inY - 1);
    if ((x1 - x0) < 1 || (y1 - y0) < 1)
        return MIFI_OK;
    // from here on the handle is being rewritten (positions shifted, tables rebuilt): a failure leaves it unusable, and it
    // says so on every later call instead of gathering through freed tables
    h->invalid = true;
    if (launch_shift(h->d_px, (long long)h->npts, (double)x0, st) != FB_OK || launch_shift(h->d_py, (long long)h->npts, (double)y0, st) != FB_OK)
        return MIFI_ERROR;
    h->inX = (size_t)(x1 - x0 + 1);
    h->inY = (size_t)(y1 - y0 + 1);
    h->xMin = x0;
    h->yMin = y0;
    h->reduced = true;
    if (compile_tables(h, st) != FB_OK)
        return MIFI_ERROR;
    h->invalid = false;
    if (reduced)
        *reduced = 1;
    if (xMin)
        *xMin = x0;
    if (yMin)
        *yMin = y0;
    return MIFI_OK;
}

size_t fb200_interp_in_x(const fb200_interp* h)
{
    return h ? h->inX : 0;
}
size_t fb200_interp_in_y(const fb200_interp* h)
{
    return h ? h->inY : 0;
}
size_t fb200_interp_out_x(const fb200_interp* h)
{
    return h ? h->outX : 0;
}
size_t fb200_interp_out_y(const fb200_interp* h)
{
    return h ? h->outY : 0;
}
int fb200_interp_method(const fb200_interp* h)
{
    return h ? h->method : -1;
}

int fb200_interp_get_points(const fb200_interp* h, double* px, double* py)
{
    FB_REQUIRE(h != nullptr && px && py, "null argument");
    if (use_device(h->device) != FB_OK)
        return MIFI_ERROR;
    if (h->npts) {
        FB_CUDA_CHECK(cudaMemcpy(px, h->d_px, sizeof(double) * h->npts, cudaMemcpyDeviceToHost));
        FB_CUDA_CHECK(cudaMemcpy(py, h->d_py, sizeof(double) * h->npts, cudaMemcpyDeviceToHost));
    }
    return MIFI_OK;
}

int fb200_interp_device_points(const fb200_interp* h, const double** d_px, const double** d_py, size_t* n)
{
    FB_REQUIRE(h != nullptr, "null interpolation handle");
    if (d_px)
        *d_px = h->d_px;
    if (d_py)
        *d_py = h->d_py;
    if (n)
        *n = h->npts;
    return MIFI_OK;
}

size_t fb200_interp_new_size(const fb200_interp* h, size_t size)
{
    if (!h || h->inX * h->inY == 0)
        return 0;
    return h->outX * h->outY * (size / (h->inX * h->inY));
}

int fb200_interp_interpolate_values(const fb200_interp* h, const float* inData, size_t size, float* outData, size_t* newSize)
{
    size_t nz = 0;
    if (check_interp_call(h, size, &nz) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    FB_REQUIRE(nz == 0 || (inData && outData), "null data pointer");
    const float* in[1] = {inData};
    float* out[1] = {outData};
    return run_host(h, nullptr, 1, in, out, nz);
}

int fb200_interp_interpolate_values_device(const fb200_interp* h, const float* d_in, size_t size, float* d_out, size_t* newSize, void* stream)
{
    size_t nz = 0;
    if (check_interp_call(h, size, &nz) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    FB_REQUIRE(nz == 0 || (d_in && d_out), "null data pointer");
    return run_device(h, d_in, nz, d_out, as_stream(stream));
}

void fb200_interp_destroy(fb200_interp* h)
{
    delete h;
}

// ---------------------------------------------------------------------------------------- CachedVectorReprojection
int fb200_vector_create(int method, const double* matrix, int ox, int oy, fb200_vector** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(ox >= 0 && oy >= 0, "negative size");
    if (use_device(default_device()) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_vector> v(new fb200_vector());
    v->method = method;
    v->ox = ox;
    v->oy = oy;
    v->device = default_device();
    const size_t on = (size_t)ox * oy;
    if (on && matrix) { // an uninitialised reprojection (no matrix) is the identity, CachedVectorReprojection.cc:37-40
        cudaStream_t st = cudaStreamPerThread;
        if (dev_alloc(&v->d_matrix, 4 * on) != FB_OK || dev_alloc(&v->d_cs, on) != FB_OK)
            return MIFI_ERROR;
        FB_CUDA_CHECK(cudaMemcpyAsync(v->d_matrix, matrix, sizeof(double) * 4 * on, cudaMemcpyHostToDevice, st));
        if (launch_matrix_to_cossin(v->d_matrix, (long long)on, v->d_cs, st) != FB_OK)
            return MIFI_ERROR;
        FB_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    *handle = v.release();
    return MIFI_OK;
}

int fb200_vector_create_from_projection(int method, const char* proj_input, const char* proj_output, const double* out_x_axis,
                                        const double* out_y_axis, int xt, int yt, int ox, int oy, fb200_vector** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(ox > 0 && oy > 0 && out_x_axis && out_y_axis, "empty target grid");
    if (use_device(default_device()) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_vector> v(new fb200_vector());
    v->method = method;
    v->ox = ox;
    v->oy = oy;
    v->device = default_device();
    const size_t on = (size_t)ox * oy;
    cudaStream_t st = cudaStreamPerThread;
    if (dev_alloc(&v->d_matrix, 4 * on) != FB_OK || dev_alloc(&v->d_cs, on) != FB_OK)
        return MIFI_ERROR;
    if (build_matrix_device(MI_AXES, proj_input, proj_output, out_x_axis, out_y_axis, xt, yt, ox, oy, 0, v->d_matrix, st) != FB_OK)
        return MIFI_ERROR;
    if (launch_matrix_to_cossin(v->d_matrix, (long long)on, v->d_cs, st) != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = v.release();
    return MIFI_OK;
}

int fb200_vector_create_from_points(int method, const char* proj_input, const char* proj_output, int inputIsMetric, const double* lon,
                                    const double* lat, int on, fb200_vector** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(on > 0 && lon && lat, "empty point list");
    if (use_device(default_device()) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_vector> v(new fb200_vector());
    v->method = method;
    v->ox = on; // CachedVectorReprojection(MIFI_VECTOR_KEEP_SIZE, matrix, outSize, 1), CDMInterpolator.cc:1823
    v->oy = 1;
    v->device = default_device();
    cudaStream_t st = cudaStreamPerThread;
    if (dev_alloc(&v->d_matrix, 4 * (size_t)on) != FB_OK || dev_alloc(&v->d_cs, (size_t)on) != FB_OK)
        return MIFI_ERROR;
    const std::vector<double> lo = axis_in_radians(lon, (size_t)on, true); // template data is in degrees (:1810-1813)
    const std::vector<double> la = axis_in_radians(lat, (size_t)on, true);
    if (build_matrix_device(MI_POINTS, proj_input, proj_output, lo.data(), la.data(), 0, 0, on, 1, inputIsMetric, v->d_matrix, st) != FB_OK)
        return MIFI_ERROR;
    if (launch_matrix_to_cossin(v->d_matrix, (long long)on, v->d_cs, st) != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = v.release();
    return MIFI_OK;
}

int fb200_vector_create_from_grid(int method, const char* proj, const double* x_axis, const double* y_axis, int nx, int ny, int isDegree,
                                  int toLatLon, fb200_vector** handle)
{
    // makeCachedVectorReprojection (src/CDMProcessor.cc:99-145): the matrix of a grid's own axes, towards geographic
    // directions (toLatLon: matrix_field on the expanded mesh) or back (matrix from WGS84 lat/long to the grid's CRS, with
    // MIFI_PROJ_AXIS "even for LAT/LON since axes already in radian")
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(nx > 0 && ny > 0 && x_axis && y_axis && proj, "empty grid");
    if (use_device(default_device()) != FB_OK)
        return MIFI_ERROR;
    std::unique_ptr<fb200_vector> v(new fb200_vector());
    v->method = method;
    v->ox = nx;
    v->oy = ny;
    v->device = default_device();
    const size_t on = (size_t)nx * ny;
    cudaStream_t st = cudaStreamPerThread;
    if (dev_alloc(&v->d_matrix, 4 * on) != FB_OK || dev_alloc(&v->d_cs, on) != FB_OK)
        return MIFI_ERROR;
    const std::vector<double> xa = axis_in_radians(x_axis, (size_t)nx, isDegree != 0);
    const std::vector<double> ya = axis_in_radians(y_axis, (size_t)ny, isDegree != 0);
    if (toLatLon) {
        std::vector<double> xf(on), yf(on);
        for (int j = 0; j < ny; ++j)
            for (int i = 0; i < nx; ++i) {
                xf[(size_t)nx * j + i] = xa[i];
                yf[(size_t)nx * j + i] = ya[j];
            }
        if (build_matrix_device(MI_FIELD, proj, kWgs84LatLon, xf.data(), yf.data(), 0, 0, nx, ny, 0, v->d_matrix, st) != FB_OK)
            return MIFI_ERROR;
    } else if (build_matrix_device(MI_AXES, kWgs84LatLon, proj, xa.data(), ya.data(), MIFI_PROJ_AXIS, MIFI_PROJ_AXIS, nx, ny, 0, v->d_matrix, st) !=
               FB_OK) {
        return MIFI_ERROR;
    }
    if (launch_matrix_to_cossin(v->d_matrix, (long long)on, v->d_cs, st) != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = v.release();
    return MIFI_OK;
}

int fb200_vector_reproject_values_device(const fb200_vector* v, float* d_u, float* d_v, size_t size, void* stream)
{
    FB_REQUIRE(v != nullptr, "null vector handle");
    if (v->ox == 0 || v->oy == 0 || v->d_cs == nullptr) {
        fprintf(stderr, "fimex_b200: CachedVectorReprojection not initialized, using identity\n");
        return MIFI_OK;
    }
    if (use_device(v->device) != FB_OK)
        return MIFI_ERROR;
    const long long layer = (long long)v->ox * v->oy;
    return launch_rotate(v->d_cs, d_u, d_v, layer, (long long)(size / (size_t)layer), as_stream(stream));
}

int fb200_vector_reproject_values(const fb200_vector* v, float* u, float* vv, size_t size)
{
    FB_REQUIRE(v != nullptr, "null vector handle");
    if (v->ox == 0 || v->oy == 0 || v->d_cs == nullptr) {
        fprintf(stderr, "fimex_b200: CachedVectorReprojection not initialized, using identity\n");
        return MIFI_OK;
    }
    if (use_device(v->device) != FB_OK)
        return MIFI_ERROR;
    const size_t layer = (size_t)v->ox * v->oy;
    const size_t n = (size / layer) * layer;
    if (n == 0)
        return MIFI_OK;
    FB_REQUIRE(u && vv, "null data pointer");
    cudaStream_t st = cudaStreamPerThread;
    Scratch tmp(st);
    float *d_u = nullptr, *d_v = nullptr;
    if (tmp.upload(&d_u, u, n) != FB_OK || tmp.upload(&d_v, vv, n) != FB_OK)
        return MIFI_ERROR;
    if (launch_rotate(v->d_cs, d_u, d_v, (long long)layer, (long long)(n / layer), st) != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(u, d_u, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(vv, d_v, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return MIFI_OK;
}

int fb200_vector_reproject_direction_values(const fb200_vector* v, float* angles, size_t size)
{
    FB_REQUIRE(v != nullptr, "null vector handle");
    if (v->ox == 0 || v->oy == 0 || v->d_matrix == nullptr) {
        fprintf(stderr, "fimex_b200: CachedVectorReprojection not initialized, using identity\n");
        return MIFI_OK;
    }
    if (use_device(v->device) != FB_OK)
        return MIFI_ERROR;
    const size_t layer = (size_t)v->ox * v->oy;
    const size_t n = (size / layer) * layer;
    if (n == 0)
        return MIFI_OK;
    cudaStream_t st = cudaStreamPerThread;
    Scratch tmp(st);
    float* d_a = nullptr;
    if (tmp.upload(&d_a, angles, n) != FB_OK)
        return MIFI_ERROR;
    if (launch_rotate_direction(v->d_matrix, d_a, (long long)layer, (long long)(n / layer), st) != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(angles, d_a, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return MIFI_OK;
}

int fb200_vector_get_matrix(const fb200_vector* v, double* matrix)
{
    FB_REQUIRE(v != nullptr && matrix, "null argument");
    if (use_device(v->device) != FB_OK)
        return MIFI_ERROR;
    if (v->d_matrix)
        FB_CUDA_CHECK(cudaMemcpy(matrix, v->d_matrix, sizeof(double) * 4 * (size_t)v->ox * v->oy, cudaMemcpyDeviceToHost));
    return MIFI_OK;
}

void fb200_vector_destroy(fb200_vector* v)
{
    delete v;
}

static int check_vector_call(const fb200_interp* h, const fb200_vector* v)
{
    FB_REQUIRE(h != nullptr, "null interpolation handle");
    FB_REQUIRE(!h->forward, "vector data cannot be interpolated with forward interpolation"); // CDMInterpolator.cc:1332
    if (v && v->d_cs)
        FB_REQUIRE((size_t)v->ox == h->outX && (size_t)v->oy == h->outY && v->device == h->device,
                   "vector reprojection and interpolation have different target grids or devices");
    return FB_OK;
}

int fb200_interp_interpolate_vector_device(const fb200_interp* h, const fb200_vector* v, const float* d_u, const float* d_v, size_t size,
                                           float* d_uo, float* d_vo, size_t* newSize, void* stream)
{
    size_t nz = 0;
    if (check_vector_call(h, v) != FB_OK || check_interp_call(h, size, &nz) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    return run_vector_device(h, (v && v->d_cs) ? v : nullptr, d_u, d_v, nz, d_uo, d_vo, as_stream(stream));
}

int fb200_interp_interpolate_vector(const fb200_interp* h, const fb200_vector* v, const float* uIn, const float* vIn, size_t size, float* uOut,
                                    float* vOut, size_t* newSize)
{
    size_t nz = 0;
    if (check_vector_call(h, v) != FB_OK || check_interp_call(h, size, &nz) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    FB_REQUIRE(nz == 0 || (uIn && vIn && uOut && vOut), "null data pointer");
    const float* in[2] = {uIn, vIn};
    float* out[2] = {uOut, vOut};
    return run_host(h, (v && v->d_cs) ? v : nullptr, 2, in, out, nz);
}

// ---------------------------------------------------------------------------------------- interpolate.preprocess / postprocess
} // extern "C"
namespace {
// string2type<T> of the reference (include/fimex/Utils.h:60-67): stream extraction; here a failed extraction is an error
template <class T>
bool parse_token(const std::string& s, T* out)
{
    std::istringstream in(s);
    in >> *out;
    return !in.fail();
}

// parseProcess, src/binSrc/fimex.cc:644-671
int parse_process(const char* procString, fb200_interp::Process* p)
{
    FB_REQUIRE(procString != nullptr, "null process string");
    std::string s(procString);
    size_t b = s.find_first_not_of(" \t\n\r");
    s = b == std::string::npos ? std::string() : s.substr(b);
    auto args_of = [&](const char* name, std::string* args) {
        const std::string head = std::string(name) + "(";
        if (s.compare(0, head.size(), head) != 0)
            return false;
        const size_t close = s.rfind(')');
        if (close == std::string::npos || close < head.size())
            return false;
        *args = s.substr(head.size(), close - head.size());
        return true;
    };
    auto split = [](const std::string& a) {
        std::vector<std::string> out;
        size_t start = 0;
        while (true) {
            const size_t c = a.find(',', start);
            out.push_back(a.substr(start, c == std::string::npos ? std::string::npos : c - start));
            if (c == std::string::npos)
                break;
            start = c + 1;
        }
        return out;
    };
    std::string args;
    if (args_of("fill2d", &args)) {
        const std::vector<std::string> v = split(args);
        double critx = 0, cor = 0;
        size_t maxLoop = 0;
        FB_REQUIRE(v.size() == 3 && parse_token(v[0], &critx) && parse_token(v[1], &cor) && parse_token(v[2], &maxLoop),
                   "undefined interpolate process: " + s + " (fill2d(critx,cor,maxLoop))");
        p->kind = 0;
        p->relaxCrit = (float)critx;
        p->corrEff = (float)cor;
        p->maxLoop = maxLoop;
        return FB_OK;
    }
    if (args_of("creepfill2d", &args)) {
        const std::vector<std::string> v = split(args);
        FB_REQUIRE(v.size() == 2 || v.size() == 3, "creepfill requires two or three arguments, got " + args);
        unsigned short repeat = 0;
        char weight = 0; // string2type<char> extracts ONE CHARACTER: "2" is the weight 50 ('2'), exactly as in the reference (:657)
        FB_REQUIRE(parse_token(v[0], &repeat) && parse_token(v[1], &weight), "undefined interpolate process: " + s);
        p->kind = 1;
        p->repeat = repeat;
        p->weight = (signed char)weight;
        if (v.size() == 3) {
            float defVal = 0.f;
            FB_REQUIRE(parse_token(v[2], &defVal), "undefined interpolate process: " + s);
            p->kind = 2;
            p->defVal = defVal;
        }
        return FB_OK;
    }
    FB_REQUIRE(false, "undefined interpolate process: " + s);
}
} // namespace
extern "C" {

int fb200_interp_add_preprocess(fb200_interp* h, const char* procString)
{
    FB_REQUIRE(h != nullptr, "null interpolation handle");
    fb200_interp::Process p;
    if (parse_process(procString, &p) != FB_OK)
        return MIFI_ERROR;
    h->preprocesses.push_back(p);
    return MIFI_OK;
}

int fb200_interp_add_postprocess(fb200_interp* h, const char* procString)
{
    FB_REQUIRE(h != nullptr, "null interpolation handle");
    fb200_interp::Process p;
    if (parse_process(procString, &p) != FB_OK)
        return MIFI_ERROR;
    h->postprocesses.push_back(p);
    return MIFI_OK;
}

// ---------------------------------------------------------------------------------------- getDataSlice in one call
static int check_slice_types(int inType, int outType)
{
    FB_REQUIRE(known_type(inType), "unsupported input data type " + std::to_string(inType));
    FB_REQUIRE(known_type(outType), "unsupported output data type " + std::to_string(outType));
    return FB_OK;
}

int fb200_interp_get_data_slice_device(const fb200_interp* h, int inType, const void* d_in, size_t size, double badValue, int outType,
                                       void* d_out, size_t* newSize, void* stream)
{
    size_t nz = 0;
    if (check_interp_call(h, size, &nz) != FB_OK || check_slice_types(inType, outType) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    FB_REQUIRE(nz == 0 || (d_in && d_out), "null data pointer");
    SliceIO io;
    io.typed = true;
    io.in_type = inType;
    io.out_type = outType;
    io.bad[0] = badValue;
    const void* in[1] = {d_in};
    void* out[1] = {d_out};
    return run_slice_device(h, nullptr, 1, in, nz, out, io, as_stream(stream));
}

int fb200_interp_get_data_slice(const fb200_interp* h, int inType, const void* inData, size_t size, double badValue, int outType,
                                void* outData, size_t* newSize)
{
    size_t nz = 0;
    if (check_interp_call(h, size, &nz) != FB_OK || check_slice_types(inType, outType) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    FB_REQUIRE(nz == 0 || (inData && outData), "null data pointer");
    SliceIO io;
    io.typed = true;
    io.in_type = inType;
    io.out_type = outType;
    io.bad[0] = badValue;
    const void* in[1] = {inData};
    void* out[1] = {outData};
    return run_slice_host(h, nullptr, 1, in, out, nz, io);
}

int fb200_interp_get_vector_slice_device(const fb200_interp* h, const fb200_vector* v, int inType, const void* d_u, const void* d_v, size_t size,
                                         double badU, double badV, int outType, void* d_uo, void* d_vo, size_t* newSize, void* stream)
{
    size_t nz = 0;
    if (check_vector_call(h, v) != FB_OK || check_interp_call(h, size, &nz) != FB_OK || check_slice_types(inType, outType) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    FB_REQUIRE(nz == 0 || (d_u && d_v && d_uo && d_vo), "null data pointer");
    SliceIO io;
    io.typed = true;
    io.in_type = inType;
    io.out_type = outType;
    io.bad[0] = badU;
    io.bad[1] = badV;
    const void* in[2] = {d_u, d_v};
    void* out[2] = {d_uo, d_vo};
    return run_slice_device(h, (v && v->d_cs) ? v : nullptr, 2, in, nz, out, io, as_stream(stream));
}

int fb200_interp_get_vector_slice(const fb200_interp* h, const fb200_vector* v, int inType, const void* uIn, const void* vIn, size_t size,
                                  double badU, double badV, int outType, void* uOut, void* vOut, size_t* newSize)
{
    size_t nz = 0;
    if (check_vector_call(h, v) != FB_OK || check_interp_call(h, size, &nz) != FB_OK || check_slice_types(inType, outType) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = h->outX * h->outY * nz;
    FB_REQUIRE(nz == 0 || (uIn && vIn && uOut && vOut), "null data pointer");
    SliceIO io;
    io.typed = true;
    io.in_type = inType;
    io.out_type = outType;
    io.bad[0] = badU;
    io.bad[1] = badV;
    const void* in[2] = {uIn, vIn};
    void* out[2] = {uOut, vOut};
    return run_slice_host(h, (v && v->d_cs) ? v : nullptr, 2, in, out, nz, io);
}

int fb200_vector_get_slice_device(const fb200_vector* v, int inType, const void* d_u, const void* d_v, size_t size, double badU, double badV,
                                  int outType, void* d_uo, void* d_vo, void* stream)
{
    // the rotation branch of CDMProcessor::getDataSlice (src/CDMProcessor.cc:579-617): both components fill -> NaN as float,
    // reprojectValues, NaN -> fill + cast back -- no gather in between
    FB_REQUIRE(v != nullptr, "null vector handle");
    if (check_slice_types(inType, outType) != FB_OK)
        return MIFI_ERROR;
    if (size == 0)
        return MIFI_OK;
    FB_REQUIRE(d_u && d_v && d_uo && d_vo, "null data pointer");
    if (use_device(v->device) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = as_stream(stream);
    Scratch tmp(st);
    float *fu = nullptr, *fv = nullptr;
    if (tmp.get(&fu, size) != FB_OK || tmp.get(&fv, size) != FB_OK)
        return MIFI_ERROR;
    const float bu = (float)badU, bv = (float)badV;
    if (launch_as_float(inType, d_u, (long long)size, !std::isnan(bu), bu, fu, st) != FB_OK ||
        launch_as_float(inType, d_v, (long long)size, !std::isnan(bv), bv, fv, st) != FB_OK)
        return MIFI_ERROR;
    if (v->ox == 0 || v->oy == 0 || v->d_cs == nullptr) {
        fprintf(stderr, "fimex_b200: CachedVectorReprojection not initialized, using identity\n"); // CachedVectorReprojection.cc:37-40
    } else {
        const long long layer = (long long)v->ox * v->oy;
        if (launch_rotate(v->d_cs, fu, fv, layer, (long long)(size / (size_t)layer), st) != FB_OK)
            return MIFI_ERROR;
    }
    if (launch_from_float(fu, (long long)size, outType, badU, d_uo, st) != FB_OK ||
        launch_from_float(fv, (long long)size, outType, badV, d_vo, st) != FB_OK)
        return MIFI_ERROR;
    return MIFI_OK;
}

int fb200_vector_get_slice(const fb200_vector* v, int inType, const void* uIn, const void* vIn, size_t size, double badU, double badV,
                           int outType, void* uOut, void* vOut)
{
    FB_REQUIRE(v != nullptr, "null vector handle");
    if (check_slice_types(inType, outType) != FB_OK)
        return MIFI_ERROR;
    if (size == 0)
        return MIFI_OK;
    FB_REQUIRE(uIn && vIn && uOut && vOut, "null data pointer");
    if (use_device(v->device) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    Scratch tmp(st);
    const size_t ib = size * type_size(inType), ob = size * type_size(outType);
    char *d_u = nullptr, *d_v = nullptr, *d_uo = nullptr, *d_vo = nullptr;
    if (tmp.upload(&d_u, static_cast<const char*>(uIn), ib) != FB_OK || tmp.upload(&d_v, static_cast<const char*>(vIn), ib) != FB_OK ||
        tmp.get(&d_uo, ob) != FB_OK || tmp.get(&d_vo, ob) != FB_OK)
        return MIFI_ERROR;
    if (fb200_vector_get_slice_device(v, inType, d_u, d_v, size, badU, badV, outType, d_uo, d_vo, st) != MIFI_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(uOut, d_uo, ob, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(vOut, d_vo, ob, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return MIFI_OK;
}

} // extern "C"

// ======================================================================================================
// vertical interpolation to pressure levels (the pressure branch of CDMVerticalInterpolator), to height and altitude levels
// (its height branch) and to depth levels (its depth branch)
// ======================================================================================================
// Depth handles reuse two slots of fb200_vcolumns: ps carries the sea surface height eta, zs the sea-floor depth.
struct fb200_vinterp {
    int device = 0;
    bool has_ps = false;   // the column pressures depend on the surface pressure (hybrid or sigma levels), and the converter uses them;
                           // depth handles of the ocean coordinates: eta is read when given (it is optional: NULL means 0)
    bool needs_t = false;  // height handles: the hypsometric converter integrates the air temperature (and q, when given)
    bool needs_z = false;  // the field converter reads the altitude field z
    bool needs_zs = false; // the surface altitude: height targets of the standard and field converters, altitude targets of the hypsometric one;
                           // depth handles of the ocean coordinates: they need the sea-floor depth
    fb::VertTable vt;
    ~fb200_vinterp()
    {
        fb::DeviceGuard on(device);
        if (vt.d_tab)
            cudaFree(vt.d_tab);
    }
};

namespace {

constexpr int kMaxVertLevels = 1024; // the coefficient table of one handle stays below 48 KB of shared memory

bool all_finite(const double* v, int n)
{
    for (int i = 0; i < n; ++i)
        if (!std::isfinite(v[i]))
            return false;
    return true;
}

// the targets in ascending order into lev[np], and the output row of each into row[np]
void sort_targets(const double* levels, int np, double* lev, double* row)
{
    std::vector<int> order(np);
    for (int i = 0; i < np; ++i)
        order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return levels[x] < levels[y]; });
    for (int i = 0; i < np; ++i) {
        lev[i] = levels[order[i]];
        row[i] = order[i];
    }
}

int upload_table(VertTable& vt, const std::vector<double>& tab, cudaStream_t st)
{
    if (dev_alloc(&vt.d_tab, tab.size()) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(vt.d_tab, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice, st));
    return FB_OK;
}

// p_k = a_k + b_k * (ps * ps_scale - shift): hybrid a = ap, shift 0; sigma a = ptop, b = sigma, shift = ptop; pressure levels b = 0
int vinterp_create(int method, const double* a, const double* b, int nk, bool sigma, double ptop, double ps_scale, const double* levels, int np,
                   int extrapolate, fb200_vinterp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(method >= FB_VINT_LIN && method <= FB_VINT_NN, "unknown vertical interpolation method " + std::to_string(method));
    FB_REQUIRE(nk >= 2 && nk <= kMaxVertLevels, "number of source levels must be in [2, 1024], got " + std::to_string(nk));
    FB_REQUIRE(np >= 1 && np <= kMaxVertLevels, "number of target levels must be in [1, 1024], got " + std::to_string(np));
    FB_REQUIRE(levels != nullptr, "null target levels");
    FB_REQUIRE(all_finite(levels, np), "target levels must be finite");
    FB_REQUIRE(a != nullptr, sigma ? "null sigma" : "null ap (or pressure levels)");
    FB_REQUIRE(all_finite(a, nk) && (b == nullptr || all_finite(b, nk)), "vertical coordinate values must be finite");
    FB_REQUIRE(std::isfinite(ps_scale) && std::isfinite(ptop), "ps_scale and ptop must be finite");
    if (use_device(default_device()) != FB_OK)
        return FB_ERROR;
    std::unique_ptr<fb200_vinterp> h(new fb200_vinterp());
    h->device = default_device();
    h->has_ps = sigma || b != nullptr;
    VertTable& vt = h->vt;
    vt.method = method;
    vt.nk = nk;
    vt.np = np;
    vt.extrapolate = extrapolate != 0;
    vt.ps_scale = ps_scale;
    vt.shift = sigma ? ptop : 0.0;
    std::vector<double> tab(2 * (size_t)nk + 3 * (size_t)np, 0.0);
    for (int k = 0; k < nk; ++k) {
        tab[k] = sigma ? ptop : a[k];
        tab[nk + k] = sigma ? a[k] : (b ? b[k] : 0.0);
    }
    double* lev = tab.data() + 2 * nk;
    sort_targets(levels, np, lev, lev + 2 * np);
    cudaStream_t st = cudaStreamPerThread;
    if (upload_table(vt, tab, st) != FB_OK)
        return FB_ERROR;
    if (launch_vert_coords(method, vt.d_tab + 2 * nk, vt.d_tab + 2 * nk + np, np, st) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = h.release();
    return FB_OK;
}

// The standard atmosphere (US Standard Atmosphere 1976 / ICAO): geopotential layers with base altitude h_b [m], base temperature
// T_b [K], lapse rate L_b [K/m] and the published base pressure p_b [hPa]; the gas constant R* [J/(mol K)], the molar masses of dry
// air M and of water M_w [kg/mol], g0 [m/s2].  tests/vertical_height_oracle.c forms the same constants with the same expressions.
constexpr double kStdH[kStdLayers] = {0.0, 11000.0, 20000.0, 32000.0, 47000.0, 51000.0, 71000.0};
constexpr double kStdT[kStdLayers] = {288.15, 216.65, 216.65, 228.65, 270.65, 270.65, 214.65};
constexpr double kStdL[kStdLayers] = {-6.5e-3, 0.0, 1e-3, 2.8e-3, 0.0, -2.8e-3, -2e-3};
constexpr double kStdP[kStdLayers] = {1013.25, 226.3206, 54.74889, 8.680187, 1.109063, 0.6693887, 0.03956420};
constexpr double kRstar = 8.31432, kMair = 0.0289644, kMwater = 0.01801528, kG0 = 9.80665;

// the a | b terms of p_k = a_k + b_k * (ps * ps_scale - shift) from the formula terms of FB200_VCOORD_PRESSURE (a = the levels),
// _HYBRID (a = ap, b) or _SIGMA (b = sigma; a_k = shift = ptop) into tab[0 .. 2 nk)
void pressure_terms(int vcoord, const double* a, const double* b, int nk, double ptop, double* tab)
{
    const bool sigma = vcoord == FB200_VCOORD_SIGMA, hybrid = vcoord == FB200_VCOORD_HYBRID;
    for (int k = 0; k < nk; ++k) {
        tab[k] = sigma ? ptop : a[k];
        tab[nk + k] = (sigma || hybrid) ? b[k] : 0.0;
    }
}

int vinterp_create_height(int method, int converter, int target, int vcoord, const double* a, const double* b, int nk, double ptop,
                          double ps_scale, double z_scale, double zs_scale, const double* levels, int np, int extrapolate, fb200_vinterp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(method == FB_VINT_LIN || method == FB_VINT_NN,
               "height levels take the methods linear and nearestneighbor only (log and loglog are defined on ln p), got " + std::to_string(method));
    FB_REQUIRE(converter >= FB_VZ_STANDARD && converter <= FB_VZ_FIELD, "unknown height converter " + std::to_string(converter));
    FB_REQUIRE(target == FB_VZ_ALTITUDE || target == FB_VZ_HEIGHT, "unknown height target " + std::to_string(target));
    const bool field = converter == FB_VZ_FIELD;
    FB_REQUIRE(field || (vcoord >= FB200_VCOORD_PRESSURE && vcoord <= FB200_VCOORD_SIGMA), "unknown source vertical coordinate " + std::to_string(vcoord));
    FB_REQUIRE(converter != FB_VZ_HYPSOMETRIC || vcoord != FB200_VCOORD_PRESSURE,
               "the hypsometric converter needs a surface pressure: hybrid or sigma source levels, not pressure levels");
    FB_REQUIRE(nk >= 2 && nk <= kMaxVertLevels, "number of source levels must be in [2, 1024], got " + std::to_string(nk));
    FB_REQUIRE(np >= 1 && np <= kMaxVertLevels, "number of target levels must be in [1, 1024], got " + std::to_string(np));
    FB_REQUIRE(levels != nullptr, "null target levels");
    FB_REQUIRE(all_finite(levels, np), "target levels must be finite");
    const bool sigma = vcoord == FB200_VCOORD_SIGMA, hybrid = vcoord == FB200_VCOORD_HYBRID;
    if (!field) { // the field converter does not use the source's formula terms
        FB_REQUIRE(sigma || a != nullptr, "null ap (or pressure levels)");
        FB_REQUIRE(!(sigma || hybrid) || b != nullptr, sigma ? "null sigma" : "null b");
        FB_REQUIRE((sigma || all_finite(a, nk)) && (!(sigma || hybrid) || all_finite(b, nk)), "vertical coordinate values must be finite");
    }
    FB_REQUIRE(std::isfinite(ps_scale) && std::isfinite(ptop) && std::isfinite(z_scale) && std::isfinite(zs_scale),
               "ps_scale, ptop, z_scale and zs_scale must be finite");
    if (use_device(default_device()) != FB_OK)
        return FB_ERROR;
    std::unique_ptr<fb200_vinterp> h(new fb200_vinterp());
    h->device = default_device();
    h->has_ps = converter == FB_VZ_HYPSOMETRIC || (converter == FB_VZ_STANDARD && vcoord != FB200_VCOORD_PRESSURE);
    h->needs_t = converter == FB_VZ_HYPSOMETRIC;
    h->needs_z = field;
    h->needs_zs = (target == FB_VZ_HEIGHT) != (converter == FB_VZ_HYPSOMETRIC);
    VertTable& vt = h->vt;
    vt.method = method;
    vt.nk = nk;
    vt.np = np;
    vt.extrapolate = extrapolate != 0;
    vt.ps_scale = ps_scale;
    vt.shift = sigma ? ptop : 0.0;
    vt.converter = converter;
    vt.target = target;
    vt.z_scale = z_scale;
    vt.zs_scale = zs_scale;
    vt.H = kRstar / (kMair * kG0);
    vt.cq = kMair / kMwater - 1.0;
    std::vector<double> tab(2 * (size_t)nk + 4 * kStdLayers + 2 * (size_t)np, 0.0);
    if (!field)
        pressure_terms(vcoord, a, b, nk, ptop, tab.data());
    double* layers = tab.data() + 2 * nk; // h_b | p_b | c_b | e_b
    for (int l = 0; l < kStdLayers; ++l) {
        layers[l] = kStdH[l];
        layers[kStdLayers + l] = kStdP[l];
        layers[2 * kStdLayers + l] = kStdL[l] != 0.0 ? kStdT[l] / kStdL[l] : vt.H * kStdT[l];
        layers[3 * kStdLayers + l] = kStdL[l] != 0.0 ? -(kRstar * kStdL[l]) / (kG0 * kMair) : 0.0;
    }
    double* lev = layers + 4 * kStdLayers;
    sort_targets(levels, np, lev, lev + np);
    cudaStream_t st = cudaStreamPerThread;
    if (upload_table(vt, tab, st) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = h.release();
    return FB_OK;
}

// ocean_sigma_coordinate, ocean_s_coordinate_g1 / _g2 or depth levels: x_k = -z_k from the terms s (sigma_k, s_k or the levels), C and
// depth_c; the table holds s (depth levels, sigma) or dcs_k = depth_c * s_k (g1, g2), and C
int vinterp_create_depth(int method, int vcoord, const double* s, const double* Ck, int nk, double depth_c, const double* levels, int np, int extrapolate,
                         fb200_vinterp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(method == FB_VINT_LIN || method == FB_VINT_NN,
               "depth levels take the methods linear and nearestneighbor only (log and loglog are defined on ln p), got " + std::to_string(method));
    FB_REQUIRE(vcoord >= FB_VD_DEPTH && vcoord <= FB_VD_OCEAN_S_G2, "unknown depth source vertical coordinate " + std::to_string(vcoord));
    const bool g = vcoord == FB_VD_OCEAN_S_G1 || vcoord == FB_VD_OCEAN_S_G2;
    FB_REQUIRE(nk >= 2 && nk <= kMaxVertLevels, "number of source levels must be in [2, 1024], got " + std::to_string(nk));
    FB_REQUIRE(np >= 1 && np <= kMaxVertLevels, "number of target levels must be in [1, 1024], got " + std::to_string(np));
    FB_REQUIRE(levels != nullptr, "null target levels");
    FB_REQUIRE(all_finite(levels, np), "target levels must be finite");
    FB_REQUIRE(s != nullptr, vcoord == FB_VD_DEPTH ? "null depth levels" : vcoord == FB_VD_OCEAN_SIGMA ? "null sigma" : "null s");
    FB_REQUIRE(!g || Ck != nullptr, "null C: ocean_s_coordinate_g1 and _g2 need the stretching function C");
    FB_REQUIRE(all_finite(s, nk) && (!g || all_finite(Ck, nk)), "vertical coordinate values must be finite");
    FB_REQUIRE(std::isfinite(depth_c) && depth_c >= 0.0, "depth_c must be finite and >= 0");
    if (use_device(default_device()) != FB_OK)
        return FB_ERROR;
    std::unique_ptr<fb200_vinterp> h(new fb200_vinterp());
    h->device = default_device();
    h->has_ps = vcoord != FB_VD_DEPTH;
    h->needs_zs = vcoord != FB_VD_DEPTH;
    VertTable& vt = h->vt;
    vt.method = method;
    vt.nk = nk;
    vt.np = np;
    vt.extrapolate = extrapolate != 0;
    vt.depth_vcoord = vcoord;
    vt.depth_c = depth_c;
    std::vector<double> tab(2 * (size_t)nk + 2 * (size_t)np, 0.0);
    for (int k = 0; k < nk; ++k) {
        tab[k] = g ? depth_c * s[k] : s[k];
        tab[nk + k] = g ? Ck[k] : 0.0;
    }
    double* lev = tab.data() + 2 * nk;
    sort_targets(levels, np, lev, lev + np);
    cudaStream_t st = cudaStreamPerThread;
    if (upload_table(vt, tab, st) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = h.release();
    return FB_OK;
}

int check_vinterp_call(const fb200_vinterp* h, const void* in, const fb200_vcolumns& cols, size_t nxy, size_t nt, const void* out)
{
    FB_REQUIRE(h != nullptr, "null vertical interpolation handle");
    FB_REQUIRE(nxy * nt == 0 || (in && out), "null data pointer");
    if (nxy * nt != 0) {
        const bool depth = h->vt.depth_vcoord != FB_VD_NONE;
        FB_REQUIRE(!h->has_ps || cols.ps || depth, "this vertical coordinate needs the surface pressure ps"); // eta is optional
        FB_REQUIRE(!h->needs_t || cols.t, "the hypsometric converter needs the air temperature t");
        FB_REQUIRE(!h->needs_z || cols.z, "the field converter needs the altitude field z");
        FB_REQUIRE(!h->needs_zs || cols.zs,
                   depth ? "ocean s- and sigma coordinates need the sea-floor depth (the zs slot of fb200_vcolumns; the calls without _columns cannot pass it)"
                         : "this converter and target need the surface altitude zs");
    }
    return use_device(h->device);
}

fb200_vcolumns ps_only(const float* ps)
{
    fb200_vcolumns cols = {};
    cols.ps = ps;
    return cols;
}

// typed: data2InterpolationArray (any CDM type, fill -> NaN) before and interpolationArray2Data (NaN -> fill, cast) after, both as
// separate passes; untyped: float in, float out.  cols: device pointers.
int vinterp_device(const fb200_vinterp* h, bool typed, int in_type, const void* d_in, const fb200_vcolumns& cols, size_t nxy, size_t nt,
                   double bad, int out_type, void* d_out, cudaStream_t st)
{
    if (nxy == 0 || nt == 0)
        return FB_OK;
    const size_t in_n = nxy * nt * (size_t)h->vt.nk, out_n = nxy * nt * (size_t)h->vt.np;
    Scratch tmp(st);
    const float* fin = static_cast<const float*>(d_in);
    const bool has_bad = typed && !std::isnan((float)bad); // mifi_bad2nanf takes a float
    if (typed && (in_type != FB_T_FLOAT || has_bad)) {
        float* conv = nullptr;
        if (tmp.get(&conv, in_n) != FB_OK || launch_as_float(in_type, d_in, (long long)in_n, has_bad, (float)bad, conv, st) != FB_OK)
            return FB_ERROR;
        fin = conv;
    }
    float* fout = static_cast<float*>(d_out);
    if (typed && out_type != FB_T_FLOAT && tmp.get(&fout, out_n) != FB_OK)
        return FB_ERROR;
    const float* ps = h->has_ps ? cols.ps : nullptr;
    const float* zs = h->needs_zs ? cols.zs : nullptr;
    const int rc = h->vt.depth_vcoord != FB_VD_NONE ? launch_vertical_depth(h->vt, fin, ps, zs, (long long)nxy, (long long)nt, fout, st)
                   : h->vt.converter == FB_VZ_NONE
                       ? launch_vertical(h->vt, fin, ps, (long long)nxy, (long long)nt, fout, st)
                       : launch_vertical_height(h->vt, fin, ps, h->needs_t ? cols.t : nullptr, h->needs_t ? cols.q : nullptr,
                                                h->needs_z ? cols.z : nullptr, zs, (long long)nxy, (long long)nt, fout, st);
    if (rc != FB_OK)
        return FB_ERROR;
    if (typed)
        return launch_from_float(fout, (long long)out_n, out_type, bad, d_out, st);
    return FB_OK;
}

// host arrays: time steps are the units of the staging pipeline of the horizontal calls; the field and up to three per-step inputs
// (ps, t, q or z) go through it, zs (no time axis) is uploaded once per call; for depth handles these are eta and the sea-floor depth
int vinterp_host(const fb200_vinterp* h, bool typed, int in_type, const void* in, const fb200_vcolumns& cols, size_t nxy, size_t nt, double bad,
                 int out_type, void* out)
{
    if (nxy == 0 || nt == 0)
        return FB_OK;
    const size_t level = nxy * sizeof(float), column = level * (size_t)h->vt.nk;
    HostArrays arrays;
    arrays.device = h->device;
    arrays.in[0] = in;
    arrays.in_unit[0] = nxy * (size_t)h->vt.nk * type_size(in_type);
    const float* steps[4] = {h->has_ps ? cols.ps : nullptr, h->needs_t ? cols.t : nullptr, h->needs_t ? cols.q : nullptr,
                             h->needs_z ? cols.z : nullptr};
    const size_t unit[4] = {level, column, column, column};
    int slot[4] = {-1, -1, -1, -1};
    for (int i = 0, n = 1; i < 4; ++i) {
        if (!steps[i])
            continue;
        FB_REQUIRE(n < kHostIn, "too many per-step inputs");
        slot[i] = n;
        arrays.in[n] = steps[i];
        arrays.in_unit[n++] = unit[i];
    }
    arrays.out[0] = out;
    arrays.out_unit[0] = nxy * (size_t)h->vt.np * type_size(out_type);
    cudaStream_t st = cudaStreamPerThread;
    Scratch tmp(st); // freed after stage_host has returned, when every kernel that read it is complete
    float* d_zs = nullptr;
    if (h->needs_zs) {
        if (tmp.upload(&d_zs, cols.zs, nxy) != FB_OK)
            return FB_ERROR;
        FB_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    return stage_host(arrays, nt, [&](const void* const* d_in, size_t n, void* const* d_out, cudaStream_t s) {
        auto arg = [&](int i) { return slot[i] < 0 ? nullptr : static_cast<const float*>(d_in[slot[i]]); };
        fb200_vcolumns dc = {arg(0), arg(1), arg(2), arg(3), d_zs};
        return vinterp_device(h, typed, in_type, d_in[0], dc, nxy, n, bad, out_type, d_out[0], s);
    });
}

const fb200_vcolumns& or_none(const fb200_vcolumns* cols)
{
    static const fb200_vcolumns none = {};
    return cols ? *cols : none;
}

} // namespace

// ======================================================================================================
// the data conversions of the vertical interpolator (CDMPressureConversions: theta2T, omega2vwind, add4Dpressure), on the model levels
// ======================================================================================================
struct fb200_vconvert {
    int device = 0;
    int op = 0, vcoord = 0;
    bool has_ps = false; // hybrid or sigma levels
    double kappa = 0.0;  // R_d / c_pd of theta2T
    fb::VertTable vt;    // a | b, ps_scale, shift and H (omega2vwind) as for the pressure and height handles; np = 0
    ~fb200_vconvert()
    {
        fb::DeviceGuard on(device);
        if (vt.d_tab)
            cudaFree(vt.d_tab);
    }
};

namespace {

int vconvert_create(int op, int vcoord, const double* a, const double* b, int nk, double ptop, double ps_scale, fb200_vconvert** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(op >= FB_VCONV_THETA2T && op <= FB_VCONV_PRESSURE, "unknown data conversion " + std::to_string(op));
    FB_REQUIRE(vcoord >= FB200_VCOORD_PRESSURE && vcoord <= FB200_VCOORD_SIGMA, "unknown source vertical coordinate " + std::to_string(vcoord));
    FB_REQUIRE(nk >= 1 && nk <= kMaxVertLevels, "number of levels must be in [1, 1024], got " + std::to_string(nk));
    const bool sigma = vcoord == FB200_VCOORD_SIGMA, hybrid = vcoord == FB200_VCOORD_HYBRID;
    FB_REQUIRE(sigma || a != nullptr, "null ap (or pressure levels)");
    FB_REQUIRE(!(sigma || hybrid) || b != nullptr, sigma ? "null sigma" : "null b");
    FB_REQUIRE((sigma || all_finite(a, nk)) && (!(sigma || hybrid) || all_finite(b, nk)), "vertical coordinate values must be finite");
    FB_REQUIRE(std::isfinite(ps_scale) && std::isfinite(ptop), "ps_scale and ptop must be finite");
    if (use_device(default_device()) != FB_OK)
        return FB_ERROR;
    std::unique_ptr<fb200_vconvert> h(new fb200_vconvert());
    h->device = default_device();
    h->op = op;
    h->vcoord = vcoord;
    h->has_ps = sigma || hybrid;
    h->kappa = 2.0 / 7.0; // R_d / c_pd of an ideal diatomic gas, c_pd = 3.5 R_d
    VertTable& vt = h->vt;
    vt.nk = nk;
    vt.ps_scale = ps_scale;
    vt.shift = sigma ? ptop : 0.0;
    vt.H = kRstar / (kMair * kG0); // H g0 = R* / M = R_d
    std::vector<double> tab(2 * (size_t)nk, 0.0);
    pressure_terms(vcoord, a, b, nk, ptop, tab.data());
    cudaStream_t st = cudaStreamPerThread;
    if (upload_table(vt, tab, st) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = h.release();
    return FB_OK;
}

int check_vconvert_call(const fb200_vconvert* h, const void* in, const fb200_vcolumns& cols, size_t nxy, size_t nt, const void* out)
{
    FB_REQUIRE(h != nullptr, "null data conversion handle");
    if (nxy * nt != 0) {
        FB_REQUIRE(out && (in || h->op == FB_VCONV_PRESSURE), "null data pointer");
        FB_REQUIRE(!h->has_ps || cols.ps, "this vertical coordinate needs the surface pressure ps");
        FB_REQUIRE(h->op != FB_VCONV_OMEGA2VWIND || cols.t, "omega2vwind needs the air temperature t");
    }
    return use_device(h->device);
}

int vconvert_device(const fb200_vconvert* h, const float* d_in, const fb200_vcolumns& cols, size_t nxy, size_t nt, float* d_out, cudaStream_t st)
{
    return launch_vconvert(h->op, h->vcoord, h->vt, h->kappa, h->op == FB_VCONV_PRESSURE ? nullptr : d_in, h->has_ps ? cols.ps : nullptr,
                           h->op == FB_VCONV_OMEGA2VWIND ? cols.t : nullptr, (long long)nxy, (long long)nt, d_out, st);
}

// host arrays: time steps are the units of the staging pipeline; the field, ps and t are its inputs where the conversion reads them
int vconvert_host(const fb200_vconvert* h, const float* in, const fb200_vcolumns& cols, size_t nxy, size_t nt, float* out)
{
    if (nxy == 0 || nt == 0)
        return FB_OK;
    const size_t level = nxy * sizeof(float), column = level * (size_t)h->vt.nk;
    const float* steps[3] = {h->op == FB_VCONV_PRESSURE ? nullptr : in, h->has_ps ? cols.ps : nullptr, h->op == FB_VCONV_OMEGA2VWIND ? cols.t : nullptr};
    const size_t unit[3] = {column, level, column};
    HostArrays arrays;
    arrays.device = h->device;
    for (int i = 0; i < 3; ++i) {
        arrays.in[i] = steps[i];
        arrays.in_unit[i] = steps[i] ? unit[i] : 0;
    }
    arrays.out[0] = out;
    arrays.out_unit[0] = column;
    return stage_host(arrays, nt, [&](const void* const* d_in, size_t n, void* const* d_out, cudaStream_t s) {
        fb200_vcolumns dc = {};
        dc.ps = static_cast<const float*>(d_in[1]);
        dc.t = static_cast<const float*>(d_in[2]);
        return vconvert_device(h, static_cast<const float*>(d_in[0]), dc, nxy, n, static_cast<float*>(d_out[0]), s);
    });
}

} // namespace

// ======================================================================================================
// time interpolation (CDMTimeInterpolator's linear change of the time axis)
// ======================================================================================================
struct fb200_tinterp {
    int device = 0;
    int nt = 0, nj = 0;
    std::vector<TimeStep> map;    // [nj] in target order: lower source step ia (-1: no bracket), weight w
    TimeStep* d_sorted = nullptr; // [nj] the targets by ia, those without a bracket last: the table of the stack call
    TimeStep* d_single = nullptr; // [nj] {0 (-1: no bracket), row 0, w_j}: the one-target tables of the step calls
    ~fb200_tinterp()
    {
        fb::DeviceGuard on(device);
        if (d_sorted)
            cudaFree(d_sorted);
        if (d_single)
            cudaFree(d_single);
    }
};

namespace {

constexpr int kMaxTimeTargets = 1 << 20;

int tinterp_create(const double* times, int nt, const double* new_times, int nj, int extrapolate, fb200_tinterp** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(nt >= 2, "number of source times must be at least 2, got " + std::to_string(nt));
    FB_REQUIRE(nj >= 1 && nj <= kMaxTimeTargets, "number of target times must be in [1, 1048576], got " + std::to_string(nj));
    FB_REQUIRE(times != nullptr && new_times != nullptr, "null time axis");
    FB_REQUIRE(all_finite(times, nt) && all_finite(new_times, nj), "times must be finite");
    for (int k = 0; k + 1 < nt; ++k)
        FB_REQUIRE(times[k] < times[k + 1], "source times must be strictly increasing");
    if (use_device(default_device()) != FB_OK)
        return FB_ERROR;
    std::unique_ptr<fb200_tinterp> h(new fb200_tinterp());
    h->device = default_device();
    h->nt = nt;
    h->nj = nj;
    h->map.resize(nj);
    std::vector<TimeStep> single(nj);
    for (int j = 0; j < nj; ++j) {
        const double tau = new_times[j];
        int k = -1;
        if (tau < times[0] || tau > times[nt - 1]) {
            if (extrapolate)
                k = tau < times[0] ? 0 : nt - 2; // the end pair on that side
        } else { // the smallest k with t_k <= tau <= t_k+1
            k = (int)(std::lower_bound(times, times + nt, tau) - times) - 1;
            k = k < 0 ? 0 : k;
        }
        const double w = k < 0 ? 0.0 : (tau - times[k]) / (times[k + 1] - times[k]);
        h->map[j] = TimeStep{k, j, w};
        single[j] = TimeStep{k < 0 ? -1 : 0, 0, w};
    }
    std::vector<TimeStep> sorted(h->map);
    std::stable_sort(sorted.begin(), sorted.end(), [](const TimeStep& x, const TimeStep& y) { return (unsigned)x.ia < (unsigned)y.ia; });
    cudaStream_t st = cudaStreamPerThread;
    if (dev_alloc(&h->d_sorted, nj) != FB_OK || dev_alloc(&h->d_single, nj) != FB_OK)
        return FB_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(h->d_sorted, sorted.data(), sizeof(TimeStep) * nj, cudaMemcpyHostToDevice, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(h->d_single, single.data(), sizeof(TimeStep) * nj, cudaMemcpyHostToDevice, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    *handle = h.release();
    return FB_OK;
}

// stack: the whole-stack call (j is not used); otherwise the step call of target j
int check_tinterp_call(const fb200_tinterp* h, bool stack, int j, int in_type, int out_type, size_t n, const void* a, const void* b, const void* out)
{
    FB_REQUIRE(h != nullptr, "null time interpolation handle");
    if (check_slice_types(in_type, out_type) != FB_OK)
        return FB_ERROR;
    FB_REQUIRE(stack || (j >= 0 && j < h->nj), "target step " + std::to_string(j) + " out of range [0, " + std::to_string(h->nj) + ")");
    const bool reads = stack || h->map[j].ia >= 0; // a target without a bracket reads no source step
    FB_REQUIRE(n == 0 || (out && (!reads || (a && b))), "null data pointer");
    return use_device(h->device);
}

bool has_bad_value(double bad)
{
    return !std::isnan((float)bad); // mifi_bad2nanf takes a float
}

// host buffers: elements are the units of the staging pipeline; a and b are its inputs (absent for a target without a bracket)
int tinterp_get_step_host(const fb200_tinterp* h, int j, int in_type, const void* a, const void* b, size_t n, double bad, int out_type, void* out)
{
    if (n == 0)
        return FB_OK;
    HostArrays arrays;
    arrays.device = h->device;
    if (h->map[j].ia >= 0) {
        arrays.in[0] = a;
        arrays.in[1] = b;
        arrays.in_unit[0] = arrays.in_unit[1] = type_size(in_type);
    }
    arrays.out[0] = out;
    arrays.out_unit[0] = type_size(out_type);
    return stage_host(arrays, n, [&](const void* const* d_in, size_t cnt, void* const* d_out, cudaStream_t s) {
        return launch_tinterp(in_type, d_in[0], d_in[1], (long long)cnt, has_bad_value(bad), (float)bad, h->d_single + j, 1, out_type, bad, d_out[0], s);
    });
}

} // namespace

// ======================================================================================================
// merger (CDMMerger: the inner grid blended into the outer one at its border, then laid over the outer one on a target grid)
// ======================================================================================================
struct fb200_merge {
    const fb200_interp* o2i = nullptr; // outer -> inner grid; all three are borrowed: the caller keeps them alive
    const fb200_interp* i2t = nullptr; // inner -> target grid
    const fb200_interp* o2t = nullptr; // outer -> target grid
    int device = 0;
    size_t innerX = 0, innerY = 0, outerX = 0, outerY = 0;
    int t = 0, b = 0; // transition and border width of CDMBorderSmoothing_Linear
    bool use_outer = true;
};

namespace {

// The device chain works through the levels in chunks whose float intermediates (the outer slab cropped to one handle's domain,
// the outer field on the inner grid, the smoothed window, the top and base fields on the target grid) take at most this many bytes,
// or one level where a single level is larger: a whole stack never needs a second copy of itself in scratch.
constexpr size_t kMergeScratchBytes = 256ull << 20;

std::string grid_str(size_t x, size_t y)
{
    return std::to_string(x) + " x " + std::to_string(y);
}

int check_merge_handle(const fb200_interp* h, const char* which, size_t srcX, size_t srcY, const char* src_name)
{
    FB_REQUIRE(h != nullptr, std::string("null ") + which + " interpolation handle");
    FB_REQUIRE(!h->forward && (h->method == FB_NN || h->method == FB_BILINEAR || h->method == FB_BICUBIC),
               std::string("the ") + which + " handle must interpolate with nearest neighbour, bilinear or bicubic (method " + std::to_string(h->method) + ")");
    FB_REQUIRE(h->srcX == srcX && h->srcY == srcY,
               std::string("the ") + which + " handle reads a " + grid_str(h->srcX, h->srcY) + " grid, the " + src_name + " grid is " + grid_str(srcX, srcY));
    return FB_OK;
}

int merge_create(const fb200_interp* o2i, const fb200_interp* i2t, const fb200_interp* o2t, size_t innerX, size_t innerY, size_t outerX, size_t outerY,
                 int t, int b, int use_outer, fb200_merge** handle)
{
    FB_REQUIRE(handle != nullptr, "null handle pointer");
    *handle = nullptr;
    FB_REQUIRE(t >= 1, "transition width must be at least 1 (the linear border smoothing divides by it), got " + std::to_string(t));
    FB_REQUIRE(b >= 0, "border width must not be negative, got " + std::to_string(b));
    FB_REQUIRE(innerX > 0 && innerY > 0 && outerX > 0 && outerY > 0, "empty inner or outer grid");
    if (check_merge_handle(o2i, "outer -> inner", outerX, outerY, "outer") != FB_OK || check_merge_handle(i2t, "inner -> target", innerX, innerY, "inner") != FB_OK ||
        check_merge_handle(o2t, "outer -> target", outerX, outerY, "outer") != FB_OK)
        return FB_ERROR;
    FB_REQUIRE(o2i->outX == innerX && o2i->outY == innerY,
               "the outer -> inner handle writes a " + grid_str(o2i->outX, o2i->outY) + " grid, the inner grid is " + grid_str(innerX, innerY));
    FB_REQUIRE(i2t->outX == o2t->outX && i2t->outY == o2t->outY, "the inner -> target handle writes a " + grid_str(i2t->outX, i2t->outY) +
                                                                      " grid, the outer -> target handle a " + grid_str(o2t->outX, o2t->outY) + " grid");
    FB_REQUIRE(o2i->device == i2t->device && o2i->device == o2t->device, "the three interpolation handles live on different devices");
    std::unique_ptr<fb200_merge> h(new fb200_merge());
    h->o2i = o2i;
    h->i2t = i2t;
    h->o2t = o2t;
    h->device = o2i->device;
    h->innerX = innerX;
    h->innerY = innerY;
    h->outerX = outerX;
    h->outerY = outerY;
    h->t = t;
    h->b = b;
    h->use_outer = use_outer != 0;
    *handle = h.release();
    return FB_OK;
}

// both sizes must hold the same whole number of levels of their grid; *nz receives it
int check_merge_call(const fb200_merge* h, int in_type, int out_type, size_t inner_size, size_t outer_size, const void* inner, const void* outer,
                     const void* out, size_t* nz)
{
    FB_REQUIRE(h != nullptr, "null merge handle");
    FB_REQUIRE(!h->o2i->invalid && !h->i2t->invalid && !h->o2t->invalid,
               "an interpolation handle of the merger is unusable: createReducedDomain failed while rebuilding its tables");
    if (check_slice_types(in_type, out_type) != FB_OK)
        return FB_ERROR;
    const size_t il = h->innerX * h->innerY, ol = h->outerX * h->outerY;
    FB_REQUIRE(inner_size % il == 0, "inner size " + std::to_string(inner_size) + " is not a whole number of " + grid_str(h->innerX, h->innerY) + " levels");
    FB_REQUIRE(outer_size % ol == 0, "outer size " + std::to_string(outer_size) + " is not a whole number of " + grid_str(h->outerX, h->outerY) + " levels");
    *nz = inner_size / il;
    FB_REQUIRE(outer_size / ol == *nz, "inner has " + std::to_string(*nz) + " levels, outer " + std::to_string(outer_size / ol));
    FB_REQUIRE(*nz == 0 || (inner && outer && out), "null data pointer");
    return use_device(h->device);
}

size_t merge_target_level(const fb200_merge* h)
{
    return h->i2t->outX * h->i2t->outY;
}

// crop + convert, outer -> inner gather, smoothing, inner -> target gather, crop + convert, outer -> target gather, overlay: all on st
int merge_device(const fb200_merge* h, int in_type, const void* d_inner, double bad_inner, const void* d_outer, double bad_outer, size_t nz, int out_type,
                 double out_fill, void* d_out, cudaStream_t st)
{
    const fb200_interp *o2i = h->o2i, *i2t = h->i2t, *o2t = h->o2t;
    const size_t inner_lvl = h->innerX * h->innerY, outer_lvl = h->outerX * h->outerY, target_lvl = merge_target_level(h);
    if (nz == 0 || target_lvl == 0)
        return FB_OK;
    const size_t crop_lvl = std::max(o2i->inX * o2i->inY, o2t->inX * o2t->inY); // one buffer: the two crops are used one after the other
    const size_t smooth_lvl = i2t->inX * i2t->inY;
    const size_t per_level = sizeof(float) * (crop_lvl + inner_lvl + smooth_lvl + 2 * target_lvl);
    const size_t zc = std::min(nz, std::max<size_t>(1, kMergeScratchBytes / per_level));
    Scratch tmp(st);
    float *crop = nullptr, *on_inner = nullptr, *smooth = nullptr, *top = nullptr, *base = nullptr;
    if (tmp.get(&crop, zc * crop_lvl) != FB_OK || tmp.get(&on_inner, zc * inner_lvl) != FB_OK || tmp.get(&smooth, zc * smooth_lvl) != FB_OK ||
        tmp.get(&top, zc * target_lvl) != FB_OK || tmp.get(&base, zc * target_lvl) != FB_OK)
        return FB_ERROR;
    SliceIO io; // the gathers as getDataSlice on float with NaN = undefined both ways (pre/postprocesses of a handle apply)
    io.typed = true;
    io.bad[0] = std::numeric_limits<double>::quiet_NaN();
    auto gather = [&](const fb200_interp* g, const float* in, size_t zn, float* out) {
        const void* i[1] = {in};
        void* o[1] = {out};
        return run_slice_device(g, nullptr, 1, i, zn, o, io, st);
    };
    const bool outer_has_bad = has_bad_value(bad_outer), inner_has_bad = !std::isnan(bad_inner);
    const size_t in_elem = type_size(in_type), out_elem = type_size(out_type);
    for (size_t z0 = 0; z0 < nz; z0 += zc) {
        const size_t zn = std::min(zc, nz - z0);
        const char* inner = static_cast<const char*>(d_inner) + z0 * inner_lvl * in_elem;
        const char* outer = static_cast<const char*>(d_outer) + z0 * outer_lvl * in_elem;
        char* out = static_cast<char*>(d_out) + z0 * target_lvl * out_elem;
        if (launch_crop_as_float(in_type, outer, h->outerX, h->outerY, o2i->xMin, o2i->yMin, o2i->inX, o2i->inY, zn, outer_has_bad, (float)bad_outer, crop,
                                 st) != FB_OK ||
            gather(o2i, crop, zn, on_inner) != FB_OK ||
            launch_border_smooth_linear(in_type, inner, inner_has_bad, bad_inner, on_inner, h->innerX, h->innerY, h->t, h->b, h->use_outer, i2t->xMin,
                                        i2t->yMin, i2t->inX, i2t->inY, zn, smooth, st) != FB_OK ||
            gather(i2t, smooth, zn, top) != FB_OK ||
            launch_crop_as_float(in_type, outer, h->outerX, h->outerY, o2t->xMin, o2t->yMin, o2t->inX, o2t->inY, zn, outer_has_bad, (float)bad_outer, crop,
                                 st) != FB_OK ||
            gather(o2t, crop, zn, base) != FB_OK || launch_merge_overlay(top, base, (long long)(zn * target_lvl), out_type, out_fill, out, st) != FB_OK)
            return FB_ERROR;
    }
    return FB_OK;
}

// host buffers: inner and outer go up once and the merged slice comes down once, pipelined over level chunks
int merge_host(const fb200_merge* h, int in_type, const void* inner, double bad_inner, const void* outer, double bad_outer, size_t nz, int out_type,
               double out_fill, void* out)
{
    const size_t target_lvl = merge_target_level(h);
    if (nz == 0 || target_lvl == 0)
        return FB_OK;
    HostArrays arrays;
    arrays.device = h->device;
    arrays.in[0] = inner;
    arrays.in_unit[0] = h->innerX * h->innerY * type_size(in_type);
    arrays.in[1] = outer;
    arrays.in_unit[1] = h->outerX * h->outerY * type_size(in_type);
    arrays.out[0] = out;
    arrays.out_unit[0] = target_lvl * type_size(out_type);
    return stage_host(arrays, nz, [&](const void* const* d_in, size_t zn, void* const* d_o, cudaStream_t s) {
        return merge_device(h, in_type, d_in[0], bad_inner, d_in[1], bad_outer, zn, out_type, out_fill, d_o[0], s);
    });
}

} // namespace

extern "C" {

int fb200_vinterp_create_hybrid(int method, const double* ap, const double* b, int nk, double ps_scale, const double* levels, int np,
                                int extrapolate, fb200_vinterp** handle)
{
    return vinterp_create(method, ap, b, nk, false, 0.0, ps_scale, levels, np, extrapolate, handle) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_vinterp_create_sigma(int method, const double* sigma, int nk, double ptop, double ps_scale, const double* levels, int np, int extrapolate,
                               fb200_vinterp** handle)
{
    return vinterp_create(method, sigma, nullptr, nk, true, ptop, ps_scale, levels, np, extrapolate, handle) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_vinterp_create_height(int method, int converter, int target, int vcoord, const double* a, const double* b, int nk, double ptop,
                                double ps_scale, double z_scale, double zs_scale, const double* levels, int np, int extrapolate,
                                fb200_vinterp** handle)
{
    return vinterp_create_height(method, converter, target, vcoord, a, b, nk, ptop, ps_scale, z_scale, zs_scale, levels, np, extrapolate, handle) ==
                   FB_OK
               ? MIFI_OK
               : MIFI_ERROR;
}

int fb200_vinterp_create_depth(int method, int vcoord, const double* s, const double* C, int nk, double depth_c, const double* levels, int np,
                               int extrapolate, fb200_vinterp** handle)
{
    return vinterp_create_depth(method, vcoord, s, C, nk, depth_c, levels, np, extrapolate, handle) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

void fb200_vinterp_destroy(fb200_vinterp* h)
{
    delete h;
}

int fb200_vinterp_interpolate_values(const fb200_vinterp* h, const float* in, const float* ps, size_t nxy, size_t nt, float* out)
{
    const fb200_vcolumns cols = ps_only(ps);
    return fb200_vinterp_interpolate_values_columns(h, in, &cols, nxy, nt, out);
}

int fb200_vinterp_interpolate_values_device(const fb200_vinterp* h, const float* d_in, const float* d_ps, size_t nxy, size_t nt, float* d_out,
                                            void* stream)
{
    const fb200_vcolumns cols = ps_only(d_ps);
    return fb200_vinterp_interpolate_values_columns_device(h, d_in, &cols, nxy, nt, d_out, stream);
}

int fb200_vinterp_get_data_slice(const fb200_vinterp* h, int inType, const void* in, const float* ps, size_t nxy, size_t nt, double badValue,
                                 int outType, void* out)
{
    const fb200_vcolumns cols = ps_only(ps);
    return fb200_vinterp_get_data_slice_columns(h, inType, in, &cols, nxy, nt, badValue, outType, out);
}

int fb200_vinterp_get_data_slice_device(const fb200_vinterp* h, int inType, const void* d_in, const float* d_ps, size_t nxy, size_t nt,
                                        double badValue, int outType, void* d_out, void* stream)
{
    const fb200_vcolumns cols = ps_only(d_ps);
    return fb200_vinterp_get_data_slice_columns_device(h, inType, d_in, &cols, nxy, nt, badValue, outType, d_out, stream);
}

int fb200_vinterp_interpolate_values_columns(const fb200_vinterp* h, const float* in, const fb200_vcolumns* cols, size_t nxy, size_t nt, float* out)
{
    if (check_vinterp_call(h, in, or_none(cols), nxy, nt, out) != FB_OK)
        return MIFI_ERROR;
    return vinterp_host(h, false, FB_T_FLOAT, in, or_none(cols), nxy, nt, 0.0, FB_T_FLOAT, out) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_vinterp_interpolate_values_columns_device(const fb200_vinterp* h, const float* d_in, const fb200_vcolumns* d_cols, size_t nxy, size_t nt,
                                                    float* d_out, void* stream)
{
    if (check_vinterp_call(h, d_in, or_none(d_cols), nxy, nt, d_out) != FB_OK)
        return MIFI_ERROR;
    return vinterp_device(h, false, FB_T_FLOAT, d_in, or_none(d_cols), nxy, nt, 0.0, FB_T_FLOAT, d_out, as_stream(stream)) == FB_OK ? MIFI_OK
                                                                                                                                     : MIFI_ERROR;
}

int fb200_vinterp_get_data_slice_columns(const fb200_vinterp* h, int inType, const void* in, const fb200_vcolumns* cols, size_t nxy, size_t nt,
                                         double badValue, int outType, void* out)
{
    if (check_slice_types(inType, outType) != FB_OK || check_vinterp_call(h, in, or_none(cols), nxy, nt, out) != FB_OK)
        return MIFI_ERROR;
    return vinterp_host(h, true, inType, in, or_none(cols), nxy, nt, badValue, outType, out) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_vinterp_get_data_slice_columns_device(const fb200_vinterp* h, int inType, const void* d_in, const fb200_vcolumns* d_cols, size_t nxy,
                                                size_t nt, double badValue, int outType, void* d_out, void* stream)
{
    if (check_slice_types(inType, outType) != FB_OK || check_vinterp_call(h, d_in, or_none(d_cols), nxy, nt, d_out) != FB_OK)
        return MIFI_ERROR;
    return vinterp_device(h, true, inType, d_in, or_none(d_cols), nxy, nt, badValue, outType, d_out, as_stream(stream)) == FB_OK ? MIFI_OK
                                                                                                                                  : MIFI_ERROR;
}

int fb200_vconvert_create(int op, int vcoord, const double* a, const double* b, int nk, double ptop, double ps_scale, fb200_vconvert** handle)
{
    return vconvert_create(op, vcoord, a, b, nk, ptop, ps_scale, handle) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

void fb200_vconvert_destroy(fb200_vconvert* h)
{
    delete h;
}

int fb200_vconvert_values(const fb200_vconvert* h, const float* in, const fb200_vcolumns* cols, size_t nxy, size_t nt, float* out)
{
    if (check_vconvert_call(h, in, or_none(cols), nxy, nt, out) != FB_OK)
        return MIFI_ERROR;
    return vconvert_host(h, in, or_none(cols), nxy, nt, out) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_vconvert_values_device(const fb200_vconvert* h, const float* d_in, const fb200_vcolumns* d_cols, size_t nxy, size_t nt, float* d_out,
                                 void* stream)
{
    if (check_vconvert_call(h, d_in, or_none(d_cols), nxy, nt, d_out) != FB_OK)
        return MIFI_ERROR;
    return vconvert_device(h, d_in, or_none(d_cols), nxy, nt, d_out, as_stream(stream)) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_tinterp_create(const double* times, int nt, const double* new_times, int nt_new, int extrapolate, fb200_tinterp** handle)
{
    return tinterp_create(times, nt, new_times, nt_new, extrapolate, handle) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

void fb200_tinterp_destroy(fb200_tinterp* h)
{
    delete h;
}

int fb200_tinterp_source_steps(const fb200_tinterp* h, int j, int* ia, int* ib, double* w)
{
    FB_REQUIRE(h != nullptr, "null time interpolation handle");
    FB_REQUIRE(j >= 0 && j < h->nj, "target step " + std::to_string(j) + " out of range [0, " + std::to_string(h->nj) + ")");
    FB_REQUIRE(ia && ib && w, "null output pointer");
    const TimeStep& m = h->map[j];
    *ia = m.ia;
    *ib = m.ia < 0 ? -1 : m.ia + 1;
    *w = m.w;
    return MIFI_OK;
}

int fb200_tinterp_get_step(const fb200_tinterp* h, int j, int inType, const void* a, const void* b, size_t n, double badValue, int outType, void* out)
{
    if (check_tinterp_call(h, false, j, inType, outType, n, a, b, out) != FB_OK)
        return MIFI_ERROR;
    return tinterp_get_step_host(h, j, inType, a, b, n, badValue, outType, out) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_tinterp_get_step_device(const fb200_tinterp* h, int j, int inType, const void* d_a, const void* d_b, size_t n, double badValue, int outType,
                                  void* d_out, void* stream)
{
    if (check_tinterp_call(h, false, j, inType, outType, n, d_a, d_b, d_out) != FB_OK)
        return MIFI_ERROR;
    return launch_tinterp(inType, d_a, d_b, (long long)n, has_bad_value(badValue), (float)badValue, h->d_single + j, 1, outType, badValue, d_out,
                          as_stream(stream)) == FB_OK
               ? MIFI_OK
               : MIFI_ERROR;
}

int fb200_tinterp_get_data_slice_device(const fb200_tinterp* h, int inType, const void* d_in, size_t n, double badValue, int outType, void* d_out,
                                        void* stream)
{
    if (check_tinterp_call(h, true, 0, inType, outType, n, d_in, d_in, d_out) != FB_OK)
        return MIFI_ERROR;
    return launch_tinterp(inType, d_in, nullptr, (long long)n, has_bad_value(badValue), (float)badValue, h->d_sorted, h->nj, outType, badValue, d_out,
                          as_stream(stream)) == FB_OK
               ? MIFI_OK
               : MIFI_ERROR;
}

int fb200_merge_create(const fb200_interp* outerToInner, const fb200_interp* innerToTarget, const fb200_interp* outerToTarget, size_t innerX, size_t innerY,
                       size_t outerX, size_t outerY, int transitionWidth, int borderWidth, int useOuterIfInnerUndefined, fb200_merge** handle)
{
    return merge_create(outerToInner, innerToTarget, outerToTarget, innerX, innerY, outerX, outerY, transitionWidth, borderWidth, useOuterIfInnerUndefined,
                        handle) == FB_OK
               ? MIFI_OK
               : MIFI_ERROR;
}

void fb200_merge_destroy(fb200_merge* h)
{
    delete h;
}

int fb200_merge_get_data_slice(const fb200_merge* h, int inType, const void* inner, size_t innerSize, double badInner, const void* outer, size_t outerSize,
                               double badOuter, int outType, double outFill, void* out, size_t* newSize)
{
    size_t nz = 0;
    if (check_merge_call(h, inType, outType, innerSize, outerSize, inner, outer, out, &nz) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = merge_target_level(h) * nz;
    return merge_host(h, inType, inner, badInner, outer, badOuter, nz, outType, outFill, out) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

int fb200_merge_get_data_slice_device(const fb200_merge* h, int inType, const void* d_inner, size_t innerSize, double badInner, const void* d_outer,
                                      size_t outerSize, double badOuter, int outType, double outFill, void* d_out, size_t* newSize, void* stream)
{
    size_t nz = 0;
    if (check_merge_call(h, inType, outType, innerSize, outerSize, d_inner, d_outer, d_out, &nz) != FB_OK)
        return MIFI_ERROR;
    if (newSize)
        *newSize = merge_target_level(h) * nz;
    return merge_device(h, inType, d_inner, badInner, d_outer, badOuter, nz, outType, outFill, d_out, as_stream(stream)) == FB_OK ? MIFI_OK : MIFI_ERROR;
}

// ---------------------------------------------------------------------------------------- mifi_* drop-ins
int mifi_string_to_interpolation_method(const char* s)
{
    // src/interpolation.c:66-101; "forward_undef_min" -> FORWARD_MIN is the reference's behaviour (:97-98)
    static const struct {
        const char* name;
        int method;
    } table[] = {{"bilinear", FB_BILINEAR},
                 {"nearestneighbor", FB_NN},
                 {"bicubic", FB_BICUBIC},
                 {"coord_nearestneighbor", FB_COORD_NN},
                 {"coord_kdtree", FB_COORD_NN_KD},
                 {"forward_sum", FB_FWD_SUM},
                 {"forward_mean", FB_FWD_MEAN},
                 {"forward_median", FB_FWD_MEDIAN},
                 {"forward_max", FB_FWD_MAX},
                 {"forward_min", FB_FWD_MIN},
                 {"forward_undef_sum", FB_FWD_UNDEF_SUM},
                 {"forward_undef_mean", FB_FWD_UNDEF_MEAN},
                 {"forward_undef_median", FB_FWD_UNDEF_MEDIAN},
                 {"forward_undef_max", FB_FWD_UNDEF_MAX},
                 {"forward_undef_min", FB_FWD_MIN}};
    if (!s)
        return -1;
    for (const auto& e : table)
        if (std::strcmp(e.name, s) == 0)
            return e.method;
    return -1;
}

int mifi_project_values(const char* proj_input, const char* proj_output, double* x, double* y, const int num)
{
    ProjDef pin, pout;
    if (parse_pair(proj_input, proj_output, &pin, &pout) != FB_OK)
        return MIFI_ERROR;
    if (num <= 0)
        return MIFI_OK;
    FB_REQUIRE(x && y, "null argument");
    if (use_device(default_device()) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    Scratch tmp(st);
    double *d_x = nullptr, *d_y = nullptr;
    int* d_status = nullptr;
    if (tmp.upload(&d_x, x, (size_t)num) != FB_OK || tmp.upload(&d_y, y, (size_t)num) != FB_OK || tmp.get(&d_status, 1) != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (launch_project_values(pin, pout, d_x, d_y, num, d_status, st) != FB_OK)
        return MIFI_ERROR;
    if (check_status(d_status, st, "mifi_project_values") != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(x, d_x, sizeof(double) * num, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(y, d_y, sizeof(double) * num, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return MIFI_OK;
}

int mifi_project_axes(const char* proj_input, const char* proj_output, const double* in_x_axis, const double* in_y_axis, const int ix,
                      const int iy, double* out_x, double* out_y)
{
    ProjDef pin, pout;
    if (parse_pair(proj_input, proj_output, &pin, &pout) != FB_OK)
        return MIFI_ERROR;
    if (ix <= 0 || iy <= 0)
        return MIFI_OK;
    FB_REQUIRE(in_x_axis && in_y_axis && out_x && out_y, "null argument");
    if (use_device(default_device()) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    const size_t n = (size_t)ix * iy;
    Scratch tmp(st);
    double *d_x = nullptr, *d_y = nullptr;
    if (tmp.get(&d_x, n) != FB_OK || tmp.get(&d_y, n) != FB_OK)
        return MIFI_ERROR;
    const std::vector<double> xa(in_x_axis, in_x_axis + ix), ya(in_y_axis, in_y_axis + iy);
    if (project_axes_device(pin, pout, xa, ya, d_x, d_y, st, "mifi_project_axes") != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(out_x, d_x, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaMemcpyAsync(out_y, d_y, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return MIFI_OK;
}

int mifi_points2position(double* points, const int n, const double* axis, const int num, const int axis_type)
{
    if (n <= 0)
        return MIFI_OK;
    FB_REQUIRE(points && axis && num >= 2, "mifi_points2position: null argument or axis shorter than 2");
    if (use_device(default_device()) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    Scratch tmp(st);
    double* d_p = nullptr;
    if (tmp.upload(&d_p, points, (size_t)n) != FB_OK)
        return MIFI_ERROR;
    const std::vector<double> ax(axis, axis + num);
    if (points2position_device(d_p, n, ax, axis_type, st) != FB_OK)
        return MIFI_ERROR;
    FB_CUDA_CHECK(cudaMemcpyAsync(points, d_p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    FB_CUDA_CHECK(cudaStreamSynchronize(st));
    return MIFI_OK;
}

int mifi_interpolate_f(int method, const char* proj_input, const float* infield, const double* in_x_axis, const double* in_y_axis,
                       const int in_x_axis_type, const int in_y_axis_type, const int ix, const int iy, const int iz, const char* proj_output,
                       float* outfield, const double* out_x_axis, const double* out_y_axis, const int out_x_axis_type,
                       const int out_y_axis_type, const int ox, const int oy)
{
    // src/interpolation.c:281-297: only the three gather methods; anything else is an error before any work
    if (method != FB_NN && method != FB_BILINEAR && method != FB_BICUBIC)
        return MIFI_ERROR;
    FB_REQUIRE(ix > 0 && iy > 0 && iz >= 0 && ox >= 0 && oy >= 0, "mifi_interpolate_f: bad dimensions");
    FB_REQUIRE(in_x_axis && in_y_axis && out_x_axis && out_y_axis, "mifi_interpolate_f: null axis");
    ProjDef pin, pout;
    // the reference ignores a failing mifi_project_axes here (:257) and interpolates garbage; failing is the
    // only defined behaviour we can offer
    if (parse_pair(proj_input, proj_output, &pin, &pout) != FB_OK)
        return MIFI_ERROR;
    auto typed_deg = [](int t) { return t == FB_AXIS_LONGITUDE || t == FB_AXIS_LATITUDE; };
    const std::vector<double> ixa = axis_in_radians(in_x_axis, (size_t)ix, typed_deg(in_x_axis_type));
    const std::vector<double> iya = axis_in_radians(in_y_axis, (size_t)iy, typed_deg(in_y_axis_type));
    const std::vector<double> oxa = axis_in_radians(out_x_axis, (size_t)ox, typed_deg(out_x_axis_type));
    const std::vector<double> oya = axis_in_radians(out_y_axis, (size_t)oy, typed_deg(out_y_axis_type));
    std::unique_ptr<fb200_interp> h;
    if (new_interp(method, false, (size_t)ix, (size_t)iy, (size_t)ox, (size_t)oy, &h) != FB_OK)
        return MIFI_ERROR;
    cudaStream_t st = cudaStreamPerThread;
    if (h->npts) {
        if (project_axes_device(pout, pin, oxa, oya, h->d_px, h->d_py, st, "mifi_interpolate_f") != FB_OK)
            return MIFI_ERROR;
        if (points2position_device(h->d_px, (long long)h->npts, ixa, in_x_axis_type, st) != FB_OK)
            return MIFI_ERROR;
        if (points2position_device(h->d_py, (long long)h->npts, iya, in_y_axis_type, st) != FB_OK)
            return MIFI_ERROR;
    }
    if (compile_tables(h.get(), st) != FB_OK)
        return MIFI_ERROR;
    if (iz == 0 || h->npts == 0)
        return MIFI_OK;
    FB_REQUIRE(infield && outfield, "mifi_interpolate_f: null field");
    const float* in[1] = {infield};
    float* out[1] = {outfield};
    return run_host(h.get(), nullptr, 1, in, out, (size_t)iz);
}

int mifi_get_vector_reproject_matrix(const char* proj_input, const char* proj_output, const double* out_x_axis, const double* out_y_axis,
                                     int xt, int yt, int ox, int oy, double* matrix)
{
    return matrix_to_host(MI_AXES, proj_input, proj_output, out_x_axis, out_y_axis, xt, yt, ox, oy, 0, matrix);
}

int mifi_get_vector_reproject_matrix_field(const char* proj_input, const char* proj_output, const double* in_x_field, const double* in_y_field,
                                           int ox, int oy, double* matrix)
{
    return matrix_to_host(MI_FIELD, proj_input, proj_output, in_x_field, in_y_field, 0, 0, ox, oy, 0, matrix);
}

int mifi_get_vector_reproject_matrix_points(const char* proj_input, const char* proj_output, int inputIsMetric, const double* out_x_points,
                                            const double* out_y_points, int on, double* matrix)
{
    return matrix_to_host(MI_POINTS, proj_input, proj_output, out_x_points, out_y_points, 0, 0, on, 1, inputIsMetric, matrix);
}

int mifi_vector_reproject_values_by_matrix_f(int method, const double* matrix, float* u_out, float* v_out, int ox, int oy, int oz)
{
    fb200_vector* v = nullptr;
    if (fb200_vector_create(method, matrix, ox, oy, &v) != MIFI_OK)
        return MIFI_ERROR;
    const int rc = (ox > 0 && oy > 0 && oz > 0) ? fb200_vector_reproject_values(v, u_out, v_out, (size_t)ox * oy * oz) : MIFI_OK;
    fb200_vector_destroy(v);
    return rc;
}

int mifi_vector_reproject_direction_by_matrix_f(int method, const double* matrix, float* angle_out, int ox, int oy, int oz)
{
    fb200_vector* v = nullptr;
    if (fb200_vector_create(method, matrix, ox, oy, &v) != MIFI_OK)
        return MIFI_ERROR;
    const int rc = (ox > 0 && oy > 0 && oz > 0) ? fb200_vector_reproject_direction_values(v, angle_out, (size_t)ox * oy * oz) : MIFI_OK;
    fb200_vector_destroy(v);
    return rc;
}

int mifi_vector_reproject_values_f(int method, const char* proj_input, const char* proj_output, float* u_out, float* v_out,
                                   const double* out_x_axis, const double* out_y_axis, int xt, int yt, int ox, int oy, int oz)
{
    // src/interpolation.c:837-859, without the round trip of the matrix through the host
    fb200_vector* v = nullptr;
    if (fb200_vector_create_from_projection(method, proj_input, proj_output, out_x_axis, out_y_axis, xt, yt, ox, oy, &v) != MIFI_OK)
        return MIFI_ERROR;
    const int rc = (oz > 0) ? fb200_vector_reproject_values(v, u_out, v_out, (size_t)ox * oy * oz) : MIFI_OK;
    fb200_vector_destroy(v);
    return rc;
}

// The per-point kernels of include/fimex/interpolation.h:231-291 exist for link-level compatibility and for tests: each call
// builds a one-point table, uploads the WHOLE field and launches a kernel.  A host that keeps the reference's function-pointer
// loop (src/CachedInterpolation.cc:133-141) instead of forwarding interpolateValues to fb200_interp_interpolate_values would
// call this millions of times per slice -- say so, once, instead of being silently slow (there is no CPU fallback to switch to).
static void warn_if_called_in_a_loop()
{
    static std::atomic<unsigned> calls{0};
    static std::atomic<long long> window_start{0};
    static std::atomic<bool> warned{false};
    if (warned.load(std::memory_order_relaxed))
        return;
    const long long now = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
    long long start = window_start.load(std::memory_order_relaxed);
    if (now - start > 1000) { // a new one-second window
        window_start.store(now, std::memory_order_relaxed);
        calls.store(0, std::memory_order_relaxed);
    }
    if (calls.fetch_add(1, std::memory_order_relaxed) + 1 > 1000 && !warned.exchange(true)) {
        fprintf(stderr, "fimex_b200: WARNING: mifi_get_values*_f called more than 1000 times within a second.  These per-point entry points "
                        "upload the whole field on every call; forward CachedInterpolation::interpolateValues to "
                        "fb200_interp_interpolate_values (see INTEGRATION.md) instead of looping over target points on the host.\n");
    }
}

static int one_point(int method, const float* infield, float* outvalues, double x, double y, int ix, int iy, int iz)
{
    warn_if_called_in_a_loop();
    fb200_interp* h = nullptr;
    if (fb200_cached_interpolation_create(method, &x, &y, (size_t)ix, (size_t)iy, 1, 1, &h) != MIFI_OK)
        return MIFI_ERROR;
    size_t ns = 0;
    const int rc = fb200_interp_interpolate_values(h, infield, (size_t)ix * iy * iz, outvalues, &ns);
    fb200_interp_destroy(h);
    return rc;
}

int mifi_get_values_f(const float* infield, float* outfield, const double x, const double y, const int ix, const int iy, const int iz)
{
    return one_point(FB_NN, infield, outfield, x, y, ix, iy, iz);
}
int mifi_get_values_bilinear_f(const float* infield, float* outvalues, const double x, const double y, const int ix, const int iy, const int iz)
{
    return one_point(FB_BILINEAR, infield, outvalues, x, y, ix, iy, iz);
}
int mifi_get_values_bicubic_f(const float* infield, float* outvalues, const double x, const double y, const int ix, const int iy, const int iz)
{
    return one_point(FB_BICUBIC, infield, outvalues, x, y, ix, iy, iz);
}

int mifi_setNumThreads(int n)
{
    (void)n; // src/ThreadPool.c:33-46 sets the OpenMP team size; the GPU path has no host threads to size
    return MIFI_OK;
}

} // extern "C"
