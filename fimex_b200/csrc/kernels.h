// fimex_b200/csrc/kernels.h -- internal launch interface between api.cu and the kernel files.
// All pointers are DEVICE pointers unless a name says host; all functions enqueue on `st` and return
// FB_OK / FB_ERROR without synchronising unless stated.
#pragma once

#include "common.cuh"
#include "proj.cuh"
#include "convert.cuh"

namespace fb {

// ---- setup_kernels.cu (K1, K2, K7, crop, table compilation) ------------------------------------------
// K1: expand axes to a mesh and transform src -> dst (mifi_project_axes, interpolation.c:1199-1244).
// d_status receives a non-zero PROJ error number when a point fails non-transiently.
int launch_project_mesh(const ProjDef& src, const ProjDef& dst, const double* d_xaxis, const double* d_yaxis, int nx, int ny, double* d_xo,
                        double* d_yo, int* d_status, cudaStream_t st);
// K1: transform arrays in place (mifi_project_values, interpolation.c:1158-1197)
int launch_project_values(const ProjDef& src, const ProjDef& dst, double* d_x, double* d_y, long long n, int* d_status, cudaStream_t st);
// K2: coordinate -> fractional array position, in place (mifi_points2position, interpolation.c:148-217)
int launch_points2position(double* d_points, long long n, const double* d_axis, const double* h_axis, int num, int axis_type,
                           cudaStream_t st);
// min/max of an array (std::min_element / max_element of CachedInterpolation.cc:165-168); synchronises
int device_minmax(const double* d_v, long long n, double* h_min, double* h_max, cudaStream_t st);
// v[i] -= delta (CachedInterpolation.cc:183-186)
int launch_shift(double* d_v, long long n, double delta, cudaStream_t st);
// deg -> rad / copy (convertAxis, interpolation.c:221-229)
int launch_scale(double* d_v, long long n, double factor, cudaStream_t st);

// positions -> gather tables
int launch_compile_nn(const double* d_px, const double* d_py, long long n, int ix, int iy, int* d_off, cudaStream_t st);
int launch_compile_bilinear(const double* d_px, const double* d_py, long long n, int ix, int iy, int4* d_tab, cudaStream_t st);
int launch_compile_bicubic(const double* d_px, const double* d_py, long long n, int ix, int iy, int* d_off, double2* d_frac,
                           cudaStream_t st);
// forward: positions (per INPUT point) -> target cell or -1 (CachedForwardInterpolation.cc:73-74, Utils.cc:42-58)
int launch_compile_forward_cells(const double* d_px, const double* d_py, long long n, int ox, int oy, int* d_cell, cudaStream_t st);

// K7: rotation matrix from the three projected fields (interpolation.c:330-438)
int launch_vector_matrix(const ProjDef& in, const ProjDef& out, const double* d_in_x, const double* d_in_y, const double* d_out_x,
                         const double* d_out_y, double dx, double dy, long long n, double* d_matrix, int* d_status, cudaStream_t st);
// matrix [n][4] -> compact (cos, sin) pairs
int launch_matrix_to_cossin(const double* d_matrix, long long n, double2* d_cs, cudaStream_t st);

// K9: coord_nearestneighbor search (CDMInterpolator.cc:1141-1220) -- see coordnn_kernels.cu
int coordnn_search(double* d_px, double* d_py, long long n, const double* h_lon, const double* h_lat, size_t nx, size_t ny,
                   long long* ties, cudaStream_t st);

// coord_kdtree search (flannTranslatePointsToClosestInputCell, CDMInterpolator.cc:991-1062): exact nearest source point by
// squared chord distance inside (max_dist_m / R)^2, else (-1000, -1000)
int coordkd_search(double* d_px, double* d_py, long long n, const double* h_lon, const double* h_lat, size_t nx, size_t ny, double max_dist_m,
                   long long* ties, cudaStream_t st);

// ---- gather_kernels.cu (K3, K4, K5, K6) -------------------------------------------------------------
struct GatherGeom {
    int ix, iy, ox, oy;
    long long in_level;  // ix*iy
    long long out_level; // ox*oy
    long long nz;
};
int z_chunks(long long ctas_x, long long nz, int levels = 64); // gridDim.y policy shared by the gather kernels
int launch_gather_nn(const GatherGeom& g, const int* d_off, const float* d_in, float* d_out, cudaStream_t st);
int launch_gather_bilinear(const GatherGeom& g, const int4* d_tab, const float* d_in, float* d_out, cudaStream_t st);
int launch_gather_bicubic(const GatherGeom& g, const int* d_off, const double2* d_frac, const float* d_in, float* d_out, cudaStream_t st);
// fused u/v: interpolate both components with one table and rotate (K6 fused); d_cs may be null (no rotation)
int launch_gather_vector(int method, const GatherGeom& g, const void* d_tab, const void* d_tab2, const double2* d_cs, const float* d_u_in,
                         const float* d_v_in, float* d_u_out, float* d_v_out, cudaStream_t st);
// K6 stand-alone: rotate u, v in place (mifi_vector_reproject_values_by_matrix_f, interpolation.c:790-812)
int launch_rotate(const double2* d_cs, float* d_u, float* d_v, long long layer, long long nz, cudaStream_t st);
// mifi_vector_reproject_direction_by_matrix_f (interpolation.c:814-835)
int launch_rotate_direction(const double* d_matrix, float* d_angle, long long layer, long long nz, cudaStream_t st);

// ---- staged_kernels.cu (K4 fast path) -------------------------------------------------------------------
struct TileTable {
    int tiles_x = 0, tiles_y = 0;
    int* d_cells = nullptr;   // [tile][4096] sorted distinct source offsets ("taps") of the tile
    int* d_ncells = nullptr;  // [tile] number of taps
    uint4* d_meta = nullptr;  // [tile][256] 4 x (a | b << 12 | mode << 24)
    float4* d_xf = nullptr;   // [tile][256]
    float4* d_yf = nullptr;   // [tile][256]
    int* d_slow = nullptr;    // ids of the tiles with more taps than the tap-major staging buffer holds (pole, seam)
    int n_slow = 0;
    bool quad = false;        // tile geometry: 128 x 8, a thread owns 4 x-neighbours (nearest neighbour; bilinear by default)
    bool nn = false;          // nearest-neighbour table (one tap per point, no xf/yf)
    bool ready() const { return d_cells != nullptr; }
};
bool tile_table_supported(int ix, int iy, int ox, int oy);
int tile_table_build(bool nn, const double* d_px, const double* d_py, int ix, int iy, int ox, int oy, TileTable* tt, cudaStream_t st);
void tile_table_free(TileTable* tt);
// staged gather for bilinear and nearest-neighbour tables; sc: fill -> NaN while staging, NaN -> fill + cast while storing
int launch_gather_bilinear_staged(const GatherGeom& g, const TileTable& tt, const float* d_in, void* d_out, const SliceConv& sc, cudaStream_t st);
bool staged_store_supports(int out_type);
// both components of a vector through the staged gather (plain float output), rotated when d_cs != nullptr
int launch_gather_staged_vector(const GatherGeom& g, const TileTable& tt, const double2* d_cs, const float* d_u, const float* d_v, float* d_uo,
                                float* d_vo, const SliceConv& sc, cudaStream_t st);

// ---- bicubic_staged.cu (K5 fast path) ------------------------------------------------------------------
struct BicubicTiles {
    int tiles_x = 0, tiles_y = 0;
    int4* d_info = nullptr;     // [tile] {first tap, ntaps (-1: direct fallback), first group, ngroups}
    int* d_taps = nullptr;      // per tile: sorted distinct source offsets
    uint4* d_gmeta = nullptr;   // [group] 8 x u16: 4 stencil-row tap indices, 4 point slots
    double2* d_gfrac = nullptr; // [group][4] (xfrac, yfrac)
    long long n_taps = 0, n_groups = 0;
    int n_direct = 0;           // tiles computed with direct global loads (tap list too long to stage)
    bool ready() const { return d_info != nullptr; }
};
bool bicubic_tiles_supported(int ix, int iy, int ox, int oy);
// d_off / d_frac: the per-point bicubic table of launch_compile_bicubic; synchronises
int bicubic_tiles_build(const int* d_off, const double2* d_frac, int ix, int iy, int ox, int oy, BicubicTiles* bt, cudaStream_t st);
void bicubic_tiles_free(BicubicTiles* bt);
// scalar field (d_in1 == d_out1 == nullptr; converts like the staged bilinear gather) or both components of a vector
// (plain float output), rotated when d_cs != nullptr
int launch_gather_bicubic_staged(const GatherGeom& g, const BicubicTiles& bt, const int* d_off, const double2* d_frac, const double2* d_cs,
                                 const float* d_in0, const float* d_in1, void* d_out0, void* d_out1, const SliceConv& sc, cudaStream_t st);

// ---- adapter_kernels.cu (K10, unfused forms) ---------------------------------------------------------------
// data2InterpolationArray: any CDM numeric type -> float with badValue -> NaN (CDMInterpolator.cc:115-119)
int launch_as_float(int in_type, const void* d_in, long long n, bool has_bad, float bad, float* d_out, cudaStream_t st);
// interpolationArray2Data: NaN -> fill, round + cast (CDMInterpolator.cc:121-124); in place allowed for FB_T_FLOAT
int launch_from_float(const float* d_in, long long n, int out_type, double fill, void* d_out, cudaStream_t st);

// ---- fill_kernels.cu (2-D pre/post-processes: fill2d, creepfill2d) -----------------------------------------------
// nz levels of nx x ny in place; d_nchanged (nz counters, may be null) receives the NaN count of every level
int launch_fill2d(float* d_field, size_t nx, size_t ny, size_t nz, float relaxCrit, float corrEff, size_t maxLoop,
                  unsigned long long* d_nchanged, cudaStream_t st);
int launch_creepfill2d(float* d_field, size_t nx, size_t ny, size_t nz, bool use_mean, float defaultVal, unsigned short repeat,
                       signed char setWeight, unsigned long long* d_nchanged, cudaStream_t st);

// ---- forward_kernels.cu (K8) ---------------------------------------------------------------------------
struct ForwardPlan {
    long long n_in = 0, n_cells = 0;
    int* d_perm = nullptr;    // input indices grouped by target cell, ascending inside each cell
    int* d_offsets = nullptr; // n_cells + 1
    long long n_mapped = 0;
};
int forward_build_plan(const int* d_cell, long long n_in, long long n_cells, ForwardPlan* plan, cudaStream_t st);
void forward_free_plan(ForwardPlan* plan);
int launch_forward(int method, const ForwardPlan& plan, const float* d_in, float* d_out, long long nz, cudaStream_t st);

// ---- vertical_kernels.cu (vertical interpolation to pressure, height, altitude and depth levels) ------------------------
// methods, numbered as the reference's MIFI_VINT_METHOD_* (include/fimex/mifi_constants.h)
enum { FB_VINT_LIN = 0, FB_VINT_LOG = 1, FB_VINT_LOGLOG = 2, FB_VINT_NN = 3 };
// height converters (FB_VZ_NONE: a pressure or depth handle) and targets, numbered as FB200_VZ_* (include/fimex_b200.h)
enum { FB_VZ_NONE = -1, FB_VZ_STANDARD = 0, FB_VZ_HYPSOMETRIC = 1, FB_VZ_FIELD = 2 };
enum { FB_VZ_ALTITUDE = 0, FB_VZ_HEIGHT = 1 };
// source coordinates of the depth handles (FB_VD_NONE: a pressure or height handle), numbered as FB200_VCOORD_* (include/fimex_b200.h)
enum { FB_VD_NONE = -1, FB_VD_DEPTH = 3, FB_VD_OCEAN_SIGMA = 4, FB_VD_OCEAN_S_G1 = 5, FB_VD_OCEAN_S_G2 = 6 };
constexpr int kStdLayers = 7; // geopotential layers of the US Standard Atmosphere 1976
struct VertTable {
    int method = 0, nk = 0, np = 0;
    bool extrapolate = true;
    double ps_scale = 1.0, shift = 0.0; // p_k = a_k + b_k * (ps * ps_scale - shift)
    // pressure handles: a[nk] | b[nk] | sorted targets[np] | their coordinates[np] | output row of each[np]
    // height handles:   a[nk] | b[nk] | standard-atmosphere layers h_b, p_b, c_b, e_b [4][kStdLayers] | sorted targets[np] | output row of each[np]
    // depth handles:    levels, sigma_k or depth_c * s_k [nk] | C_k (0 for depth and sigma) [nk] | sorted targets[np] | output row of each[np]
    double* d_tab = nullptr;
    int converter = FB_VZ_NONE, target = FB_VZ_ALTITUDE;
    double z_scale = 1.0, zs_scale = 1.0; // z = z_scale * Z (field converter); z_s = zs_scale * zs
    double H = 0.0, cq = 0.0;             // R* / (M g0) [m/K]; M / M_w - 1 (virtual temperature)
    int depth_vcoord = FB_VD_NONE;
    double depth_c = 0.0; // ocean_s_coordinate_g1 / _g2
};
// the coordinate of each target the weights are linear in (p, ln p or ln ln p), computed with the kernel's own ln()
int launch_vert_coords(int method, const double* d_lev, double* d_x, int np, cudaStream_t st);
// in [nt][nk][nxy], ps [nt][nxy] (null for pressure levels), out [nt][np][nxy]
int launch_vertical(const VertTable& vt, const float* d_in, const float* d_ps, long long nxy, long long nt, float* d_out, cudaStream_t st);
// height handles: in, t, q, z [nt][nk][nxy], ps [nt][nxy], zs [nxy] (null where the converter and target do not use them), out [nt][np][nxy]
int launch_vertical_height(const VertTable& vt, const float* d_in, const float* d_ps, const float* d_t, const float* d_q, const float* d_z,
                           const float* d_zs, long long nxy, long long nt, float* d_out, cudaStream_t st);
// depth handles: in [nt][nk][nxy], eta [nt][nxy] (null: 0), depth [nxy] (null for depth levels), out [nt][np][nxy]
int launch_vertical_depth(const VertTable& vt, const float* d_in, const float* d_eta, const float* d_depth, long long nxy, long long nt, float* d_out,
                          cudaStream_t st);
// data conversions, numbered as FB200_VCONV_* (include/fimex_b200.h); source coordinates FB200_VCOORD_PRESSURE, _HYBRID, _SIGMA
enum { FB_VCONV_THETA2T = 0, FB_VCONV_OMEGA2VWIND = 1, FB_VCONV_PRESSURE = 2 };
enum { FB_VCOORD_PRESSURE = 0, FB_VCOORD_HYBRID = 1, FB_VCOORD_SIGMA = 2 };
// vt: a[nk] | b[nk], ps_scale, shift and H of a pressure or height handle (np = 0).  in [nt][nk][nxy] (theta or omega; null for
// FB_VCONV_PRESSURE), ps [nt][nxy] (null for pressure levels), t [nt][nk][nxy] (omega2vwind), out [nt][nk][nxy]; d_out == d_in is allowed
int launch_vconvert(int op, int vcoord, const VertTable& vt, double kappa, const float* d_in, const float* d_ps, const float* d_t, long long nxy,
                    long long nt, float* d_out, cudaStream_t st);

// ---- time_kernels.cu (time interpolation: CDMTimeInterpolator's linear change of the time axis) ------------------------
// one target step: output row `row` = step ia + w * (step ia+1 - step ia); ia = -1: no bracket (NaN, stored as the fill value)
struct alignas(16) TimeStep {
    int ia, row;
    double w;
};
// d_tab [nj]: the targets in non-decreasing ia, those with ia = -1 last.  in [.][n] of in_type (step k at d_in + k n; d_in_b != null:
// a two-step call with step 1 at d_in_b), badValue -> NaN while loading when has_bad; out [.][n] of out_type, NaN -> fill + cast
int launch_tinterp(int in_type, const void* d_in, const void* d_in_b, long long n, bool has_bad, float bad, const TimeStep* d_tab, int nj, int out_type,
                   double fill, void* d_out, cudaStream_t st);

// ---- merge_kernels.cu (CDMMerger: crop, linear border smoothing, overlay) -------------------------------------------------
// [nz][ny][nx] of in_type -> the window [x0, x0 + w) x [y0, y0 + h) of every level as float [nz][h][w], badValue -> NaN when has_bad
// (the gather's own input adapter, mifi_bad2nanf)
int launch_crop_as_float(int in_type, const void* d_in, long long nx, long long ny, long long x0, long long y0, long long w, long long h, long long nz,
                         bool has_bad, float bad, float* d_out, cudaStream_t st);
// the linear border smoothing (DESIGN.md section 2) of inner [nz][ny][nx] of in_type (values equal to (in_type)bad -> NaN when has_bad)
// with outer [nz][ny][nx] float on the inner grid, in fp64; only the window [x0, x0 + w) x [y0, y0 + h) is written, as float [nz][h][w]
int launch_border_smooth_linear(int in_type, const void* d_inner, bool has_bad, double bad, const float* d_outer, long long nx, long long ny, int t, int b,
                                bool use_outer, long long x0, long long y0, long long w, long long h, long long nz, float* d_out, cudaStream_t st);
// out[i] = top[i] where it is not NaN, else base[i]; NaN -> fill, round + cast to out_type
int launch_merge_overlay(const float* d_top, const float* d_base, long long n, int out_type, double fill, void* d_out, cudaStream_t st);

} // namespace fb
