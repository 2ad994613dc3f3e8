/*
 * fimex_b200.h -- C ABI of libfimex_b200.so: Fimex's horizontal-regridding hot path on NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary.  Two groups of entry points:
 *
 *  (1) HANDLE API -- what the three C++ classes of the reference forward to after a one-line patch
 *      (INTEGRATION.md):  CachedInterpolation / CachedForwardInterpolation (both behind
 *      CachedInterpolationInterface::interpolateValues) and CachedVectorReprojection::reprojectValues.
 *  (2) mifi_* FUNCTIONS -- the reference's own C symbols for this path, same names, same signatures, same
 *      MIFI_OK / MIFI_ERROR convention (reference include/fimex/interpolation.h), so a program linked
 *      against libfimex's C interface can link against this library for them instead.
 *
 * All file:line citations are relative to the reference tree (arebru/fimex 0.67.2).
 *
 * Conventions (SURVEY.md 8b):
 *  - plain pointers and sizes only; fp32 data is C-ordered [z][y][x], x fastest
 *    (mifi_3d_array_position, include/fimex/interpolation.h:423-426); tables are fp64 [outY][outX]
 *    (backward methods) or [inY][inX] (forward methods); the rotation matrix is fp64 [oy][ox][4]
 *    = (cos, sin, -sin, phi) (src/interpolation.c:429-432).
 *  - the caller owns every host buffer; nothing is retained after a call returns.
 *  - return MIFI_OK (1) or MIFI_ERROR (-1); the message is available from fb200_last_error() (per
 *    thread) and is also printed to stderr like the reference does; no C++ exception crosses the ABI.
 *  - handles are immutable after creation (createReducedDomain is part of creation) and every
 *    interpolate/reproject call is re-entrant: concurrent calls on one handle from several host threads are
 *    safe (the reference calls them from OpenMP tasks, src/NetCDF_CDMWriter.cc:749-753).
 *  - "_device" variants take DEVICE pointers (and a cudaStream_t passed as void*, NULL = per-thread
 *    default stream), do no host<->device copies and do not synchronise.
 *  - there is NO CPU fallback: every call fails with MIFI_ERROR when no CUDA device is usable.
 *  - device selection: environment variable FIMEX_B200_DEVICE (default: the current CUDA device) or
 *    fb200_set_device(); no new user option is needed (the fimex --interpolate.* options are untouched).
 */
#ifndef FIMEX_B200_H_
#define FIMEX_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef MIFI_OK
#define MIFI_ERROR -1 /* include/fimex/mifi_constants.h:259 */
#define MIFI_OK 1     /* include/fimex/mifi_constants.h:261 */
#endif
#ifndef MIFI_PROJ_AXIS
#define MIFI_PROJ_AXIS 0 /* include/fimex/mifi_constants.h:264-268 */
#define MIFI_LONGITUDE 1
#define MIFI_LATITUDE 2
#endif
#ifndef MIFI_VECTOR_KEEP_SIZE
#define MIFI_VECTOR_KEEP_SIZE 0 /* include/fimex/mifi_constants.h:154-160 */
#define MIFI_VECTOR_RESIZE 1
#endif

/* enum mifi_interpol_method, include/fimex/mifi_constants.h:52-147 (same numbering) */
#ifndef FIMEX_B200_NO_METHOD_ENUM
enum fb200_interpol_method {
    FB200_INTERPOL_UNKNOWN = -1,
    FB200_INTERPOL_NEAREST_NEIGHBOR = 0,
    FB200_INTERPOL_BILINEAR,
    FB200_INTERPOL_BICUBIC,
    FB200_INTERPOL_COORD_NN,
    FB200_INTERPOL_COORD_NN_KD,
    FB200_INTERPOL_FORWARD_SUM,
    FB200_INTERPOL_FORWARD_MEAN,
    FB200_INTERPOL_FORWARD_MEDIAN,
    FB200_INTERPOL_FORWARD_MAX,
    FB200_INTERPOL_FORWARD_MIN,
    FB200_INTERPOL_FORWARD_UNDEF_SUM,
    FB200_INTERPOL_FORWARD_UNDEF_MEAN,
    FB200_INTERPOL_FORWARD_UNDEF_MEDIAN,
    FB200_INTERPOL_FORWARD_UNDEF_MAX,
    FB200_INTERPOL_FORWARD_UNDEF_MIN
};
#endif

/* enum CDMDataType, include/fimex/CDMDataType.h:35-49 (same numbering) */
enum fb200_datatype {
    FB200_NAT = 0,
    FB200_CHAR,
    FB200_SHORT,
    FB200_INT,
    FB200_FLOAT,
    FB200_DOUBLE,
    FB200_STRING,
    FB200_UCHAR,
    FB200_USHORT,
    FB200_UINT,
    FB200_INT64,
    FB200_UINT64
};

/* ------------------------------------------------------------------------------------------------
 * library state
 * ---------------------------------------------------------------------------------------------- */
const char* fb200_version(void);
/* message of the last failed call made by the calling thread ("" if none) */
const char* fb200_last_error(void);
/* choose the CUDA device for handles created afterwards by this thread (default: $FIMEX_B200_DEVICE or current) */
int fb200_set_device(int device);
int fb200_get_device(void);
/* number of kernels this library has launched so far in the process (bench.py's gpu_launches) */
unsigned long long fb200_kernel_launches(void);
/* Page-locked host buffers for full-rate PCIe copies in the host-buffer calls (pageable buffers work too, at a third of
 * the rate).  Freed buffers stay page-locked in a size-keyed cache and are handed out again, because locking pages costs
 * about as much as copying them and the reference allocates a new output array per interpolateValues call
 * (src/CachedInterpolation.cc:123).  The cache keeps at most FIMEX_B200_PINNED_CACHE_MB (parsed once; default: an eighth of
 * the physical RAM, at most 8192 MB; 0 disables caching); fb200_host_trim releases it.  The buffers are portable
 * (usable from every device); the calls never change the calling thread's current device.  Thread-safe. */
void* fb200_host_alloc(size_t bytes);
void fb200_host_free(void* p);
void fb200_host_trim(void);

/* ------------------------------------------------------------------------------------------------
 * (1a) CachedInterpolationInterface: CachedInterpolation and CachedForwardInterpolation
 * ---------------------------------------------------------------------------------------------- */
typedef struct fb200_interp fb200_interp; /* opaque */

/* CachedInterpolation::CachedInterpolation(xDimName, yDimName, funcType, pointsOnXAxis, pointsOnYAxis, inX, inY,
 * outX, outY) -- include/fimex/CachedInterpolation.h:126-128, src/CachedInterpolation.cc:93-116.
 * funcType: NEAREST_NEIGHBOR, BILINEAR, BICUBIC, COORD_NN, COORD_NN_KD (the last two gather like NN).
 * pointsOn?Axis: outX*outY fractional source positions (host memory).  The dimension names are host
 * metadata and stay with the caller. */
int fb200_cached_interpolation_create(int funcType, const double* pointsOnXAxis, const double* pointsOnYAxis, size_t inX, size_t inY,
                                      size_t outX, size_t outY, fb200_interp** handle);
/* same, positions already on the device (used when the tables are computed or broadcast on the GPU) */
int fb200_cached_interpolation_create_device(int funcType, const double* d_pointsOnXAxis, const double* d_pointsOnYAxis, size_t inX,
                                             size_t inY, size_t outX, size_t outY, fb200_interp** handle);

/* The table-producing part of CDMInterpolator::changeProjectionByProjectionParameters
 * (src/CDMInterpolator.cc:1440-1481) on the device: target axes -> source CRS (mifi_project_axes :1458) ->
 * fractional source positions (mifi_points2position x2, :1475-1476) -> CachedInterpolation.
 * Axis values are in the projection's unit or DEGREES; *_is_degree mirrors the reference's unit regex
 * ".*degree.*" (:1443-1451) for the target and Projection::isDegree() (:1468-1473) for the source. */
int fb200_cached_interpolation_create_from_projection(int funcType, const char* proj_target, const double* out_x_axis,
                                                      const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                      int out_y_is_degree, const char* proj_source, const double* in_x_axis,
                                                      const double* in_y_axis, size_t inX, size_t inY, int in_is_degree,
                                                      fb200_interp** handle);

/* The table-producing part of CDMInterpolator::changeProjectionByProjectionParametersToLatLonTemplate
 * (src/CDMInterpolator.cc:1755-1803): the target is a 2-D lon/lat template (DEGREES, outX*outY values each, any curvilinear
 * grid or a 1-D point list with outY = 1) in CRS proj_template (normally MIFI_WGS84_LATLON_PROJ4): deg -> rad,
 * mifi_project_values(template -> source) (:1770), mifi_points2position on both source axes (:1789-1790), CachedInterpolation. */
int fb200_cached_interpolation_create_from_template(int funcType, const char* proj_template, const double* tmplLon, const double* tmplLat,
                                                    size_t outX, size_t outY, const char* proj_source, const double* in_x_axis,
                                                    const double* in_y_axis, size_t inX, size_t inY, int in_is_degree, fb200_interp** handle);

/* The table-producing part of CDMInterpolator::changeProjectionByCoordinates for MIFI_INTERPOL_COORD_NN
 * (src/CDMInterpolator.cc:1387-1412 with fastTranslatePointsToClosestInputCell :1141-1220): target axes ->
 * WGS84 lat/lon -> nearest source cell by great-circle distance.  lon2d/lat2d: source coordinates in
 * DEGREES, inX*inY values each, index ix + iy*inX. */
int fb200_cached_interpolation_create_from_coordinates(int funcType, const char* proj_target, const double* out_x_axis,
                                                       const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                       int out_y_is_degree, const double* lon2d, const double* lat2d, size_t inX,
                                                       size_t inY, fb200_interp** handle);

/* The same for MIFI_INTERPOL_COORD_NN_KD (coord_kdtree; flannTranslatePointsToClosestInputCell, src/CDMInterpolator.cc:991-1062):
 * the source point with the smallest squared chord distance on the unit sphere inside (maxDistance / 6371000)^2, else
 * (-1000, -1000).  maxDistance (metres) > 0 is the reference's setDistanceOfInterest; <= 0 derives it from the output
 * axes like getMaxDistanceOfInterest (:304-326).  funcType COORD_NN is accepted too (maxDistance is ignored then), and
 * fb200_cached_interpolation_create_from_coordinates accepts COORD_NN_KD with the derived distance. */
int fb200_cached_interpolation_create_from_coordinates_kd(int funcType, const char* proj_target, const double* out_x_axis,
                                                          const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                          int out_y_is_degree, const double* lon2d, const double* lat2d, size_t inX,
                                                          size_t inY, double maxDistance, fb200_interp** handle);

/* CachedForwardInterpolation::CachedForwardInterpolation(..., funcType, pOnX, pOnY, inX, inY, outX, outY) --
 * src/CachedForwardInterpolation.h:51-53, src/CachedForwardInterpolation.cc:62-90.  funcType: FORWARD_*.
 * pOnX/pOnY: inX*inY fractional TARGET positions of every source point. */
int fb200_cached_forward_interpolation_create(int funcType, const double* pOnX, const double* pOnY, size_t inX, size_t inY, size_t outX,
                                              size_t outY, fb200_interp** handle);
/* The table-producing part of CDMInterpolator::changeProjectionByForwardInterpolation
 * (src/CDMInterpolator.cc:1289-1332): source lon/lat (DEGREES, inX*inY each) -> target CRS
 * (mifi_project_values :1311) -> positions on the target axes (:1316-1317) -> CachedForwardInterpolation. */
int fb200_cached_forward_interpolation_create_from_coordinates(int funcType, const char* proj_target, const double* out_x_axis,
                                                               const double* out_y_axis, size_t outX, size_t outY, int out_x_is_degree,
                                                               int out_y_is_degree, const double* lon2d, const double* lat2d,
                                                               size_t inX, size_t inY, fb200_interp** handle);

/* CachedInterpolation::createReducedDomain -- src/CachedInterpolation.cc:159-200.  Crops the expected input to
 * the target footprint (+2 cells).  Returns MIFI_OK; *reduced tells whether a crop was applied, in which case
 * xMin and yMin receive the offsets into the original source grid and fb200_interp_in_x/y() shrink.
 * Must be called before the handle is shared between threads (it is part of construction). */
int fb200_interp_create_reduced_domain(fb200_interp* handle, int* reduced, long long* xMin, long long* yMin);

size_t fb200_interp_in_x(const fb200_interp* handle);  /* getInX()  */
size_t fb200_interp_in_y(const fb200_interp* handle);  /* getInY()  */
size_t fb200_interp_out_x(const fb200_interp* handle); /* getOutX() */
size_t fb200_interp_out_y(const fb200_interp* handle); /* getOutY() */
int fb200_interp_method(const fb200_interp* handle);
/* copy the fractional positions (after any crop) to host arrays / expose the device arrays */
int fb200_interp_get_points(const fb200_interp* handle, double* pointsOnXAxis, double* pointsOnYAxis);
int fb200_interp_device_points(const fb200_interp* handle, const double** d_pointsOnXAxis, const double** d_pointsOnYAxis, size_t* n);

/* CachedInterpolationInterface::interpolateValues(inData, size, newSize) -- include/fimex/CachedInterpolation.h:66,
 * src/CachedInterpolation.cc:118-147 and src/CachedForwardInterpolation.cc:92-131.
 * inData: `size` floats = [inZ][inY][inX]; outData: caller-allocated, outX*outY*inZ floats (query with
 * fb200_interp_new_size); *newSize receives that count.  Host buffers; copies are pipelined with the kernels. */
size_t fb200_interp_new_size(const fb200_interp* handle, size_t size);
int fb200_interp_interpolate_values(const fb200_interp* handle, const float* inData, size_t size, float* outData, size_t* newSize);
int fb200_interp_interpolate_values_device(const fb200_interp* handle, const float* d_inData, size_t size, float* d_outData,
                                           size_t* newSize, void* cuda_stream);
void fb200_interp_destroy(fb200_interp* handle);

/* ------------------------------------------------------------------------------------------------
 * (1b) CachedVectorReprojection
 * ---------------------------------------------------------------------------------------------- */
typedef struct fb200_vector fb200_vector; /* opaque */

/* CachedVectorReprojection(int method, shared_array<double> matrix, int ox, int oy) --
 * include/fimex/CachedVectorReprojection.h:36-44.  matrix: ox*oy*4 doubles (host). */
int fb200_vector_create(int method, const double* matrix, int ox, int oy, fb200_vector** handle);
/* mifi_get_vector_reproject_matrix (src/interpolation.c:719-788) evaluated on the device, as called from
 * src/CDMInterpolator.cc:1492-1500; axis values in the projection's unit or degrees (axis types as there) */
int fb200_vector_create_from_projection(int method, const char* proj_input, const char* proj_output, const double* out_x_axis,
                                        const double* out_y_axis, int out_x_axis_type, int out_y_axis_type, int ox, int oy,
                                        fb200_vector** handle);
/* mifi_get_vector_reproject_matrix_points (src/interpolation.c:719-788) on the device for a list of `on` points given as
 * lon/lat in DEGREES, as the lat/lon-template path builds it (src/CDMInterpolator.cc:1805-1823: proj_output =
 * MIFI_WGS84_LATLON_PROJ4, inputIsMetric = !isDegree(source)); the handle has ox = on, oy = 1 */
int fb200_vector_create_from_points(int method, const char* proj_input, const char* proj_output, int inputIsMetric, const double* lon,
                                    const double* lat, int on, fb200_vector** handle);
/* makeCachedVectorReprojection(dataReader, cs, toLatLon) (src/CDMProcessor.cc:99-145), the matrix behind
 * CDMProcessor::rotateVectorToLatLon / rotateDirectionToLatLon: the grid's OWN axes (degrees when isDegree, else metres).
 * toLatLon != 0: grid directions -> geographic (mifi_get_vector_reproject_matrix_field on the expanded mesh, :124-135);
 * toLatLon == 0: geographic -> grid directions (mifi_get_vector_reproject_matrix from MIFI_WGS84_LATLON_PROJ4, :137-140). */
int fb200_vector_create_from_grid(int method, const char* proj, const double* x_axis, const double* y_axis, int nx, int ny, int isDegree,
                                  int toLatLon, fb200_vector** handle);
/* reprojectValues(uValues, vValues, size): rotate in place -- src/CachedVectorReprojection.cc:35-44 */
int fb200_vector_reproject_values(const fb200_vector* handle, float* uValues, float* vValues, size_t size);
int fb200_vector_reproject_values_device(const fb200_vector* handle, float* d_uValues, float* d_vValues, size_t size, void* cuda_stream);
/* reprojectDirectionValues(angles, size) -- src/CachedVectorReprojection.cc:46-55 */
int fb200_vector_reproject_direction_values(const fb200_vector* handle, float* angles, size_t size);
int fb200_vector_get_matrix(const fb200_vector* handle, double* matrix);
/* The rotation branch of CDMProcessor::getDataSlice (src/CDMProcessor.cc:579-617) for one x/y pair: both components
 * fill -> NaN as float (data2InterpolationArray), reprojectValues, NaN -> fill and cast back (interpolationArray2Data).
 * inType/outType: enum fb200_datatype; `size` values per component; the caller keeps the component it asked for. */
int fb200_vector_get_slice(const fb200_vector* handle, int inType, const void* uIn, const void* vIn, size_t size, double badU, double badV,
                           int outType, void* uOut, void* vOut);
int fb200_vector_get_slice_device(const fb200_vector* handle, int inType, const void* d_uIn, const void* d_vIn, size_t size, double badU,
                                  double badV, int outType, void* d_uOut, void* d_vOut, void* cuda_stream);
void fb200_vector_destroy(fb200_vector* handle);

/* Fused form of src/CDMInterpolator.cc:255-276: interpolate both components of an x/y vector with ONE table
 * pass and rotate them in the same kernel (vector may be NULL: no rotation).  Outputs are outX*outY*inZ each. */
int fb200_interp_interpolate_vector(const fb200_interp* handle, const fb200_vector* vector, const float* uIn, const float* vIn,
                                    size_t size, float* uOut, float* vOut, size_t* newSize);
int fb200_interp_interpolate_vector_device(const fb200_interp* handle, const fb200_vector* vector, const float* d_uIn, const float* d_vIn,
                                           size_t size, float* d_uOut, float* d_vOut, size_t* newSize, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * (1c) the whole per-slice body of CDMInterpolator::getDataSlice in ONE call (src/CDMInterpolator.cc:250-285)
 *
 *   data2InterpolationArray  (:115-119)  Data::asFloat() + mifi_bad2nanf(badValue)      any CDM numeric type in
 *   interpolateValues        (:258)
 *   [reprojectValues         (:259-283)  with the counterpart component]
 *   interpolationArray2Data  (:121-124)  NaN -> badValue, round + cast to the variable's type
 *
 * inType / outType: enum fb200_datatype of the input slice and of the variable; badValue: CDM::getFillValue(varName)
 * (src/CDM.cc:505-522; NaN switches the input pass off, src/interpolation.c:1776).  On the staged gathers (bilinear,
 * nearest neighbour / coord_nn, bicubic) both adapter passes run INSIDE the gather kernel: the fill -> NaN compare is
 * applied once per staged source value and the output is written once, in the variable's type (a `short` variable
 * halves the bytes stored).  Other methods / 64-bit integer outputs take a float slab and one conversion pass.
 * outData: outX*outY*inZ elements of outType.  Pre/post-processes added with fb200_interp_add_pre/postprocess run inside the call.
 * ---------------------------------------------------------------------------------------------- */
/* CDMInterpolator::addPreprocess / addPostprocess (src/CDMInterpolator.cc:1886-1896) with the option strings of
 * --interpolate.preprocess / --interpolate.postprocess as parseProcess reads them (src/binSrc/fimex.cc:644-671):
 * "fill2d(critx,cor,maxLoop)", "creepfill2d(repeat,weight)" or "creepfill2d(repeat,weight,defaultValue)" (weight is ONE
 * CHARACTER and its code is the weight, as in the reference: "2" means 50).  They run on the device inside the slice calls
 * below (before / after the gather, :256, :284) and switch the fused adapters to the three-pass form.  Part of construction:
 * call before the handle is shared between threads. */
int fb200_interp_add_preprocess(fb200_interp* handle, const char* procString);
int fb200_interp_add_postprocess(fb200_interp* handle, const char* procString);

int fb200_interp_get_data_slice(const fb200_interp* handle, int inType, const void* inData, size_t size, double badValue, int outType,
                                void* outData, size_t* newSize);
int fb200_interp_get_data_slice_device(const fb200_interp* handle, int inType, const void* d_inData, size_t size, double badValue,
                                       int outType, void* d_outData, size_t* newSize, void* cuda_stream);
/* the vector branch (:259-283): both components, each with its own fill value, rotated (vector may be NULL), converted */
int fb200_interp_get_vector_slice(const fb200_interp* handle, const fb200_vector* vector, int inType, const void* uIn, const void* vIn,
                                  size_t size, double badValueU, double badValueV, int outType, void* uOut, void* vOut, size_t* newSize);
int fb200_interp_get_vector_slice_device(const fb200_interp* handle, const fb200_vector* vector, int inType, const void* d_uIn,
                                         const void* d_vIn, size_t size, double badValueU, double badValueV, int outType, void* d_uOut,
                                         void* d_vOut, size_t* newSize, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * (1d) vertical interpolation to pressure levels: the pressure branch of CDMVerticalInterpolator
 *      (--verticalInterpolate.type=pressure; DESIGN.md section 2 states the arithmetic)
 *
 * Source vertical coordinates, all pressures in ONE unit, that of the target levels (hPa, as the reference's level1 option):
 *   pressure levels                          p_k = ap_k                                  (create_hybrid with b == NULL)
 *   atmosphere_hybrid_sigma_pressure_coordinate  p_k = ap_k + b_k * (ps * ps_scale)      (a, p0 form: pass ap_k = a_k * p0)
 *   atmosphere_sigma_coordinate              p_k = ptop + sigma_k * (ps * ps_scale - ptop)
 * ps_scale converts the surface pressure field to that unit (0.01 for a Pa field against hPa levels).
 * method: MIFI_VINT_METHOD_LIN 0, _LOG 1, _LOGLOG 2, _NN 3 (the reference's numbering).  extrapolate != 0: targets outside a
 * column's pressure range use the end pair of levels on that side; 0: they give NaN.  2 <= nk, np <= 1024, all values finite.
 * The handle is immutable and every call re-entrant, as for the horizontal handles.
 * ---------------------------------------------------------------------------------------------- */
#ifndef MIFI_VINT_METHOD_LIN
#define MIFI_VINT_METHOD_LIN 0
#define MIFI_VINT_METHOD_LOG 1
#define MIFI_VINT_METHOD_LOGLOG 2
#define MIFI_VINT_METHOD_NN 3
#endif
typedef struct fb200_vinterp fb200_vinterp; /* opaque */

int fb200_vinterp_create_hybrid(int method, const double* ap, const double* b, int nk, double ps_scale, const double* levels, int np,
                                int extrapolate, fb200_vinterp** handle);
int fb200_vinterp_create_sigma(int method, const double* sigma, int nk, double ptop, double ps_scale, const double* levels, int np, int extrapolate,
                               fb200_vinterp** handle);
void fb200_vinterp_destroy(fb200_vinterp* handle);
/* in: [nt][nk][nxy] floats (NaN = undefined), ps: [nt][nxy] floats (may be NULL for pressure levels), out: [nt][np][nxy] floats,
 * the target levels in the order they were given.  Host buffers (copies pipelined over the time steps) or, for _device, device
 * pointers on `cuda_stream` without synchronisation. */
int fb200_vinterp_interpolate_values(const fb200_vinterp* handle, const float* in, const float* ps, size_t nxy, size_t nt, float* out);
int fb200_vinterp_interpolate_values_device(const fb200_vinterp* handle, const float* d_in, const float* d_ps, size_t nxy, size_t nt, float* d_out,
                                            void* cuda_stream);
/* the per-slice body of the vertical getDataSlice: inType / outType as in (1c), badValue -> NaN on the way in, NaN -> badValue and
 * round + cast on the way out */
int fb200_vinterp_get_data_slice(const fb200_vinterp* handle, int inType, const void* in, const float* ps, size_t nxy, size_t nt, double badValue,
                                 int outType, void* out);
int fb200_vinterp_get_data_slice_device(const fb200_vinterp* handle, int inType, const void* d_in, const float* d_ps, size_t nxy, size_t nt,
                                        double badValue, int outType, void* d_out, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * (1e) vertical interpolation to height and altitude levels: the height branch of CDMVerticalInterpolator
 *      (--verticalInterpolate.type=height / altitude; DESIGN.md section 2 states the arithmetic)
 *
 * Targets in metres: FB200_VZ_ALTITUDE above sea level, FB200_VZ_HEIGHT above the ground.  The altitude z_k of every source level
 * comes from a converter:
 *   FB200_VZ_STANDARD     the standard-atmosphere altitude (US Standard Atmosphere 1976 / ICAO) of the column pressure p_k [hPa];
 *   FB200_VZ_HYPSOMETRIC  integrated upward from the surface over the air temperature t [K] and, when given, the specific humidity
 *                         q [kg/kg] (virtual temperature); hybrid or sigma source levels only;
 *   FB200_VZ_FIELD        z_k = z_scale * z, a per-level field (geopotential: z_scale = 1 / 9.80665; altitude: 1); the formula
 *                         terms are not used and may be NULL.
 * vcoord and a, b, ptop, ps_scale give the column pressures as for the pressure handles: FB200_VCOORD_PRESSURE (a = the levels),
 * _HYBRID (a = ap, b) or _SIGMA (b = sigma, ptop).  The surface altitude is zs * zs_scale (surface geopotential: zs_scale =
 * 1 / 9.80665); height targets of the standard and field converters and altitude targets of the hypsometric one need it.
 * method: MIFI_VINT_METHOD_LIN or _NN only (log and loglog are defined on ln p).  Other rules as for the pressure handles.
 * ---------------------------------------------------------------------------------------------- */
#define FB200_VCOORD_PRESSURE 0
#define FB200_VCOORD_HYBRID 1
#define FB200_VCOORD_SIGMA 2
#define FB200_VZ_STANDARD 0
#define FB200_VZ_HYPSOMETRIC 1
#define FB200_VZ_FIELD 2
#define FB200_VZ_ALTITUDE 0
#define FB200_VZ_HEIGHT 1
/* the per-column inputs of a call, float32, NULL = not given: ps [nt][nxy], t, q, z [nt][nk][nxy], zs [nxy] (no time axis).
 * Depth handles (1f) read two slots: ps carries the sea surface height eta [m] (NULL: 0) and zs the sea-floor depth h [m, positive
 * down]; t, q and z are not read. */
typedef struct fb200_vcolumns {
    const float* ps;
    const float* t;
    const float* q;
    const float* z;
    const float* zs;
} fb200_vcolumns;

int fb200_vinterp_create_height(int method, int converter, int target, int vcoord, const double* a, const double* b, int nk, double ptop,
                                double ps_scale, double z_scale, double zs_scale, const double* levels, int np, int extrapolate,
                                fb200_vinterp** handle);
/* The calls above with every per-column input: they take pressure handles too (only ps is read).  A height handle on the calls
 * above, which pass ps alone, fails when it needs t, z or zs.  `cols` holds host pointers, `d_cols` (itself a host struct) device
 * pointers. */
int fb200_vinterp_interpolate_values_columns(const fb200_vinterp* handle, const float* in, const fb200_vcolumns* cols, size_t nxy, size_t nt,
                                             float* out);
int fb200_vinterp_interpolate_values_columns_device(const fb200_vinterp* handle, const float* d_in, const fb200_vcolumns* d_cols, size_t nxy,
                                                    size_t nt, float* d_out, void* cuda_stream);
int fb200_vinterp_get_data_slice_columns(const fb200_vinterp* handle, int inType, const void* in, const fb200_vcolumns* cols, size_t nxy,
                                         size_t nt, double badValue, int outType, void* out);
int fb200_vinterp_get_data_slice_columns_device(const fb200_vinterp* handle, int inType, const void* d_in, const fb200_vcolumns* d_cols,
                                                size_t nxy, size_t nt, double badValue, int outType, void* d_out, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * (1f) vertical interpolation to depth levels: the depth branch of CDMVerticalInterpolator
 *      (--verticalInterpolate.type=depth; DESIGN.md section 2 states the arithmetic)
 *
 * Targets in metres below the datum of eta, positive down.  Source vertical coordinates (CF standard names), with z_k the
 * altitude of level k (negative below the datum) and x_k = -z_k:
 *   FB200_VCOORD_DEPTH           depth levels, positive down: x_k = s_k (C, depth_c not used)
 *   FB200_VCOORD_OCEAN_SIGMA     ocean_sigma_coordinate: z = eta + sigma_k * (h + eta), sigma_k = s_k
 *   FB200_VCOORD_OCEAN_S_G1      ocean_s_coordinate_g1: S = depth_c * s_k + (h - depth_c) * C_k, z = S + eta * (1 + S / h)
 *   FB200_VCOORD_OCEAN_S_G2      ocean_s_coordinate_g2: S = (depth_c * s_k + h * C_k) / (depth_c + h), z = eta + (eta + h) * S
 * eta [nt][nxy] is the sea surface height (the ps slot of fb200_vcolumns, or the ps argument of the calls without _columns; NULL
 * means 0), h [nxy] the sea-floor depth (the zs slot, no time axis).  The ocean coordinates need h, so the calls without _columns
 * refuse them; depth-level handles read neither and work on every call.  A column with h NaN or <= 0 (land), a NaN eta, or equal
 * ends of x gives NaN and reads no field value.  method: MIFI_VINT_METHOD_LIN or _NN only.  C != NULL for g1 and g2;
 * 0 <= depth_c < inf; 2 <= nk <= 1024, 1 <= np <= 1024, all values finite.  Other rules as for the height handles.
 * ---------------------------------------------------------------------------------------------- */
#define FB200_VCOORD_DEPTH 3
#define FB200_VCOORD_OCEAN_SIGMA 4
#define FB200_VCOORD_OCEAN_S_G1 5
#define FB200_VCOORD_OCEAN_S_G2 6

int fb200_vinterp_create_depth(int method, int vcoord, const double* s, const double* C, int nk, double depth_c, const double* levels, int np,
                               int extrapolate, fb200_vinterp** handle);

/* ------------------------------------------------------------------------------------------------
 * (1g) the data conversions of the vertical interpolator on the model levels (--verticalInterpolate.dataConversion, the reference's
 *      CDMPressureConversions; DESIGN.md section 2 states the arithmetic)
 *
 *   FB200_VCONV_THETA2T      air_potential_temperature theta [K] -> air_temperature T = theta * (p_k / 1000 hPa)^(2/7) [K]
 *   FB200_VCONV_OMEGA2VWIND  lagrangian_tendency_of_air_pressure omega [Pa/s] and air_temperature T [K] -> upward_air_velocity
 *                            w = -omega R_d T / (g0 p_k) [m/s], R_d = R* / M
 *   FB200_VCONV_PRESSURE     add4Dpressure: the column pressure p_k itself [hPa], an [nt][nk][nxy] field; no input field
 * vcoord, a, b, ptop and ps_scale give p_k [hPa] as for fb200_vinterp_create_height: FB200_VCOORD_PRESSURE (a = the levels), _HYBRID
 * (a = ap, b) or _SIGMA (b = sigma, ptop).  1 <= nk <= 1024, all values finite.  Float in, float out; NaN in the field, t or ps gives
 * NaN for the values it enters.  The handle is immutable and every call re-entrant, as for the other handles.
 * ---------------------------------------------------------------------------------------------- */
#define FB200_VCONV_THETA2T 0
#define FB200_VCONV_OMEGA2VWIND 1
#define FB200_VCONV_PRESSURE 2
typedef struct fb200_vconvert fb200_vconvert; /* opaque */

int fb200_vconvert_create(int op, int vcoord, const double* a, const double* b, int nk, double ptop, double ps_scale, fb200_vconvert** handle);
void fb200_vconvert_destroy(fb200_vconvert* handle);
/* in: [nt][nk][nxy] float (theta or omega; NULL for FB200_VCONV_PRESSURE); cols->ps [nt][nxy] (hybrid and sigma levels), cols->t
 * [nt][nk][nxy] (omega2vwind); the other slots are not read.  out: [nt][nk][nxy] float.  Host buffers (copies pipelined over the time
 * steps) or, for _device, device pointers on `cuda_stream` without synchronisation.  The _device form may run in place (d_out == d_in). */
int fb200_vconvert_values(const fb200_vconvert* handle, const float* in, const fb200_vcolumns* cols, size_t nxy, size_t nt, float* out);
int fb200_vconvert_values_device(const fb200_vconvert* handle, const float* d_in, const fb200_vcolumns* d_cols, size_t nxy, size_t nt,
                                 float* d_out, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * (1h) time interpolation: the linear change of the time axis of CDMTimeInterpolator (--timeInterpolate.timeSpec; DESIGN.md
 *      section 2 states the arithmetic)
 *
 * times [nt]: the source times, strictly increasing, 2 <= nt; new_times [nt_new]: the target times in any order, repeats allowed,
 * 1 <= nt_new <= 1048576; all finite and in ONE unit.  Target j takes the smallest bracket k with t_k <= tau_j <= t_k+1 and
 * w = (tau_j - t_k) / (t_k+1 - t_k) in fp64; outside [t_0, t_nt-1] the end pair on that side when extrapolate != 0, else no bracket
 * (the step is NaN, stored as badValue).  Every value: r = (float)((double)A + w * ((double)B - (double)A)), no FMA.  The slices are
 * typed as in (1c): inType in with badValue -> NaN, NaN -> badValue and round + cast to outType out (float: inType = outType =
 * FB200_FLOAT, badValue = NaN); no scale or offset is applied.  The handle is immutable and every call re-entrant.
 * ---------------------------------------------------------------------------------------------- */
typedef struct fb200_tinterp fb200_tinterp; /* opaque */

int fb200_tinterp_create(const double* times, int nt, const double* new_times, int nt_new, int extrapolate, fb200_tinterp** handle);
void fb200_tinterp_destroy(fb200_tinterp* handle);
/* the time-change map of target step j: source steps ia < ib and weight w; ia = ib = -1 where no bracket applies */
int fb200_tinterp_source_steps(const fb200_tinterp* handle, int j, int* ia, int* ib, double* w);
/* one target step from the two source slices the map names (n elements each; NULL allowed where no bracket applies): the shape of
 * the reference's getDataSlice(var, unLimDimPos).  Host buffers (copies pipelined over element chunks) or, for _device, device
 * pointers on `cuda_stream` without synchronisation. */
int fb200_tinterp_get_step(const fb200_tinterp* handle, int j, int inType, const void* a, const void* b, size_t n, double badValue, int outType,
                           void* out);
int fb200_tinterp_get_step_device(const fb200_tinterp* handle, int j, int inType, const void* d_a, const void* d_b, size_t n, double badValue,
                                  int outType, void* d_out, void* cuda_stream);
/* the whole stack on the device: d_in [nt][n] -> d_out [nt_new][n], every source step the targets need read once */
int fb200_tinterp_get_data_slice_device(const fb200_tinterp* handle, int inType, const void* d_in, size_t n, double badValue, int outType,
                                        void* d_out, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * (1i) CDMMerger: an inner (fine, small) grid merged into an outer (coarse, large) one on a target grid, with the linear border
 *      smoothing of CDMBorderSmoothing_Linear (--merge.smoothing=LINEAR(transitionWidth,borderWidth); DESIGN.md section 2 states
 *      the arithmetic)
 *
 * The handle BORROWS three interpolation handles of (1a) -- the caller keeps them alive, as with fb200_vector in
 * fb200_interp_get_vector_slice: outerToInner reads the outer grid and writes the inner grid, innerToTarget reads the inner grid,
 * outerToTarget reads the outer grid, and both write the same target grid.  Each may carry a reduced domain (createReducedDomain);
 * the slabs are cropped to it inside.  All three use nearest neighbour, bilinear or bicubic, on one device.  transitionWidth >= 1
 * (the blend divides by it), borderWidth >= 0.  create refuses anything else with MIFI_ERROR and a message.
 *
 * One slice: outer -> inner grid, the border blend on the inner grid, blended inner -> target, outer -> target, and the overlay
 * (the blended inner where defined, else the outer).  inner [nz][innerY][innerX] and outer [nz][outerY][outerX] (the full grids,
 * same nz; innerSize and outerSize in values) are both of inType; the inner value equal to badInner cast to inType and the outer
 * value whose float equals (float)badOuter (mifi_bad2nanf, as the gathers of (1c)) are undefined; NaN never matches.  out
 * [nz][outY][outX] of outType, undefined -> outFill, rounded and cast as in (1c); *newSize receives its number of values.  No
 * scale or offset is applied.  The host form uploads inner and outer once and downloads out once, pipelined over level chunks;
 * _device takes device pointers and enqueues everything on cuda_stream without synchronising.  The device chain keeps at most
 * 256 MB of float intermediates (or one level, where one level needs more).  The handle is immutable and every call re-entrant.
 * ---------------------------------------------------------------------------------------------- */
typedef struct fb200_merge fb200_merge; /* opaque */

int fb200_merge_create(const fb200_interp* outerToInner, const fb200_interp* innerToTarget, const fb200_interp* outerToTarget, size_t innerX,
                       size_t innerY, size_t outerX, size_t outerY, int transitionWidth, int borderWidth, int useOuterIfInnerUndefined,
                       fb200_merge** handle);
void fb200_merge_destroy(fb200_merge* handle);
int fb200_merge_get_data_slice(const fb200_merge* handle, int inType, const void* inner, size_t innerSize, double badInner, const void* outer,
                               size_t outerSize, double badOuter, int outType, double outFill, void* out, size_t* newSize);
int fb200_merge_get_data_slice_device(const fb200_merge* handle, int inType, const void* d_inner, size_t innerSize, double badInner,
                                      const void* d_outer, size_t outerSize, double badOuter, int outType, double outFill, void* d_out,
                                      size_t* newSize, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * (2) the reference's C symbols for this path -- include/fimex/interpolation.h (line of each prototype given)
 * ---------------------------------------------------------------------------------------------- */
int mifi_string_to_interpolation_method(const char* stringMethod); /* :44 */

int mifi_interpolate_f(int method, const char* proj_input, const float* infield, const double* in_x_axis, const double* in_y_axis,
                       const int in_x_axis_type, const int in_y_axis_type, const int ix, const int iy, const int iz,
                       const char* proj_output, float* outfield, const double* out_x_axis, const double* out_y_axis,
                       const int out_x_axis_type, const int out_y_axis_type, const int ox, const int oy); /* :71-75 */

int mifi_vector_reproject_values_f(int method, const char* proj_input, const char* proj_output, float* u_out, float* v_out,
                                   const double* out_x_axis, const double* out_y_axis, int out_x_axis_type, int out_y_axis_type, int ox,
                                   int oy, int oz); /* :124-130 */
int mifi_vector_reproject_values_by_matrix_f(int method, const double* matrix, float* u_out, float* v_out, int ox, int oy,
                                             int oz); /* :142-145 */
int mifi_vector_reproject_direction_by_matrix_f(int method, const double* matrix, float* angle_out, int ox, int oy, int oz); /* :158-161 */
int mifi_get_vector_reproject_matrix(const char* proj_input, const char* proj_output, const double* out_x_axis, const double* out_y_axis,
                                     int out_x_axis_type, int out_y_axis_type, int ox, int oy, double* matrix); /* :177-182 */
int mifi_get_vector_reproject_matrix_field(const char* proj_input, const char* proj_output, const double* in_x_field,
                                           const double* in_y_field, int ox, int oy, double* matrix); /* :197-201 */
int mifi_get_vector_reproject_matrix_points(const char* proj_input, const char* proj_output, int inputIsMetric, const double* out_x_points,
                                            const double* out_y_points, int on, double* matrix); /* :216-222 */

/* per-point gathers (:231, :274, :291).  Exported for link compatibility; each call moves the whole field to
 * the device, so use the handle API for anything but spot checks. */
int mifi_get_values_f(const float* infield, float* outfield, const double x, const double y, const int ix, const int iy, const int iz);
int mifi_get_values_bilinear_f(const float* infield, float* outvalues, const double x, const double y, const int ix, const int iy,
                               const int iz);
int mifi_get_values_bicubic_f(const float* infield, float* outvalues, const double x, const double y, const int ix, const int iy,
                              const int iz);

int mifi_points2position(double* points, const int n, const double* axis, const int num, const int axis_type); /* :415 */
int mifi_project_values(const char* proj_input, const char* proj_output, double* in_out_x_vals, double* in_out_y_vals,
                        const int num); /* :443 */
int mifi_project_axes(const char* proj_input, const char* proj_output, const double* in_x_axis, const double* in_y_axis, const int ix,
                      const int iy, double* out_xproj_axis, double* out_yproj_axis); /* :461 */

/* bad <-> NaN adapters on either side of the path (src/interpolation.c:1775-1793); :586-587 */
size_t mifi_bad2nanf(float* posPtr, float* endPtr, float badVal);
size_t mifi_nanf2bad(float* posPtr, float* endPtr, float badVal);

/* The 2-D pre/post-processes of getDataSlice (--interpolate.preprocess / postprocess, src/CDMInterpolator.cc:126-159, 256, 284;
 * include/fimex/interpolation.h:520-560): same prototypes as the reference, one level of host data per call.  nx, ny >= 2. */
int mifi_fill2d_f(size_t nx, size_t ny, float* field, float relaxCrit, float corrEff, size_t maxLoop, size_t* nChanged);
int mifi_creepfill2d_f(size_t nx, size_t ny, float* field, unsigned short repeat, char setWeight, size_t* nChanged);
int mifi_creepfillval2d_f(size_t nx, size_t ny, float* field, float defaultVal, unsigned short repeat, char setWeight, size_t* nChanged);
/* the same for nz levels resident on the device, in place (processArray_, src/CDMInterpolator.cc:136-159): one CTA per level
 * walks the anti-diagonals of the lexicographic Gauss-Seidel sweeps, so results are bit-identical to the reference.
 * useDefaultVal != 0: creepfillval2d(defaultVal), else creepfill2d (mean of the defined values as first guess). */
int fb200_fill2d_device(float* d_field, size_t nx, size_t ny, size_t nz, float relaxCrit, float corrEff, size_t maxLoop, void* cuda_stream);
int fb200_creepfill2d_device(float* d_field, size_t nx, size_t ny, size_t nz, int useDefaultVal, float defaultVal, unsigned short repeat,
                             char setWeight, void* cuda_stream);

/* ThreadPool.c's knob (src/ThreadPool.c:33-46): kept as a symbol, has no effect on this path */
int mifi_setNumThreads(int n);

#ifdef __cplusplus
}
#endif

#endif /* FIMEX_B200_H_ */
