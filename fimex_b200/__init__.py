"""fimex_b200 -- Fimex's horizontal-regridding hot path on NVIDIA B200, behind Fimex's own interface.

The product is ``fimex_b200/lib/libfimex_b200.so`` (hand-written sm_100a CUDA behind the C ABI of
``include/fimex_b200.h``).  This package is the thin Python host side used by the tests and the benchmark:

* :mod:`fimex_b200.capi`    -- ctypes binding of every entry point of the header (fails loudly if the library
  is missing or no GPU is usable; there is no CPU fallback anywhere in this package);
* :mod:`fimex_b200.cached`  -- mirrors of the reference's ``CachedInterpolation``,
  ``CachedForwardInterpolation`` and ``CachedVectorReprojection`` classes (same constructor arguments, same
  method names) working on numpy arrays (host path) or torch CUDA tensors (device-resident path);
* :mod:`fimex_b200.interpolator` -- the table-producing part of ``CDMInterpolator::changeProjection*`` and the
  per-slice driver ``getDataSlice`` for in-memory slices;
* :mod:`fimex_b200.processor` -- ``CDMProcessor::rotateVectorToLatLon`` / ``rotateDirectionToLatLon`` on the same rotation kernels;
* :mod:`fimex_b200.vertical` -- the pressure, height and depth branches of ``CDMVerticalInterpolator`` (model levels -> pressure, height,
  altitude or depth levels) and its data conversions (``PressureConversion``: theta2T, omega2vwind, add4Dpressure) on the GPU;
* :mod:`fimex_b200.timeinterp` -- the linear change of the time axis of ``CDMTimeInterpolator`` (``TimeInterpolator``) on the GPU;
* :mod:`fimex_b200.merger` -- ``CDMMerger`` (inner grid merged into an outer one with linear border smoothing): the three gathers, the
  blend and the overlay of a merged slice in one call on the GPU;
* :mod:`fimex_b200.slab`    -- one-process-per-GPU slab partition of the (time x level) stack with a single
  NCCL broadcast of the cached tables.
"""
from .capi import (DataType, cdm_type, default_fill_value, LATITUDE, LONGITUDE, PROJ_AXIS, MIFI_ERROR, MIFI_OK, MIFI_VECTOR_KEEP_SIZE, FimexB200Error, Method, kernel_launches,
                   last_error, lib_path, load, mifi_get_values_bicubic_f, mifi_get_values_bilinear_f, mifi_get_values_f,
                   mifi_get_vector_reproject_matrix, mifi_get_vector_reproject_matrix_field, mifi_get_vector_reproject_matrix_points,
                   mifi_interpolate_f, mifi_points2position, mifi_project_axes, mifi_project_values, mifi_string_to_interpolation_method,
                   mifi_vector_reproject_direction_by_matrix_f, mifi_vector_reproject_values_by_matrix_f, mifi_vector_reproject_values_f,
                   mifi_bad2nanf, mifi_nanf2bad, mifi_fill2d_f, mifi_creepfill2d_f, fill2d_device, creepfill2d_device, set_device,
                   version)
from .cached import CachedForwardInterpolation, CachedInterpolation, CachedVectorReprojection
from .interpolator import Interpolator, axis_spec_requires_start_end, spatial_axis_spec, tokenize_dotted
from .processor import Processor
from .merger import Merger, extend_inner_axis, linear_border_smoothing, parse_smoothing
from .timeinterp import TimeInterpolator
from .vertical import DepthInterpolator, HeightInterpolator, PressureConversion, VerticalInterpolator, vertical_method

#: opt-in arithmetic modes of the bicubic gather (environment, read at every launch): FIMEX_B200_BICUBIC_FP32=1 (fp32 weights and
#: FMAs, <= 1e-5 relative, identical NaN masks), FIMEX_B200_BICUBIC_CONTRACT=1 (fp64 FMA chains); default: bit-identical
BICUBIC_FP32_AVAILABLE = True

__all__ = [
    "CachedInterpolation", "CachedForwardInterpolation", "CachedVectorReprojection", "Interpolator", "Processor", "Merger", "VerticalInterpolator", "HeightInterpolator", "DepthInterpolator", "PressureConversion", "TimeInterpolator", "vertical_method", "extend_inner_axis", "linear_border_smoothing", "parse_smoothing", "spatial_axis_spec", "axis_spec_requires_start_end", "tokenize_dotted", "Method", "DataType", "cdm_type", "default_fill_value", "FimexB200Error",
    "MIFI_OK", "MIFI_ERROR", "PROJ_AXIS", "LONGITUDE", "LATITUDE", "MIFI_VECTOR_KEEP_SIZE", "load", "lib_path", "version", "last_error",
    "set_device", "kernel_launches", "mifi_interpolate_f", "mifi_points2position", "mifi_project_axes", "mifi_project_values",
    "mifi_get_vector_reproject_matrix", "mifi_get_vector_reproject_matrix_field", "mifi_get_vector_reproject_matrix_points",
    "mifi_vector_reproject_values_by_matrix_f", "mifi_vector_reproject_direction_by_matrix_f", "mifi_vector_reproject_values_f",
    "mifi_get_values_f", "mifi_get_values_bilinear_f", "mifi_get_values_bicubic_f", "mifi_string_to_interpolation_method",
    "mifi_bad2nanf", "mifi_nanf2bad", "mifi_fill2d_f", "mifi_creepfill2d_f", "fill2d_device", "creepfill2d_device",
]
