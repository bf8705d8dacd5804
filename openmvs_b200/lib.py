"""ctypes binding of include/b200mvs.h.  There is no CPU fallback: if the CUDA library is
missing or no GPU is present, calls raise."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

MAX_VIEWS = 32
ABI_VERSION = 5  # B200MVS_ABI_VERSION of include/b200mvs.h these structs mirror


class View(C.Structure):
	"""b200mvs_view"""
	_fields_ = [("image", C.c_void_p), ("width", C.c_int), ("height", C.c_int), ("stride_bytes", C.c_int),
		("K", C.c_double*9), ("R", C.c_double*9), ("C", C.c_double*3),
		("depth", C.c_void_p), ("dwidth", C.c_int), ("dheight", C.c_int), ("dstride_bytes", C.c_int),
		("Kd", C.c_double*9), ("Rd", C.c_double*9), ("Cd", C.c_double*3),
		("image8", C.c_void_p), ("channels8", C.c_int), ("bgr8", C.c_int), ("stride8_bytes", C.c_int)]


class Params(C.Structure):
	"""b200mvs_params"""
	_fields_ = [("nEstimationIters", C.c_int), ("nEstimationGeometricIters", C.c_int), ("nRandomIters", C.c_int),
		("nSubResolutionLevels", C.c_int),
		("fNCCThresholdKeep", C.c_float), ("fDescriptorMinMagnitudeThreshold", C.c_float),
		("fRandomDepthRatio", C.c_float), ("fRandomAngle1Range", C.c_float), ("fRandomAngle2Range", C.c_float),
		("fRandomSmoothDepth", C.c_float), ("fRandomSmoothNormal", C.c_float), ("fRandomSmoothBonus", C.c_float),
		("fEstimationGeometricWeight", C.c_float),
		("nSweepsPerIter", C.c_int), ("nPropagation", C.c_int), ("seed", C.c_uint32),
		("nPropagationFar", C.c_int), ("bSkipUnchanged", C.c_int), ("nEvalCap", C.c_int)]


class Debug(C.Structure):
	"""b200mvs_debug"""
	_fields_ = [("scalarTaps", C.c_int), ("noTMA", C.c_int), ("sgmAggregation", C.c_int), ("sgmCost", C.c_int),
		("sweepFourCtas", C.c_int), ("frontLayout", C.c_int), ("frontSerial", C.c_int), ("frontBlock", C.c_int), ("frontLag", C.c_int),
		("frontCtas", C.c_int), ("frontDepth", C.c_int), ("frontSubCell", C.c_int), ("reserved", C.c_int*4)]


class Stats(C.Structure):
	"""b200mvs_stats"""
	_fields_ = [("ms_total", C.c_double), ("ms_device", C.c_double), ("bytes_h2d", C.c_uint64), ("bytes_d2h", C.c_uint64),
		("kernel_launches", C.c_int), ("levels", C.c_int),
		("ms_sweep_kernels", C.c_double), ("sweep_launches", C.c_int), ("tma_active", C.c_int)]


class Job(C.Structure):
	"""b200mvs_job"""
	_fields_ = [("views", C.POINTER(View)), ("nViews", C.c_int), ("dMin", C.c_float), ("dMax", C.c_float), ("nGeometricIter", C.c_int),
		("depth", C.c_void_p), ("normal", C.c_void_p), ("conf", C.c_void_p), ("viewsMap", C.c_void_p), ("status", C.c_int)]


class SgmPixel(C.Structure):
	"""b200mvs_sgm_pixel"""
	_fields_ = [("idx", C.c_uint64), ("dmin", C.c_int16), ("dmax", C.c_int16), ("reserved", C.c_int32)]


class SgmParams(C.Structure):
	"""b200mvs_sgm_params"""
	_fields_ = [("P1", C.c_int), ("P2", C.c_int), ("P2alpha", C.c_float), ("P2beta", C.c_float)]


class DMap(C.Structure):
	"""b200mvs_dmap"""
	_fields_ = [("depth", C.c_void_p), ("conf", C.c_void_p), ("width", C.c_int), ("height", C.c_int),
		("K", C.c_double*9), ("R", C.c_double*9), ("C", C.c_double*3)]


class FilterParams(C.Structure):
	"""b200mvs_filter_params"""
	_fields_ = [("nMinViews", C.c_int), ("nMinViewsAdjust", C.c_int), ("fDepthDiffThreshold", C.c_float), ("bAdjust", C.c_int)]


class FuseView(C.Structure):
	"""b200mvs_fuse_view"""
	_fields_ = [("width", C.c_int), ("height", C.c_int), ("depth", C.c_void_p), ("normal", C.c_void_p), ("conf", C.c_void_p),
		("color", C.c_void_p), ("K", C.c_double*9), ("R", C.c_double*9), ("C", C.c_double*3), ("neighbors", C.c_void_p),
		("nNeighbors", C.c_int), ("nSceneNeighbors", C.c_int)]


class FuseParams(C.Structure):
	"""b200mvs_fuse_params"""
	_fields_ = [("nMinViewsFuse", C.c_int), ("fDepthDiffThreshold", C.c_float), ("fNormalDiffThreshold", C.c_float),
		("bEstimateColor", C.c_int), ("bEstimateNormal", C.c_int)]


MAX_FILTER_VIEWS = 16

# every symbol include/b200mvs.h declares (checked by tests/test_capi_symbols.py)
SYMBOLS = [
	"b200mvs_create", "b200mvs_destroy", "b200mvs_default_params", "b200mvs_set_params", "b200mvs_last_error",
	"b200mvs_set_debug", "b200mvs_get_schedule", "b200mvs_abi_version", "b200mvs_sizeof", "b200mvs_set_ignore_mask",
	"b200mvs_device_count", "b200mvs_estimate", "b200mvs_estimate_device", "b200mvs_estimate_async", "b200mvs_sync", "b200mvs_estimate_batch",
	"b200mvs_pm_pack", "b200mvs_pm_unpack", "b200mvs_pm_score", "b200mvs_pm_sweep", "b200mvs_pm_finalize",
	"b200mvs_sgm_default_params", "b200mvs_sgm_match", "b200mvs_sgm_match_device",
	"b200mvs_sgm_cross_check_device", "b200mvs_sgm_refine_device",
	"b200mvs_sgm_tsgm_levels", "b200mvs_sgm_match_tsgm_device", "b200mvs_sgm_match_tsgm", "b200mvs_sgm_range_map_device",
	"b200mvs_sgm_flip_direction_device", "b200mvs_sgm_filter_speckles_device", "b200mvs_sgm_extract_mask_device",
	"b200mvs_sgm_upscale_mask_device", "b200mvs_resize_area_bgr8_device",
	"b200mvs_filter_default_params", "b200mvs_filter_depth_map", "b200mvs_filter_depth_map_device",
	"b200mvs_remove_small_segments", "b200mvs_remove_small_segments_device",
	"b200mvs_gap_interpolation", "b200mvs_gap_interpolation_device",
	"b200mvs_to_gray_device", "b200mvs_scaled_size", "b200mvs_scale_image_device",
	"b200mvs_fuse_default_params", "b200mvs_fuse_depth_maps", "b200mvs_pointcloud_size", "b200mvs_pointcloud_depths",
	"b200mvs_pointcloud_points", "b200mvs_pointcloud_normals", "b200mvs_pointcloud_colors", "b200mvs_pointcloud_view_offsets",
	"b200mvs_pointcloud_views", "b200mvs_pointcloud_weights", "b200mvs_pointcloud_projs", "b200mvs_pointcloud_free",
]

_LIB = None


def load(build_if_missing: bool = True):
	"""Load libb200mvs.so (building it in-tree when stale and nvcc is available)."""
	global _LIB
	if _LIB is not None:
		return _LIB
	path = _build.LIB_PATH
	if build_if_missing:
		# a stale library whose rebuild fails is NOT used: its struct layouts may differ from these bindings
		path = _build.build_extension()
	if not os.path.exists(path):
		raise RuntimeError("CUDA extension %s is missing: run __graft_entry__.build() (no CPU fallback exists)" % path)
	lib = C.CDLL(path)
	if not hasattr(lib, "b200mvs_abi_version") or lib.b200mvs_abi_version() != ABI_VERSION:
		raise RuntimeError("%s was built from another version of include/b200mvs.h (ABI %s, bindings %d): rebuild it" % (
			path, lib.b200mvs_abi_version() if hasattr(lib, "b200mvs_abi_version") else "?", ABI_VERSION))
	lib.b200mvs_sizeof.restype = C.c_size_t
	lib.b200mvs_sizeof.argtypes = [C.c_int]
	for what, T in enumerate((View, Params, Stats, Job, SgmPixel, SgmParams, DMap, FilterParams, Debug)):
		if lib.b200mvs_sizeof(what) != C.sizeof(T):
			raise RuntimeError("struct %s: library %d bytes, bindings %d bytes" % (T.__name__, lib.b200mvs_sizeof(what), C.sizeof(T)))
	lib.b200mvs_last_error.restype = C.c_char_p
	lib.b200mvs_last_error.argtypes = [C.c_void_p]
	lib.b200mvs_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
	lib.b200mvs_destroy.argtypes = [C.c_void_p]
	lib.b200mvs_set_params.argtypes = [C.c_void_p, C.POINTER(Params)]
	lib.b200mvs_default_params.argtypes = [C.POINTER(Params)]
	lib.b200mvs_set_debug.argtypes = [C.c_void_p, C.POINTER(Debug)]
	lib.b200mvs_get_schedule.argtypes = [C.POINTER(Params), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
	lib.b200mvs_set_ignore_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
	F = C.c_float
	P = C.c_void_p
	lib.b200mvs_estimate.argtypes = [P, C.POINTER(View), C.c_int, F, F, C.c_int, P, P, P, P, C.POINTER(Stats)]
	lib.b200mvs_estimate_async.argtypes = [P, C.POINTER(View), C.c_int, F, F, C.c_int, P, P, P, P]
	lib.b200mvs_sync.argtypes = [P, C.POINTER(Stats)]
	lib.b200mvs_estimate_batch.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(Job), C.c_int]
	lib.b200mvs_estimate_device.argtypes = [P, C.POINTER(View), C.c_int, F, F, C.c_int, P, P, P, P, P, C.POINTER(Stats)]
	lib.b200mvs_pm_pack.argtypes = [P, C.c_int, C.c_int, P, P, P, P]
	lib.b200mvs_pm_unpack.argtypes = [P, C.c_int, C.c_int, P, P, P, P]
	lib.b200mvs_pm_score.argtypes = [P, C.POINTER(View), C.c_int, F, F, P, P, P, P]
	lib.b200mvs_pm_sweep.argtypes = [P, C.POINTER(View), C.c_int, F, F, P, C.c_int, C.c_int, C.c_int, P, P, P]
	lib.b200mvs_pm_finalize.argtypes = [P, C.c_int, C.c_int, F, P, P, P, P, P, P]
	lib.b200mvs_sgm_default_params.argtypes = [C.POINTER(SgmParams)]
	lib.b200mvs_sgm_match.argtypes = [P, P, P, P, C.c_int, C.c_int, P, C.c_uint64, C.POINTER(SgmParams), P, P, C.POINTER(Stats)]
	lib.b200mvs_sgm_match_device.argtypes = [P, P, P, P, C.c_int, C.c_int, P, C.c_uint64, C.POINTER(SgmParams), C.c_int, P, P, P, P, P, C.POINTER(Stats)]
	lib.b200mvs_fuse_default_params.argtypes = [C.POINTER(FuseParams)]
	lib.b200mvs_fuse_depth_maps.argtypes = [C.POINTER(FuseView), C.c_int, C.POINTER(FuseParams), C.POINTER(C.c_void_p)]
	for name, rt in (("size", C.c_uint64), ("depths", C.c_uint64), ("points", C.POINTER(C.c_float)), ("normals", C.POINTER(C.c_float)),
			("colors", C.POINTER(C.c_uint8)), ("view_offsets", C.POINTER(C.c_uint32)), ("views", C.POINTER(C.c_uint32)),
			("weights", C.POINTER(C.c_float)), ("projs", C.POINTER(C.c_uint16))):
		f = getattr(lib, "b200mvs_pointcloud_"+name)
		f.restype = rt; f.argtypes = [C.c_void_p]
	lib.b200mvs_pointcloud_free.argtypes = [C.c_void_p]
	lib.b200mvs_pointcloud_free.restype = None
	lib.b200mvs_sgm_cross_check_device.argtypes = [P, P, P, C.c_int, C.c_int, C.c_int, P]
	lib.b200mvs_sgm_refine_device.argtypes = [P, P, P, P, C.c_int, C.c_int, P]
	I = C.c_int
	lib.b200mvs_sgm_tsgm_levels.argtypes = [I, I, I, C.POINTER(I), C.POINTER(I), C.POINTER(I)]
	lib.b200mvs_sgm_match_tsgm_device.argtypes = [P, P, P, P, P, I, I, P, P, I, I, P, I, I, I, I, I, C.POINTER(SgmParams), P, P, P, C.POINTER(Stats)]
	lib.b200mvs_sgm_match_tsgm.argtypes = [P, P, P, P, P, I, I, P, P, I, I, P, I, I, I, I, I, C.POINTER(SgmParams), P, P, C.POINTER(Stats)]
	lib.b200mvs_sgm_range_map_device.argtypes = [P, P, I, I, P, I, I, I, I, P, C.POINTER(C.c_uint64), C.POINTER(I), P]
	lib.b200mvs_sgm_flip_direction_device.argtypes = [P, P, P, I, I, P]
	lib.b200mvs_sgm_filter_speckles_device.argtypes = [P, P, I, I, I, I, I, P]
	lib.b200mvs_sgm_extract_mask_device.argtypes = [P, P, P, I, I, I, P]
	lib.b200mvs_sgm_upscale_mask_device.argtypes = [P, P, I, I, P, I, I, P]
	lib.b200mvs_resize_area_bgr8_device.argtypes = [P, P, I, I, I, P, P]
	lib.b200mvs_filter_default_params.argtypes = [C.POINTER(FilterParams)]
	lib.b200mvs_filter_depth_map.argtypes = [P, C.POINTER(DMap), C.POINTER(DMap), C.c_int, C.POINTER(FilterParams), F, F, P, P,
		C.POINTER(C.c_int), C.POINTER(Stats)]
	lib.b200mvs_filter_depth_map_device.argtypes = [P, C.POINTER(DMap), C.POINTER(DMap), C.c_int, C.POINTER(FilterParams), F, F, P, P, P, P,
		C.POINTER(C.c_int), P]
	lib.b200mvs_remove_small_segments.argtypes = [P, P, P, P, C.c_int, C.c_int, F, C.c_uint, C.POINTER(Stats)]
	lib.b200mvs_remove_small_segments_device.argtypes = [P, P, P, P, C.c_int, C.c_int, F, C.c_uint, P]
	lib.b200mvs_gap_interpolation.argtypes = [P, P, P, P, C.c_int, C.c_int, F, C.c_uint, C.POINTER(Stats)]
	lib.b200mvs_gap_interpolation_device.argtypes = [P, P, P, P, C.c_int, C.c_int, F, C.c_uint, P]
	lib.b200mvs_to_gray_device.argtypes = [P, P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, C.c_int, P]
	lib.b200mvs_scaled_size.argtypes = [C.c_int, C.c_int, F, C.POINTER(C.c_int), C.POINTER(C.c_int)]
	lib.b200mvs_scale_image_device.argtypes = [P, P, C.c_int, C.c_int, C.c_int, F, P, C.POINTER(C.c_int), P]
	_LIB = lib
	return lib


class B200MVSError(RuntimeError):
	pass


def check(lib, ctx, rc: int, what: str):
	if rc != 0:
		msg = lib.b200mvs_last_error(ctx).decode() if ctx else ""
		raise B200MVSError("%s failed with status %d: %s" % (what, rc, msg))
