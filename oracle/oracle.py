"""ctypes binding of the CPU oracle (TEST INFRASTRUCTURE — see oracle.h).

Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference) may
import this module.  The product package openmvs_b200 never does.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class OView(C.Structure):
	_fields_ = [("image", C.c_void_p), ("width", C.c_int), ("height", C.c_int),
		("K", C.c_double*9), ("R", C.c_double*9), ("C", C.c_double*3),
		("depth", C.c_void_p), ("dwidth", C.c_int), ("dheight", C.c_int),
		("Kd", C.c_double*9), ("Rd", C.c_double*9), ("Cd", C.c_double*3)]


class OParams(C.Structure):
	_fields_ = [("nEstimationIters", C.c_int), ("nEstimationGeometricIters", C.c_int), ("nRandomIters", C.c_int),
		("fNCCThresholdKeep", C.c_float), ("fDescriptorMinMagnitudeThreshold", C.c_float),
		("fRandomDepthRatio", C.c_float), ("fRandomAngle1Range", C.c_float), ("fRandomAngle2Range", C.c_float),
		("fRandomSmoothDepth", C.c_float), ("fRandomSmoothNormal", C.c_float), ("fRandomSmoothBonus", C.c_float),
		("fEstimationGeometricWeight", C.c_float), ("nSubResolutionLevels", C.c_int),
		("schedule", C.c_int), ("propagation", C.c_int), ("seed", C.c_uint32), ("threads", C.c_int)]


def build(force: bool = False) -> str:
	so = os.path.join(_HERE, "liboracle.so")
	srcs = [os.path.join(_HERE, f) for f in ("pm_oracle.cpp", "sgm_oracle.cpp", "filter_oracle.cpp", "oracle.h")]
	if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs if os.path.exists(s)):
		subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
	return so


_FAST_SO = None


def build_fast() -> str:
	"""Throughput build of the same sources (-O3 -march=native, FP contraction allowed) for the CPU baseline of bench.py.  It is
	compiled once per process into a temporary directory: -march=native code must not travel, and the tree may be read-only."""
	global _FAST_SO
	if _FAST_SO is None:
		tmp = tempfile.mkdtemp(prefix="oracle_fast_")
		atexit.register(shutil.rmtree, tmp, True)
		so = os.path.join(tmp, "liboracle_fast.so")
		subprocess.check_call(["make", "-C", _HERE, "-s", "FAST_SO="+so, so])
		_FAST_SO = so
	return _FAST_SO


_LIBS = {}
_FAST = False


def use_fast_build(on: bool) -> bool:
	"""Route the calls of this module to the throughput build (True) or back to the parity build (False).  Returns True when
	the fast build is in use.  Parity tests never call this: they run the -O2 -ffp-contract=off build."""
	global _FAST, _LIB
	if on:
		try:
			build_fast()
		except Exception:
			return False
	_FAST = bool(on)
	_LIB = None
	return _FAST


def lib():
	global _LIB
	if _LIB is None:
		key = "fast" if _FAST else "parity"
		if key not in _LIBS:
			L = C.CDLL(build_fast() if _FAST else build())
			L.oracle_pm_score_pixel.restype = C.c_float
			L.oracle_interpolate_pixel.restype = C.c_float
			_LIBS[key] = L
		_LIB = _LIBS[key]
	return _LIB


def default_params(**kw) -> OParams:
	p = OParams()
	lib().oracle_default_params(C.byref(p))
	for k, v in kw.items():
		if not hasattr(p, k):
			raise AttributeError(k)
		setattr(p, k, v)
	return p


def _fptr(a):
	return a.ctypes.data_as(C.c_void_p)


def make_views(views, depths=None):
	"""views: list of objects with .image .K .R .C (reference first); depths: optional list of
	(depth, K, R, C) or None per view. Returns (ctypes array, keepalive)."""
	arr = (OView*len(views))()
	keep = []
	for i, v in enumerate(views):
		img = np.ascontiguousarray(v.image, np.float32)
		keep.append(img)
		o = arr[i]
		o.image = _fptr(img); o.width = img.shape[1]; o.height = img.shape[0]
		o.K[:] = np.asarray(v.K, np.float64).ravel(); o.R[:] = np.asarray(v.R, np.float64).ravel(); o.C[:] = np.asarray(v.C, np.float64).ravel()
		o.depth = None
		if depths is not None and depths[i] is not None:
			d, Kd, Rd, Cd = depths[i]
			d = np.ascontiguousarray(d, np.float32)
			keep.append(d)
			o.depth = _fptr(d); o.dwidth = d.shape[1]; o.dheight = d.shape[0]
			o.Kd[:] = np.asarray(Kd, np.float64).ravel(); o.Rd[:] = np.asarray(Rd, np.float64).ravel(); o.Cd[:] = np.asarray(Cd, np.float64).ravel()
	return arr, keep


def _state(views, depth, normal):
	h, w = views[0].image.shape
	d = np.zeros((h, w), np.float32) if depth is None else np.array(depth, np.float32, copy=True, order="C")
	n = np.zeros((h, w, 3), np.float32) if normal is None else np.array(normal, np.float32, copy=True, order="C")
	c = np.zeros((h, w), np.float32)
	return d, n, c


def pm_score(views, prm, dmin, dmax, depth=None, normal=None, lowres=None, depths=None):
	arr, keep = make_views(views, depths)
	d, n, c = _state(views, depth, normal)
	lr = None if lowres is None else np.ascontiguousarray(lowres, np.float32)
	rc = lib().oracle_pm_score(arr, len(views), C.byref(prm), C.c_float(dmin), C.c_float(dmax),
		None if lr is None else _fptr(lr), _fptr(d), _fptr(n), _fptr(c))
	assert rc == 0
	return d, n, c


def pm_iterate(views, prm, dmin, dmax, depth, normal, conf, it, half=-1, lowres=None, depths=None):
	arr, keep = make_views(views, depths)
	d = np.array(depth, np.float32, copy=True, order="C")
	n = np.array(normal, np.float32, copy=True, order="C")
	c = np.array(conf, np.float32, copy=True, order="C")
	lr = None if lowres is None else np.ascontiguousarray(lowres, np.float32)
	rc = lib().oracle_pm_iterate(arr, len(views), C.byref(prm), C.c_float(dmin), C.c_float(dmax),
		None if lr is None else _fptr(lr), int(it), int(half), _fptr(d), _fptr(n), _fptr(c))
	assert rc == 0
	return d, n, c


def pm_iterate_flags(views, prm, dmin, dmax, depth, normal, conf, changed, it, half=-1, lowres=None, depths=None):
	"""pm_iterate carrying the changed-flag memory (uint8 H x W, updated copy returned as 4th value)"""
	arr, keep = make_views(views, depths)
	d = np.array(depth, np.float32, copy=True, order="C")
	n = np.array(normal, np.float32, copy=True, order="C")
	c = np.array(conf, np.float32, copy=True, order="C")
	f = np.array(changed, np.uint8, copy=True, order="C")
	lr = None if lowres is None else np.ascontiguousarray(lowres, np.float32)
	rc = lib().oracle_pm_iterate_flags(arr, len(views), C.byref(prm), C.c_float(dmin), C.c_float(dmax),
		None if lr is None else _fptr(lr), int(it), int(half), _fptr(d), _fptr(n), _fptr(c), _fptr(f))
	assert rc == 0
	return d, n, c, f


def rb_propagation(nPropagation=4, nPropagationFar=2, bSkipUnchanged=1, nEvalCap=0):
	"""oracle_params.propagation for the engine's red-black schedule (include/b200mvs.h b200mvs_params)"""
	return int(nPropagation) | (int(nPropagationFar) << 4) | (0x100 if bSkipUnchanged else 0) | (int(nEvalCap) << 12)


def pm_estimate_range(views, prm, dmin, dmax, it_begin, it_end, geometric=False, mask=None, depth=None, normal=None, depths=None):
	"""passes A, B (iterations / RB sweeps [it_begin, it_end)), C with the scale loop (photometric) and an optional ignore-mask"""
	arr, keep = make_views(views, depths)
	d, n, c = _state(views, depth, normal)
	m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
	rc = lib().oracle_pm_estimate_range(arr, len(views), C.byref(prm), C.c_float(dmin), C.c_float(dmax), int(bool(geometric)),
		int(it_begin), int(it_end), None if m is None else _fptr(m), _fptr(d), _fptr(n), _fptr(c))
	assert rc == 0
	return d, n, c


def pm_finalize(depth, normal, conf, keep):
	d = np.array(depth, np.float32, copy=True, order="C")
	n = np.array(normal, np.float32, copy=True, order="C")
	c = np.array(conf, np.float32, copy=True, order="C")
	lib().oracle_pm_finalize(d.shape[1], d.shape[0], C.c_float(keep), _fptr(d), _fptr(n), _fptr(c))
	return d, n, c


def pm_estimate(views, prm, dmin, dmax, geometric_iter=-1, depth=None, normal=None, depths=None):
	arr, keep = make_views(views, depths)
	d, n, c = _state(views, depth, normal)
	rc = lib().oracle_pm_estimate(arr, len(views), C.byref(prm), C.c_float(dmin), C.c_float(dmax),
		int(geometric_iter), _fptr(d), _fptr(n), _fptr(c))
	assert rc == 0
	return d, n, c


def pm_score_pixel(views, prm, dmin, dmax, x, y, depth, normal, close=None, lowres=None, depths=None):
	arr, keep = make_views(views, depths)
	nrm = (C.c_float*3)(*[float(v) for v in normal])
	cl = np.zeros((0, 7), np.float32) if close is None else np.ascontiguousarray(close, np.float32).reshape(-1, 7)
	vs = np.zeros(len(views)-1, np.float32)
	lr = None if lowres is None else np.ascontiguousarray(lowres, np.float32)
	s = lib().oracle_pm_score_pixel(arr, len(views), C.byref(prm), C.c_float(dmin), C.c_float(dmax),
		None if lr is None else _fptr(lr), int(x), int(y), C.c_float(depth), nrm,
		_fptr(cl) if len(cl) else None, len(cl), _fptr(vs))
	return float(s), vs


def philox(ctr, key):
	c = (C.c_uint32*4)(*ctr); k = (C.c_uint32*2)(*key); o = (C.c_uint32*4)()
	lib().oracle_philox4x32(c, k, o)
	return [int(v) for v in o]


def sgm_match(left_gray, left_bgr, right_gray, pixels, num_costs, P1=3, P2=4, alpha=14.0, beta=38.0, stage=3, costs=None):
	"""-> (costs u8, accums u16, disparity i16, cost u16); costs given => skip the cost stage"""
	lg = np.ascontiguousarray(left_gray, np.float32); rg = np.ascontiguousarray(right_gray, np.float32)
	lc = np.ascontiguousarray(left_bgr, np.uint8)
	h, w = lg.shape
	px = np.ascontiguousarray(pixels)
	assert px.itemsize == 16 and px.size == (w-6)*(h-6)
	st = int(stage)
	if costs is None:
		c = np.zeros(num_costs, np.uint8)
	else:
		c = np.array(costs, np.uint8, copy=True); st |= 8
	a = np.zeros(num_costs, np.uint16)
	disp = np.zeros((h-6, w-6), np.int16); cost = np.zeros((h-6, w-6), np.uint16)
	f = lib().oracle_sgm_match
	f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_uint16, C.c_uint16,
		C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
	rc = f(_fptr(lg), _fptr(lc), _fptr(rg), w, h, _fptr(px), num_costs, P1, P2, alpha, beta, st, _fptr(c), _fptr(a), _fptr(disp), _fptr(cost))
	assert rc == 0
	return c, a, disp, cost


def sgm_cross_check(l2r, r2l, th=1):
	a = np.array(l2r, np.int16, copy=True, order="C"); b = np.ascontiguousarray(r2l, np.int16)
	lib().oracle_sgm_cross_check(_fptr(a), _fptr(b), a.shape[1], a.shape[0], int(th))
	return a


def sgm_refine(pixels, accums, disparity, steps=4):
	d = np.array(disparity, np.int16, copy=True, order="C")
	px = np.ascontiguousarray(pixels); a = np.ascontiguousarray(accums, np.uint16)
	lib().oracle_sgm_refine(_fptr(px), _fptr(a), _fptr(d), d.size, int(steps))
	return d


# ---- depth-map post-processing (filter_oracle.cpp) ----
class ODMap(C.Structure):
	_fields_ = [("depth", C.c_void_p), ("conf", C.c_void_p), ("width", C.c_int), ("height", C.c_int),
		("K", C.c_double*9), ("R", C.c_double*9), ("C", C.c_double*3)]


def make_dmaps(maps):
	"""maps: list of (depth HxW, conf HxW or None, K, R, C) -> (ctypes array, keepalive)"""
	arr = (ODMap*len(maps))()
	keep = []
	for i, (d, c, K, R, Cc) in enumerate(maps):
		d = np.ascontiguousarray(d, np.float32); keep.append(d)
		o = arr[i]
		o.depth = _fptr(d); o.conf = None
		if c is not None:
			c = np.ascontiguousarray(c, np.float32); keep.append(c); o.conf = _fptr(c)
		o.width = d.shape[1]; o.height = d.shape[0]
		o.K[:] = np.asarray(K, np.float64).ravel(); o.R[:] = np.asarray(R, np.float64).ravel(); o.C[:] = np.asarray(Cc, np.float64).ravel()
	return arr, keep


def filter_project(ref, nbr, with_conf=True):
	arr, keep = make_dmaps([ref, nbr])
	h, w = arr[0].height, arr[0].width
	pd = np.zeros((h, w), np.float32); pc = np.zeros((h, w), np.float32)
	lib().oracle_filter_project(C.byref(arr[0]), C.byref(arr[1]), _fptr(pd), _fptr(pc) if with_conf else None)
	return pd, pc


def filter_depth_map(ref, nbrs, nMinViews=2, nMinViewsAdjust=1, fDepthDiffThreshold=0.01, bAdjust=True, dmin=0.0, dmax=1e30):
	"""ref / nbrs: (depth, conf, K, R, C).  -> (ok, depth, conf, projected N x H x W)"""
	arr, keep = make_dmaps([ref]+list(nbrs))
	h, w = arr[0].height, arr[0].width
	od = np.zeros((h, w), np.float32); oc = np.zeros((h, w), np.float32)
	proj = np.zeros((max(len(nbrs), 1), h, w), np.float32)
	nb = C.cast(C.byref(arr, C.sizeof(ODMap)), C.POINTER(ODMap))
	ok = lib().oracle_filter_depth_map(C.byref(arr[0]), nb, len(nbrs), int(nMinViews), int(nMinViewsAdjust),
		C.c_float(fDepthDiffThreshold), int(bool(bAdjust)), C.c_float(dmin), C.c_float(dmax), _fptr(od), _fptr(oc), _fptr(proj))
	return bool(ok), od, oc, proj


def remove_small_segments(depth, normal=None, conf=None, th=0.007, speckle=100):
	d = np.array(depth, np.float32, copy=True, order="C")
	n = None if normal is None else np.array(normal, np.float32, copy=True, order="C")
	c = None if conf is None else np.array(conf, np.float32, copy=True, order="C")
	lib().oracle_remove_small_segments(_fptr(d), None if n is None else _fptr(n), None if c is None else _fptr(c),
		d.shape[1], d.shape[0], C.c_float(th), C.c_uint(speckle))
	return d, n, c


def count_asymmetric_edges(depth, th=0.007):
	d = np.ascontiguousarray(depth, np.float32)
	return int(lib().oracle_count_asymmetric_edges(_fptr(d), d.shape[1], d.shape[0], C.c_float(th)))


def gap_interpolation(depth, normal=None, conf=None, th=0.025, gap=7):
	d = np.array(depth, np.float32, copy=True, order="C")
	n = None if normal is None else np.array(normal, np.float32, copy=True, order="C")
	c = None if conf is None else np.array(conf, np.float32, copy=True, order="C")
	lib().oracle_gap_interpolation(_fptr(d), None if n is None else _fptr(n), None if c is None else _fptr(c),
		d.shape[1], d.shape[0], C.c_float(th), C.c_uint(gap))
	return d, n, c


def to_gray(image, bgr=True):
	"""uint8 (H, W, 3|4) -> float32 gray in [0, 1] (toGray with bNormalize)"""
	a = np.ascontiguousarray(image, np.uint8)
	h, w, ch = a.shape
	out = np.zeros((h, w), np.float32)
	lib().oracle_to_gray(_fptr(a), w, h, w*ch, ch, int(bool(bgr)), _fptr(out))
	return out
