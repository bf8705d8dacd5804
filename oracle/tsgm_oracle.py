"""ctypes binding of the CPU oracle of the coarse-to-fine (tSGM) level loop (TEST INFRASTRUCTURE — see tsgm_oracle.h).

tsgm_oracle.cpp is compiled together with the oracle sources it calls (the matcher in sgm_oracle.cpp, the cv::resize
restatements in pm_oracle.cpp) into liboracle_tsgm.so, with the flags of the parity build of oracle/Makefile.  Only tests/ and
scripts/profile_tsgm.py load it; the product package openmvs_b200 never does.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = ("tsgm_oracle.cpp", "sgm_oracle.cpp", "pm_oracle.cpp")
_DEPS = _SRCS + ("tsgm_oracle.h", "oracle.h")
_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall", "-Wno-unused-function", "-pthread", "-shared"]
_LIB = None


def build(force: bool = False) -> str:
	so = os.path.join(_HERE, "liboracle_tsgm.so")
	if force or not os.path.exists(so) or any(os.path.getmtime(os.path.join(_HERE, s)) > os.path.getmtime(so) for s in _DEPS):
		tmp = "%s.tmp.%d" % (so, os.getpid())
		cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
		try:
			subprocess.check_call([cxx] + _FLAGS + ["-o", tmp] + [os.path.join(_HERE, s) for s in _SRCS])
			os.replace(tmp, so)
		finally:
			if os.path.exists(tmp):
				os.unlink(tmp)
	return so


def _lib():
	global _LIB
	if _LIB is None:
		_LIB = C.CDLL(build())
	return _LIB


def _fptr(a):
	return a.ctypes.data_as(C.c_void_p)


def sgm_tsgm_levels(width, height, min_resolution=320):
	"""-> (nLevels, seedWidth, seedHeight)"""
	o = [C.c_int() for _ in range(3)]
	_lib().oracle_sgm_tsgm_levels(int(width), int(height), int(min_resolution), *[C.byref(v) for v in o])
	return tuple(v.value for v in o)


def resize_area_u8(image, factor):
	"""cv::resize(image, Size(), 1/factor, 1/factor, INTER_AREA) of a uint8 (H, W) or (H, W, C) image"""
	a = np.ascontiguousarray(image, np.uint8)
	h, w = a.shape[:2]
	ch = 1 if a.ndim == 2 else a.shape[2]
	dw, dh = int(round(w/factor)), int(round(h/factor))
	out = np.zeros((dh, dw) + a.shape[2:], np.uint8)
	_lib().oracle_resize_area_u8(_fptr(a), w, h, ch, int(factor), _fptr(out))
	return out


def _pixel_records(n):
	return np.zeros(n, dtype=np.dtype([("idx", "<u8"), ("dmin", "<i2"), ("dmax", "<i2"), ("reserved", "<i4")]))


def sgm_range_map(disparity, mask, min_num_disp, min_num_disp_invalid):
	"""Disparity2RangeMap -> (pixels (mh*mw records), numCosts, maxNumDisp)"""
	d = np.ascontiguousarray(disparity, np.int16); m = np.ascontiguousarray(mask, np.uint8)
	px = _pixel_records(m.size)
	mx = C.c_int()
	f = _lib().oracle_sgm_range_map
	f.restype = C.c_uint64
	n = f(_fptr(d), d.shape[1], d.shape[0], _fptr(m), m.shape[1], m.shape[0], int(min_num_disp), int(min_num_disp_invalid), _fptr(px), C.byref(mx))
	return px, int(n), mx.value


def sgm_flip_direction(l2r):
	a = np.ascontiguousarray(l2r, np.int16); out = np.empty_like(a)
	_lib().oracle_sgm_flip_direction(_fptr(a), _fptr(out), a.shape[1], a.shape[0])
	return out


def sgm_extract_mask(disparity, mask, th_valid=3):
	d = np.ascontiguousarray(disparity, np.int16); m = np.array(mask, np.uint8, copy=True, order="C")
	_lib().oracle_sgm_extract_mask(_fptr(d), _fptr(m), d.shape[1], d.shape[0], int(th_valid))
	return m


def sgm_upscale_mask(mask, width2, height2):
	m = np.ascontiguousarray(mask, np.uint8); out = np.zeros((height2, width2), np.uint8)
	_lib().oracle_sgm_upscale_mask(_fptr(m), m.shape[1], m.shape[0], _fptr(out), int(width2), int(height2))
	return out


def filter_speckles(img, new_val=32767, max_speckle_size=100, max_diff=5):
	a = np.array(img, np.int16, copy=True, order="C")
	_lib().oracle_filter_speckles(_fptr(a), a.shape[1], a.shape[0], int(new_val), int(max_speckle_size), int(max_diff))
	return a


def sgm_match_tsgm(left_gray, left_bgr, right_gray, right_bgr, left_mask=None, right_mask=None, seed=None, min_resolution=320,
		speckle_size=100, subpixel_steps=4, P1=3, P2=4, alpha=14.0, beta=38.0, level_costs=False):
	"""the tSGM level loop -> (left disparity x subpixel_steps, cost) over the (w-6) x (h-6) valid region
	(+ the (right, left) cost-volume sizes of every level with level_costs=True)"""
	lg = np.ascontiguousarray(left_gray, np.float32); rg = np.ascontiguousarray(right_gray, np.float32)
	lc = np.ascontiguousarray(left_bgr, np.uint8); rc = np.ascontiguousarray(right_bgr, np.uint8)
	h, w = lg.shape
	keep = [None if m is None else np.ascontiguousarray(m, np.uint8) for m in (left_mask, right_mask)]
	sd = None if seed is None else np.ascontiguousarray(seed, np.int16)
	disp = np.zeros((h-6, w-6), np.int16); cost = np.zeros((h-6, w-6), np.uint16)
	f = _lib().oracle_sgm_match_tsgm
	f.argtypes = [C.c_void_p]*4 + [C.c_int]*2 + [C.c_void_p]*3 + [C.c_int]*5 + [C.c_uint16, C.c_uint16, C.c_float, C.c_float] + [C.c_void_p]*3
	lc_ = np.zeros((16, 2), np.uint64)
	rc_ = f(_fptr(lg), _fptr(lc), _fptr(rg), _fptr(rc), w, h, None if keep[0] is None else _fptr(keep[0]),
		None if keep[1] is None else _fptr(keep[1]), None if sd is None else _fptr(sd), 0 if sd is None else sd.shape[1],
		0 if sd is None else sd.shape[0], int(min_resolution), int(speckle_size), int(subpixel_steps), P1, P2, alpha, beta,
		_fptr(disp), _fptr(cost), _fptr(lc_))
	assert rc_ == 0
	if level_costs:
		return disp, cost, [tuple(int(v) for v in r) for r in lc_[:sgm_tsgm_levels(w, h, min_resolution)[0]]]
	return disp, cost
