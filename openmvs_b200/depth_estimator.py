"""Host-side mirror of the reference interface of the hot path.

Names, argument meaning and error behaviour follow the reference so that the parity tests
read like tests of the reference:

  OPTDENSE            option namespace              libs/MVS/DepthMap.cpp:69-114
  Camera              K, R, C                       libs/MVS/Camera.h
  ViewData, DepthData in/out container              libs/MVS/DepthMap.h:157-271
  PatchMatchB200      the PatchMatchCUDA seam       libs/MVS/PatchMatchCUDA.inl:78-131
                      (ctor(device), Init(bGeomConsistency), Release(), EstimateDepthMap(DepthData&))
  DepthMapsData       EstimateDepthMap(idxImage, nGeometricIter)   libs/MVS/SceneDensify.cpp:616-805
                      FilterDepthMap / RemoveSmallSegments / GapInterpolation   libs/MVS/SceneDensify.cpp:810-1299

Everything here is plumbing above the C-ABI (include/b200mvs.h); the arithmetic runs in the
CUDA kernels of openmvs_b200/csrc.  numpy arrays take the host path (H2D/D2H inside the
call, like the reference seam); torch CUDA tensors take the device-resident path.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import List, Optional

import numpy as np

from . import lib as _lib


class OPTDENSE:
	"""The OPTDENSE knobs the estimator consumes, with the reference defaults
	(libs/MVS/DepthMap.cpp:69-114).  Class attributes, like the reference's globals."""
	nSubResolutionLevels = 2
	nNumViews = 0
	nEstimationIters = 3
	nEstimationGeometricIters = 2
	fEstimationGeometricWeight = 0.1
	nRandomIters = 6
	fNCCThresholdKeep = 0.9
	fDescriptorMinMagnitudeThreshold = 0.02
	fRandomDepthRatio = 0.003
	fRandomAngle1Range = 16.0
	fRandomAngle2Range = 10.0
	fRandomSmoothDepth = 0.02
	fRandomSmoothNormal = 13.0
	fRandomSmoothBonus = 0.93
	# depth-map post-processing (FilterDepthMap / RemoveSmallSegments / GapInterpolation)
	nMinViewsFilter = 2
	nMinViewsFilterAdjust = 1
	bFilterAdjust = True
	fDepthDiffThreshold = 0.01
	nSpeckleSize = 100
	nIpolGapSize = 7
	# engine schedule (not in the reference; include/b200mvs.h b200mvs_params): 0 = automatic number of red-black sweeps
	nSweepsPerIter = 0
	nPropagation = 4
	nPropagationFar = 2
	bSkipUnchanged = 1
	nEvalCap = 0
	nSeed = 1234

	@classmethod
	def schedule(cls, geometric: bool = False):
		"""(red-black sweeps, refinement tries per sweep) the engine runs for the current options (b200mvs_get_schedule)."""
		n, r = C.c_int(), C.c_int()
		p = cls.snapshot()
		_lib.load().b200mvs_get_schedule(C.byref(p), int(bool(geometric)), C.byref(n), C.byref(r))
		return n.value, r.value

	@classmethod
	def snapshot(cls) -> _lib.Params:
		p = _lib.Params()
		for name, _ in _lib.Params._fields_:
			if name == "seed":
				p.seed = cls.nSeed
			else:
				setattr(p, name, getattr(cls, name))
		return p


@dataclasses.dataclass
class Camera:
	K: np.ndarray
	R: np.ndarray
	C: np.ndarray


@dataclasses.dataclass
class ViewData:
	"""DepthData::ViewData: gray float image in [0,1] + camera (+ known depth-map and its camera)."""
	image: object            # (H, W) float32 gray image, or the (H, W, 3|4) uint8 colour image (converted on the device); numpy or torch CUDA
	camera: Camera
	depthMap: object = None  # optional (H, W) float32
	cameraDepthMap: Optional[Camera] = None
	bgr: bool = True         # channel order of a uint8 colour image: B,G,R as cv::imread delivers (False: R,G,B)


@dataclasses.dataclass
class DepthData:
	images: List[ViewData]   # reference view first
	dMin: float
	dMax: float
	depthMap: object = None
	normalMap: object = None
	confMap: object = None
	viewsMap: object = None

	def IsValid(self) -> bool:
		return len(self.images) > 0

	def IsEmpty(self) -> bool:
		return self.depthMap is None

	def Save(self, fileName: str, IDs=None, imageFileName: str = "image.jpg") -> bool:
		"""DepthData::Save (libs/MVS/DepthMap.cpp:237-251): write depth/normal/conf/views as a .dmap file."""
		from . import dmap_io
		tonp = lambda a: None if a is None else (a.detach().cpu().numpy() if _is_torch(a) else np.asarray(a))
		ref = self.images[0]
		h, w = tonp(self.depthMap).shape
		ids = list(IDs) if IDs is not None else list(range(len(self.images)))
		return dmap_io.ExportDepthDataRaw(fileName, imageFileName, ids, (w, h), ref.camera.K, ref.camera.R, ref.camera.C,
			self.dMin, self.dMax, tonp(self.depthMap), tonp(self.normalMap), tonp(self.confMap), tonp(self.viewsMap))

	def Load(self, fileName: str, flags: int = 15) -> bool:
		"""DepthData::Load: read the maps and the depth range back from a .dmap file."""
		from . import dmap_io
		d = dmap_io.ImportDepthDataRaw(fileName, flags)
		self.depthMap, self.normalMap, self.confMap, self.viewsMap = d["depthMap"], d["normalMap"], d["confMap"], d["viewsMap"]
		self.dMin, self.dMax = d["dMin"], d["dMax"]
		return True


def _stream_handle(device) -> int:
	"""cudaStream_t of torch's current stream.  The C-ABI treats NULL as "use the context's own
	stream", so torch's legacy default stream (handle 0) is passed as cudaStreamLegacy (0x1)."""
	import torch
	h = torch.cuda.current_stream(device).cuda_stream
	return h if h else 1


def _is_torch(a) -> bool:
	return type(a).__module__.startswith("torch")


def _mask_size(leftMask, rightMask):
	"""(height, width) shared by the given masks of a pair, (0, 0) without masks"""
	shapes = {tuple(m.shape) for m in (leftMask, rightMask) if m is not None}
	if len(shapes) > 1:
		raise ValueError("left and right masks must have one size")
	return shapes.pop() if shapes else (0, 0)


def _make_views(images: List[ViewData]):
	"""-> (ctypes View array, keepalive list, on_device flag)"""
	n = len(images)
	arr = (_lib.View*n)()
	keep = []
	dev = _is_torch(images[0].image)
	for i, v in enumerate(images):
		o = arr[i]
		if dev != _is_torch(v.image):
			raise ValueError("mixing host and device images in one DepthData")
		if dev:
			img = v.image
			if not img.is_cuda or img.device != images[0].image.device:
				raise ValueError("all views of a DepthData must live on the same CUDA device")
			if img.dtype.__str__() == "torch.uint8":
				# 8-bit colour image: toGray runs on the device inside the call
				if img.dim() != 3 or img.shape[2] not in (3, 4) or img.stride(2) != 1 or img.stride(1) != img.shape[2]:
					raise ValueError("device colour image must be a (H, W, 3|4) uint8 CUDA tensor with packed pixels")
				keep.append(img)
				o.image = None; o.image8 = img.data_ptr(); o.height, o.width, o.channels8 = (int(x) for x in img.shape)
				o.stride8_bytes = img.stride(0); o.bgr8 = int(bool(v.bgr))
			else:
				if img.dtype.__str__() != "torch.float32" or img.dim() != 2 or img.stride(1) != 1:
					raise ValueError("device image must be a 2-D float32 CUDA tensor with unit column stride")
				keep.append(img)
				o.image = img.data_ptr(); o.height, o.width = img.shape; o.stride_bytes = img.stride(0)*4
		else:
			img = np.asarray(v.image)
			if img.dtype == np.uint8:
				if img.ndim != 3 or img.shape[2] not in (3, 4) or img.strides[2] != 1 or img.strides[1] != img.shape[2]:
					raise ValueError("colour image must be a (H, W, 3|4) uint8 array with packed pixels (Image8U3)")
				keep.append(img)
				o.image = None; o.image8 = img.ctypes.data; o.height, o.width, o.channels8 = img.shape
				o.stride8_bytes = img.strides[0]; o.bgr8 = int(bool(v.bgr))
			else:
				if img.dtype != np.float32 or img.ndim != 2 or img.strides[1] != 4:
					raise ValueError("image must be a 2-D float32 array with contiguous rows (Image32F)")
				keep.append(img)
				o.image = img.ctypes.data; o.height, o.width = img.shape; o.stride_bytes = img.strides[0]
		o.K[:] = np.asarray(v.camera.K, np.float64).ravel()
		o.R[:] = np.asarray(v.camera.R, np.float64).ravel()
		o.C[:] = np.asarray(v.camera.C, np.float64).ravel()
		o.depth = None
		if v.depthMap is not None and i > 0:
			cam = v.cameraDepthMap or v.camera
			if dev:
				dm = v.depthMap
				if not _is_torch(dm) or dm.dtype.__str__() != "torch.float32" or not dm.is_cuda or dm.dim() != 2 or dm.stride(1) != 1 or dm.device != images[0].image.device:
					raise ValueError("device depth-map must be a 2-D float32 CUDA tensor with unit column stride on the images' device")
				keep.append(dm)
				o.depth = dm.data_ptr(); o.dheight, o.dwidth = dm.shape; o.dstride_bytes = dm.stride(0)*4
			else:
				dm = np.ascontiguousarray(v.depthMap, np.float32)
				keep.append(dm)
				o.depth = dm.ctypes.data; o.dheight, o.dwidth = dm.shape; o.dstride_bytes = dm.strides[0]
			o.Kd[:] = np.asarray(cam.K, np.float64).ravel()
			o.Rd[:] = np.asarray(cam.R, np.float64).ravel()
			o.Cd[:] = np.asarray(cam.C, np.float64).ravel()
	return arr, keep, dev


class PatchMatchB200:
	"""Drop-in for the reference's `PatchMatchCUDA` (libs/MVS/PatchMatchCUDA.inl:78-131)."""

	def __init__(self, device: int = 0):
		self._lib = _lib.load()
		self._ctx = C.c_void_p()
		rc = self._lib.b200mvs_create(int(device), C.byref(self._ctx))
		if rc != 0:
			raise _lib.B200MVSError("b200mvs_create(device=%d) failed with status %d (no GPU => no fallback)" % (device, rc))
		self.device = int(device)
		self.bGeomConsistency = False
		self.stats = _lib.Stats()

	def Init(self, bGeomConsistency: bool = False):
		"""PatchMatchCUDA::Init: select photometric (false) or geometric-consistency (true) passes."""
		self.bGeomConsistency = bool(bGeomConsistency)

	def Release(self):
		if self._ctx:
			self._lib.b200mvs_destroy(self._ctx)
			self._ctx = C.c_void_p()

	def __del__(self):
		try:
			self.Release()
		except Exception:
			pass

	def ToGray(self, image, bgr: bool = True):
		"""TImage::toGray(out, COLOR_BGR2GRAY, bNormalize=true) (libs/Common/Types.inl:2377-2431) on the device: uint8 CUDA tensor
		(H, W, 3|4), channel order B,G,R(,A) as cv::imread delivers (bgr=False: R,G,B) -> float32 gray (H, W) in [0, 1]."""
		import torch
		if not (_is_torch(image) and image.is_cuda and image.dtype == torch.uint8 and image.dim() == 3 and image.shape[2] in (3, 4) and image.is_contiguous()):
			raise ValueError("ToGray needs a contiguous uint8 CUDA tensor of shape (H, W, 3|4)")
		h, w, ch = (int(v) for v in image.shape)
		out = torch.empty((h, w), dtype=torch.float32, device=image.device)
		rc = self._lib.b200mvs_to_gray_device(self._ctx, image.data_ptr(), w, h, w*ch, ch, int(bool(bgr)), out.data_ptr(), w*4,
			C.c_void_p(_stream_handle(image.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_to_gray_device")
		return out

	def ScaleImage(self, image, scale: float):
		"""DepthData::ViewData::ScaleImage (libs/MVS/DepthMap.h:193-203) on the device: float32 CUDA tensor (H, W) ->
		cv::resize(image, Size(), scale, scale, scale > 1 ? INTER_CUBIC : INTER_AREA), or None when |scale - 1| < 0.15
		(the reference keeps the image then)."""
		import torch
		if not (_is_torch(image) and image.is_cuda and image.dtype == torch.float32 and image.dim() == 2 and image.stride(1) == 1):
			raise ValueError("ScaleImage needs a 2-D float32 CUDA tensor with unit column stride")
		h, w = (int(v) for v in image.shape)
		dw, dh, ok = C.c_int(), C.c_int(), C.c_int()
		self._lib.b200mvs_scaled_size(w, h, C.c_float(scale), C.byref(dw), C.byref(dh))
		out = torch.empty((max(dh.value, 1), max(dw.value, 1)), dtype=torch.float32, device=image.device)
		rc = self._lib.b200mvs_scale_image_device(self._ctx, image.data_ptr(), w, h, image.stride(0)*4, C.c_float(scale), out.data_ptr(),
			C.byref(ok), C.c_void_p(_stream_handle(image.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_scale_image_device")
		return out if ok.value else None

	def _set_params(self):
		p = OPTDENSE.snapshot()
		_lib.check(self._lib, self._ctx, self._lib.b200mvs_set_params(self._ctx, C.byref(p)), "b200mvs_set_params")

	def SetDebug(self, **kw):
		"""b200mvs_set_debug: diagnostic kernel switches (the fields of b200mvs_debug: scalarTaps, noTMA, sweepFourCtas, ...);
		no arguments = defaults."""
		d = _lib.Debug()
		for k, v in kw.items():
			if k == "reserved" or not hasattr(d, k):
				raise AttributeError(k)
			setattr(d, k, int(v))
		_lib.check(self._lib, self._ctx, self._lib.b200mvs_set_debug(self._ctx, C.byref(d)), "b200mvs_set_debug")

	def SetIgnoreMask(self, mask=None):
		"""Ignore-mask of the reference view for the following EstimateDepthMap calls (OPTDENSE::nIgnoreMaskLabel >= 0,
		libs/MVS/DepthMap.cpp:215-230,300-323): (H, W) uint8, 0 = ignored; numpy array (copied) or torch CUDA tensor
		(kept by reference until cleared); None clears it."""
		self._mask_keep = None
		if mask is None:
			rc = self._lib.b200mvs_set_ignore_mask(self._ctx, None, 0, 0, 0, 0)
		elif _is_torch(mask):
			import torch
			if mask.dtype != torch.uint8 or not mask.is_cuda or mask.dim() != 2 or mask.stride(1) != 1:
				raise ValueError("device mask must be a 2-D uint8 CUDA tensor with unit column stride")
			self._mask_keep = mask
			rc = self._lib.b200mvs_set_ignore_mask(self._ctx, mask.data_ptr(), int(mask.shape[1]), int(mask.shape[0]), int(mask.stride(0)), 1)
		else:
			m = np.ascontiguousarray(mask, np.uint8)
			if m.ndim != 2:
				raise ValueError("mask must be 2-D")
			rc = self._lib.b200mvs_set_ignore_mask(self._ctx, m.ctypes.data, m.shape[1], m.shape[0], m.strides[0], 0)
		_lib.check(self._lib, self._ctx, rc, "b200mvs_set_ignore_mask")

	def EstimateDepthMap(self, depthData: DepthData, nGeometricIter: Optional[int] = None, stream=None, sync: bool = True):
		"""PatchMatchCUDA::EstimateDepthMap(DepthData&): estimate depthMap/normalMap/confMap/viewsMap
		of depthData in place.  nGeometricIter defaults to -1 (photometric) or 0 (after Init(true))."""
		if not depthData.IsValid() or len(depthData.images) < 2:
			raise ValueError("DepthData needs the reference view and at least one neighbour")
		if nGeometricIter is None:
			nGeometricIter = 0 if self.bGeomConsistency else -1
		self._set_params()
		arr, keep, dev = _make_views(depthData.images)
		h, w = depthData.images[0].image.shape[:2]
		if dev:
			import torch
			t0 = depthData.images[0].image
			def dmap(a, shape, dtype):
				if a is None:
					return torch.zeros(shape, dtype=dtype, device=t0.device)
				if not _is_torch(a) or tuple(a.shape) != tuple(shape) or not a.is_contiguous() or a.dtype != dtype or a.device != t0.device:
					raise ValueError("map must be a contiguous %s CUDA tensor of shape %s on the images' device" % (dtype, tuple(shape)))
				return a
			depthData.depthMap = dmap(depthData.depthMap, (h, w), torch.float32)
			depthData.normalMap = dmap(depthData.normalMap, (h, w, 3), torch.float32)
			depthData.confMap = dmap(depthData.confMap, (h, w), torch.float32)
			depthData.viewsMap = dmap(depthData.viewsMap, (h, w, 4), torch.uint8)
			if stream is None:
				stream = _stream_handle(t0.device)
			rc = self._lib.b200mvs_estimate_device(self._ctx, arr, len(arr), C.c_float(depthData.dMin), C.c_float(depthData.dMax),
				int(nGeometricIter), depthData.depthMap.data_ptr(), depthData.normalMap.data_ptr(),
				depthData.confMap.data_ptr(), depthData.viewsMap.data_ptr(), C.c_void_p(stream),
				C.byref(self.stats) if sync else None)
			_lib.check(self._lib, self._ctx, rc, "b200mvs_estimate_device")
		else:
			def hmap(a, shape, dtype):
				if a is None:
					return np.zeros(shape, dtype)
				a = np.ascontiguousarray(a, dtype)
				if a.shape != tuple(shape):
					raise ValueError("map has the wrong shape")
				return a
			depthData.depthMap = hmap(depthData.depthMap, (h, w), np.float32)
			depthData.normalMap = hmap(depthData.normalMap, (h, w, 3), np.float32)
			depthData.confMap = hmap(depthData.confMap, (h, w), np.float32)
			depthData.viewsMap = hmap(depthData.viewsMap, (h, w, 4), np.uint8)
			if sync:
				rc = self._lib.b200mvs_estimate(self._ctx, arr, len(arr), C.c_float(depthData.dMin), C.c_float(depthData.dMax),
					int(nGeometricIter), depthData.depthMap.ctypes.data, depthData.normalMap.ctypes.data,
					depthData.confMap.ctypes.data, depthData.viewsMap.ctypes.data, C.byref(self.stats))
				_lib.check(self._lib, self._ctx, rc, "b200mvs_estimate")
			else:
				# asynchronous host path: the caller keeps depthData alive and calls Wait() before reading the maps
				rc = self._lib.b200mvs_estimate_async(self._ctx, arr, len(arr), C.c_float(depthData.dMin), C.c_float(depthData.dMax),
					int(nGeometricIter), depthData.depthMap.ctypes.data, depthData.normalMap.ctypes.data,
					depthData.confMap.ctypes.data, depthData.viewsMap.ctypes.data)
				_lib.check(self._lib, self._ctx, rc, "b200mvs_estimate_async")
				self._inflight = (depthData, keep)
		return depthData

	def Wait(self):
		"""b200mvs_sync: wait for an EstimateDepthMap(..., sync=False) on host buffers and fetch its stats."""
		rc = self._lib.b200mvs_sync(self._ctx, C.byref(self.stats))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sync")
		self._inflight = None

	# ---- building blocks on device tensors (used by the parity tests) -----------------------
	def _dev_views(self, images):
		arr, keep, dev = _make_views(images)
		if not dev:
			raise ValueError("building blocks need device-resident views")
		return arr, keep

	def ScoreDepthMap(self, images, dMin, dMax, plane4, cost, lowres=None):
		"""pass A (ScoreDepthMapTmp) on a packed plane field (H, W, 4) = {nx,ny,nz,depth}."""
		import torch
		self._set_params()
		arr, keep = self._dev_views(images)
		s = _stream_handle(plane4.device)
		rc = self._lib.b200mvs_pm_score(self._ctx, arr, len(arr), C.c_float(dMin), C.c_float(dMax),
			lowres.data_ptr() if lowres is not None else None, plane4.data_ptr(), cost.data_ptr(), C.c_void_p(s))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_pm_score")

	def SweepDepthMap(self, images, dMin, dMax, plane4, cost, sweep, half=-1, nRandomIters=None, lowres=None):
		"""pass B: one red-black sweep (both colours, or one if half in {0,1})."""
		import torch
		self._set_params()
		arr, keep = self._dev_views(images)
		if nRandomIters is None:
			nRandomIters = OPTDENSE.schedule()[1]
		s = _stream_handle(plane4.device)
		rc = self._lib.b200mvs_pm_sweep(self._ctx, arr, len(arr), C.c_float(dMin), C.c_float(dMax),
			lowres.data_ptr() if lowres is not None else None, int(sweep), int(half), int(nRandomIters),
			plane4.data_ptr(), cost.data_ptr(), C.c_void_p(s))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_pm_sweep")


def EstimateDepthMapsBatch(arrDepthData: List[DepthData], engines: List["PatchMatchB200"], nGeometricIter: int = -1):
	"""b200mvs_estimate_batch: estimate every DepthData (host buffers) with the given engines — one per GPU of
	the box, or two on one GPU — dealt round-robin inside this process."""
	lib = engines[0]._lib
	for e in engines:
		e._set_params()
	jobs = (_lib.Job*len(arrDepthData))()
	keep = []
	for j, dd in enumerate(arrDepthData):
		arr, k, dev = _make_views(dd.images)
		if dev:
			raise ValueError("the batch call takes host buffers")
		h, w = dd.images[0].image.shape[:2]
		dd.depthMap = np.zeros((h, w), np.float32) if dd.depthMap is None else np.ascontiguousarray(dd.depthMap, np.float32)
		dd.normalMap = np.zeros((h, w, 3), np.float32) if dd.normalMap is None else np.ascontiguousarray(dd.normalMap, np.float32)
		dd.confMap = np.zeros((h, w), np.float32); dd.viewsMap = np.zeros((h, w, 4), np.uint8)
		keep.append((arr, k))
		J = jobs[j]
		J.views = arr; J.nViews = len(arr); J.dMin = dd.dMin; J.dMax = dd.dMax; J.nGeometricIter = int(nGeometricIter)
		J.depth = dd.depthMap.ctypes.data; J.normal = dd.normalMap.ctypes.data; J.conf = dd.confMap.ctypes.data; J.viewsMap = dd.viewsMap.ctypes.data
	ctxs = (C.c_void_p*len(engines))(*[e._ctx for e in engines])
	rc = lib.b200mvs_estimate_batch(ctxs, len(engines), jobs, len(arrDepthData))
	if rc != 0:
		bad = [j for j in range(len(arrDepthData)) if jobs[j].status]
		raise _lib.B200MVSError("b200mvs_estimate_batch: jobs %s failed with status %d" % (bad, rc))
	return arrDepthData


class DepthMapsData:
	"""The slice of the reference's DepthMapsData around the hot path (libs/MVS/SceneDensify.h:52-93):
	arrDepthData + EstimateDepthMap(idxImage, nGeometricIter), and the per-view post-processing that
	follows it: RemoveSmallSegments, GapInterpolation, FilterDepthMap (SceneDensify.cpp:810-1299)."""

	def __init__(self, arrDepthData: List[DepthData], device: int = 0, nCalibratedImages: Optional[int] = None):
		self.arrDepthData = arrDepthData
		self.pmCUDA = PatchMatchB200(device)
		self.nCalibratedImages = len(arrDepthData) if nCalibratedImages is None else int(nCalibratedImages)
		self.stats = _lib.Stats()

	def EstimateDepthMap(self, idxImage: int, nGeometricIter: int = -1) -> bool:
		self.pmCUDA.Init(nGeometricIter >= 0)
		self.pmCUDA.EstimateDepthMap(self.arrDepthData[idxImage], nGeometricIter)
		return True

	@staticmethod
	def _ptr(a):
		return a.data_ptr() if _is_torch(a) else a.ctypes.data

	@staticmethod
	def _dmap(o: "_lib.DMap", depthData: DepthData, need_conf: bool, keep: list):
		cam = depthData.images[0].camera
		d, c = depthData.depthMap, depthData.confMap
		if not _is_torch(d):
			d = np.ascontiguousarray(d, np.float32)
			c = None if c is None else np.ascontiguousarray(c, np.float32)
		elif not d.is_contiguous() or (c is not None and not c.is_contiguous()):
			raise ValueError("depth/confidence maps must be contiguous")
		if need_conf and c is None:
			raise ValueError("FilterDepthMap needs the confidence map of every view")
		keep += [d, c]
		o.depth = DepthMapsData._ptr(d); o.conf = DepthMapsData._ptr(c) if c is not None else None
		o.height, o.width = int(d.shape[0]), int(d.shape[1])
		o.K[:] = np.asarray(cam.K, np.float64).ravel(); o.R[:] = np.asarray(cam.R, np.float64).ravel(); o.C[:] = np.asarray(cam.C, np.float64).ravel()
		return d

	def FilterDepthMap(self, depthDataRef: DepthData, neighbors: List[DepthData], bAdjust: Optional[bool] = None, projected: bool = False):
		"""DepthMapsData::FilterDepthMap(depthDataRef, idxNeighbors, bAdjust) (SceneDensify.cpp:1050-1299).
		`neighbors` are the DepthData of the (at most 8, SceneDensify.cpp:2152) neighbour views whose depth-maps are valid.
		Returns (newDepthMap, newConfMap) — what the reference saves as filtered.dmap / filtered.cmap — or None when the map
		can not be filtered; with projected=True also the N projected neighbour depth and confidence maps (device path)."""
		lib, ctx = self.pmCUDA._lib, self.pmCUDA._ctx
		bAdjust = OPTDENSE.bFilterAdjust if bAdjust is None else bool(bAdjust)
		prm = _lib.FilterParams(min(OPTDENSE.nMinViewsFilter, self.nCalibratedImages-1),
			min(OPTDENSE.nMinViewsFilterAdjust, self.nCalibratedImages-1), OPTDENSE.fDepthDiffThreshold, int(bAdjust))
		arr = (_lib.DMap*(len(neighbors)+1))()
		keep: list = []
		dref = self._dmap(arr[0], depthDataRef, True, keep)
		for i, nb in enumerate(neighbors):
			self._dmap(arr[i+1], nb, bAdjust, keep)
		nbrs = C.cast(C.byref(arr, C.sizeof(_lib.DMap)), C.POINTER(_lib.DMap))
		ok = C.c_int(0)
		if _is_torch(dref):
			import torch
			od = torch.empty_like(dref); oc = torch.empty_like(dref)
			pd = pc = None
			if projected:
				pd = torch.empty((max(len(neighbors), 1),)+tuple(dref.shape), dtype=torch.float32, device=dref.device)
				pc = torch.zeros_like(pd)
			rc = lib.b200mvs_filter_depth_map_device(ctx, C.byref(arr[0]), nbrs, len(neighbors), C.byref(prm), depthDataRef.dMin, depthDataRef.dMax,
				od.data_ptr(), oc.data_ptr(), pd.data_ptr() if projected else None, pc.data_ptr() if projected and bAdjust else None,
				C.byref(ok), C.c_void_p(_stream_handle(dref.device)))
			_lib.check(lib, ctx, rc, "b200mvs_filter_depth_map_device")
			if not ok.value:
				return None
			return (od, oc, pd, pc) if projected else (od, oc)
		od = np.empty_like(dref); oc = np.empty_like(dref)
		rc = lib.b200mvs_filter_depth_map(ctx, C.byref(arr[0]), nbrs, len(neighbors), C.byref(prm), depthDataRef.dMin, depthDataRef.dMax,
			od.ctypes.data, oc.ctypes.data, C.byref(ok), C.byref(self.stats))
		_lib.check(lib, ctx, rc, "b200mvs_filter_depth_map")
		return (od, oc) if ok.value else None

	def _post(self, name: str, depthData: DepthData, arg: int) -> bool:
		lib, ctx = self.pmCUDA._lib, self.pmCUDA._ctx
		d, n, c = depthData.depthMap, depthData.normalMap, depthData.confMap
		h, w = int(d.shape[0]), int(d.shape[1])
		if _is_torch(d):
			for a in (d, n, c):
				if a is not None and not a.is_contiguous():
					raise ValueError("maps must be contiguous")
			rc = getattr(lib, name+"_device")(ctx, d.data_ptr(), n.data_ptr() if n is not None else None, c.data_ptr() if c is not None else None,
				w, h, OPTDENSE.fDepthDiffThreshold, int(arg), C.c_void_p(_stream_handle(d.device)))
		else:
			for a in (d, n, c):
				if a is not None and not (a.flags.c_contiguous and a.dtype == np.float32):
					raise ValueError("maps must be contiguous float32 arrays (processed in place)")
			rc = getattr(lib, name)(ctx, d.ctypes.data, n.ctypes.data if n is not None else None, c.ctypes.data if c is not None else None,
				w, h, OPTDENSE.fDepthDiffThreshold, int(arg), C.byref(self.stats))
		_lib.check(lib, ctx, rc, name)
		return True

	def RemoveSmallSegments(self, depthData: DepthData) -> bool:
		"""DepthMapsData::RemoveSmallSegments (SceneDensify.cpp:810-900), depthData's maps in place."""
		return self._post("b200mvs_remove_small_segments", depthData, OPTDENSE.nSpeckleSize)

	def GapInterpolation(self, depthData: DepthData) -> bool:
		"""DepthMapsData::GapInterpolation (SceneDensify.cpp:904-1045), depthData's maps in place."""
		return self._post("b200mvs_gap_interpolation", depthData, OPTDENSE.nIpolGapSize)


class SemiGlobalMatcher:
	"""The pair matcher of the reference's STEREO::SemiGlobalMatcher
	(libs/MVS/SemiGlobalMatcher.h:61-203): Match(left, right) -> (disparityMap, costMap) over the
	valid region, with the ctor parameters P1, P2, P2alpha, P2beta (defaults 3, 4, 14, 38)."""
	NO_DISP = 32767
	NO_ACCUMCOST = 65535

	def __init__(self, P1: int = 3, P2: int = 4, P2alpha: float = 14.0, P2beta: float = 38.0, device: int = 0):
		self._lib = _lib.load()
		self._ctx = C.c_void_p()
		rc = self._lib.b200mvs_create(int(device), C.byref(self._ctx))
		if rc != 0:
			raise _lib.B200MVSError("b200mvs_create(device=%d) failed with status %d (no GPU => no fallback)" % (device, rc))
		self.prm = _lib.SgmParams(int(P1), int(P2), float(P2alpha), float(P2beta))
		self.stats = _lib.Stats()

	def Release(self):
		if getattr(self, "_peer", None) is not None:
			self._peer.Release(); self._peer = None
		if self._ctx:
			self._lib.b200mvs_destroy(self._ctx)
			self._ctx = C.c_void_p()

	def __del__(self):
		try:
			self.Release()
		except Exception:
			pass

	def SetDebug(self, **kw):
		"""b200mvs_set_debug: sgmAggregation (0 auto, 1 general, 2 register-pipelined uniform, 3 bulk-copy ring, 4 wave fronts),
		sgmCost, frontLayout / frontSerial / frontBlock / frontLag / frontCtas / frontDepth (b200mvs_debug); no arguments = defaults."""
		d = _lib.Debug()
		for k, v in kw.items():
			if k == "reserved" or not hasattr(d, k):
				raise AttributeError(k)
			setattr(d, k, int(v))
		_lib.check(self._lib, self._ctx, self._lib.b200mvs_set_debug(self._ctx, C.byref(d)), "b200mvs_set_debug")

	def Match(self, leftGray, leftColor, rightGray, imagePixels, numCosts: int):
		"""Host path: numpy images (gray float32 HxW, colour uint8 HxWx3 BGR) and the PixelMap
		(structured array from synth.sgm_pixel_map or any {u8 idx, i2 dmin, i2 dmax, i4} records)."""
		lg = np.ascontiguousarray(leftGray, np.float32); rg = np.ascontiguousarray(rightGray, np.float32)
		lc = np.ascontiguousarray(leftColor, np.uint8)
		h, w = lg.shape
		if rg.shape != (h, w) or lc.shape != (h, w, 3):
			raise ValueError("left/right/colour images must share one size")
		px = np.ascontiguousarray(imagePixels)
		if px.itemsize != 16 or px.size != (w-6)*(h-6):
			raise ValueError("PixelMap must hold (w-6)*(h-6) 16-byte records")
		disp = np.zeros((h-6, w-6), np.int16); cost = np.zeros((h-6, w-6), np.uint16)
		rc = self._lib.b200mvs_sgm_match(self._ctx, lg.ctypes.data, lc.ctypes.data, rg.ctypes.data, w, h, px.ctypes.data,
			C.c_uint64(numCosts), C.byref(self.prm), disp.ctypes.data, cost.ctypes.data, C.byref(self.stats))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_match")
		return disp, cost

	def MatchDevice(self, leftGray, leftColor, rightGray, imagePixels, numCosts: int, stages: int = 7, costs=None, accums=None, sync: bool = True):
		"""Device-resident path on torch CUDA tensors; costs (uint8) / accums (uint16 viewed as int16)
		are optional in/out volumes of numCosts entries.  Returns (disparity, cost) int16 tensors
		(cost holds the uint16 bit pattern)."""
		import torch
		h, w = leftGray.shape
		dev = leftGray.device
		disp = torch.zeros((h-6, w-6), dtype=torch.int16, device=dev)
		cost = torch.zeros((h-6, w-6), dtype=torch.int16, device=dev)
		s = _stream_handle(dev)
		rc = self._lib.b200mvs_sgm_match_device(self._ctx, leftGray.data_ptr(), leftColor.data_ptr(), rightGray.data_ptr(), w, h,
			imagePixels.data_ptr(), C.c_uint64(numCosts), C.byref(self.prm), int(stages),
			costs.data_ptr() if costs is not None else None, accums.data_ptr() if accums is not None else None,
			disp.data_ptr(), cost.data_ptr(), C.c_void_p(s), C.byref(self.stats) if sync else None)
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_match_device")
		return disp, cost

	def ConsistencyCrossCheck(self, l2r, r2l, thCross: int = 1):
		"""SemiGlobalMatcher::ConsistencyCrossCheck on int16 CUDA tensors; l2r is modified in place."""
		h, w = l2r.shape
		rc = self._lib.b200mvs_sgm_cross_check_device(self._ctx, l2r.data_ptr(), r2l.data_ptr(), w, h, int(thCross), C.c_void_p(_stream_handle(l2r.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_cross_check_device")
		return l2r

	def RefineDisparityMap(self, disparityMap, imagePixels, accums=None, subpixelSteps: int = 4):
		"""SemiGlobalMatcher::RefineDisparityMap (LC-blend) on CUDA tensors; disparityMap in place."""
		rc = self._lib.b200mvs_sgm_refine_device(self._ctx, imagePixels.data_ptr(), accums.data_ptr() if accums is not None else None,
			disparityMap.data_ptr(), disparityMap.numel(), int(subpixelSteps), C.c_void_p(_stream_handle(disparityMap.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_refine_device")
		return disparityMap

	def MatchPairDevice(self, leftGray, leftColor, rightGray, rightColor, minDisp: int, maxDisp: int, thCross: int = 1, subpixelSteps: int = 4,
			overlap: bool = True):
		"""The per-level body of SemiGlobalMatcher::Match(scene, ...) for one global range (non-tSGM branch,
		libs/MVS/SemiGlobalMatcher.cpp:643-725) on CUDA tensors: right->left match with the range [minDisp, maxDisp),
		left->right match with the mirrored range, cross-check of the left map, sub-pixel refinement.
		Returns (leftDisparity * subpixelSteps, rightDisparity) as int16 tensors (NO_DISP = 32767).
		overlap (default): the two matches run on two contexts / streams (they are independent until the cross-check), so the
		aggregation kernels of the two share the SMs: 7.98 ms instead of 9.11 ms per 1080p pair at D = 128 (profiles/sgm_pair_r02.txt)."""
		import torch
		h, w = leftGray.shape
		nv = (w-6)*(h-6)
		num = int(maxDisp-minDisp)
		dev = leftGray.device
		def pixel_map(lo, hi):
			# PixelData{u64 idx; i16 dmin, dmax; i32 pad} of a dense volume with one range, built on the device and kept: 16 B per
			# pixel would otherwise be generated and uploaded for every pair (33 MB at 1080p)
			key = (nv, num, int(lo), int(hi), str(dev))
			cache = self.__dict__.setdefault("_pxmaps", {})
			if key not in cache:
				if len(cache) > 8:
					cache.clear()
				rec = torch.empty((nv, 2), dtype=torch.int64, device=dev)
				rec[:, 0] = torch.arange(nv, dtype=torch.int64, device=dev)*num
				rec[:, 1] = (int(lo) & 0xFFFF) | ((int(hi) & 0xFFFF) << 16)       # little endian: dmin, dmax, pad = 0
				cache[key] = rec.view(torch.uint8).reshape(nv, 16)
			return cache[key]
		# Match(rightDataLevel, leftDataLevel): the right image plays "left" with range [minDisp, maxDisp)
		pxr = pixel_map(minDisp, maxDisp)
		# ranges are mirrored for the left->right match (SemiGlobalMatcher.cpp:677-682)
		pxl = pixel_map(-maxDisp, -minDisp)
		if not overlap:
			rdisp, _ = self.MatchDevice(rightGray, rightColor, leftGray, pxr, nv*num)
			ldisp, _ = self.MatchDevice(leftGray, leftColor, rightGray, pxl, nv*num)
		else:
			if getattr(self, "_peer", None) is None:
				self._peer = SemiGlobalMatcher(device=dev.index or 0)
				self._peer.prm = self.prm
				self._side = torch.cuda.Stream(device=dev)
			main = torch.cuda.current_stream(dev)
			self._side.wait_stream(main)
			with torch.cuda.stream(self._side):
				rdisp, _ = self._peer.MatchDevice(rightGray, rightColor, leftGray, pxr, nv*num, sync=False)
				for t in (rightGray, rightColor, leftGray, pxr, rdisp):
					t.record_stream(self._side)
			ldisp, _ = self.MatchDevice(leftGray, leftColor, rightGray, pxl, nv*num, sync=False)
			main.wait_stream(self._side)
		self.ConsistencyCrossCheck(ldisp, rdisp, thCross)
		self.RefineDisparityMap(ldisp, pxl, None, subpixelSteps)  # accumulated costs of the last (left) match
		torch.cuda.current_stream(dev).synchronize()
		return ldisp, rdisp

	# ---- coarse-to-fine (tSGM) matching, the reference's default SGM path ----
	@staticmethod
	def TsgmLevels(width: int, height: int, minResolution: int = 320):
		"""-> (number of levels, seed width, seed height) of the coarse-to-fine loop (b200mvs_sgm_tsgm_levels)."""
		lib = _lib.load()
		o = [C.c_int() for _ in range(3)]
		rc = lib.b200mvs_sgm_tsgm_levels(int(width), int(height), int(minResolution), *[C.byref(v) for v in o])
		if rc != 0:
			raise _lib.B200MVSError("b200mvs_sgm_tsgm_levels(%d, %d, %d) failed with status %d" % (width, height, minResolution, rc))
		return tuple(v.value for v in o)

	def MatchPyramidDevice(self, leftGray, leftColor, rightGray, rightColor, leftMask=None, rightMask=None, seed=None,
			minResolution: int = 320, nSpeckleSize: int = 100, subpixelSteps: int = 4, sync: bool = True):
		"""The level loop of SemiGlobalMatcher::Match(scene, ...) (libs/MVS/SemiGlobalMatcher.cpp:584-718) for one rectified pair on
		CUDA tensors: gray float32 (H, W), colour uint8 (H, W, 3) BGR, masks uint8 (H, W) 0 = invalid (None = all valid), seed int16
		of the size TsgmLevels gives (32767 = unknown; None = all unknown).  Returns (leftDisparity * subpixelSteps, cost) over the
		(H-6, W-6) valid region as int16 tensors (NO_DISP = 32767; cost holds the uint16 bit pattern)."""
		import torch
		h, w = leftGray.shape
		dev = leftGray.device
		disp = torch.empty((h-6, w-6), dtype=torch.int16, device=dev)
		cost = torch.empty((h-6, w-6), dtype=torch.int16, device=dev)
		mh, mw = _mask_size(leftMask, rightMask)
		sh, sw = seed.shape if seed is not None else (0, 0)
		ptr = lambda t: t.data_ptr() if t is not None else None
		rc = self._lib.b200mvs_sgm_match_tsgm_device(self._ctx, leftGray.data_ptr(), leftColor.data_ptr(), rightGray.data_ptr(),
			rightColor.data_ptr(), w, h, ptr(leftMask), ptr(rightMask), mw, mh, ptr(seed), sw, sh, int(minResolution),
			int(nSpeckleSize), int(subpixelSteps), C.byref(self.prm), disp.data_ptr(), cost.data_ptr(),
			C.c_void_p(_stream_handle(dev)), C.byref(self.stats) if sync else None)
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_match_tsgm_device")
		return disp, cost

	def MatchPyramid(self, leftGray, leftColor, rightGray, rightColor, leftMask=None, rightMask=None, seed=None,
			minResolution: int = 320, nSpeckleSize: int = 100, subpixelSteps: int = 4):
		"""Host form of MatchPyramidDevice on numpy arrays -> (leftDisparity * subpixelSteps int16, cost uint16)."""
		lg = np.ascontiguousarray(leftGray, np.float32); rg = np.ascontiguousarray(rightGray, np.float32)
		lc = np.ascontiguousarray(leftColor, np.uint8); rcol = np.ascontiguousarray(rightColor, np.uint8)
		h, w = lg.shape
		lm = None if leftMask is None else np.ascontiguousarray(leftMask, np.uint8)
		rm = None if rightMask is None else np.ascontiguousarray(rightMask, np.uint8)
		sd = None if seed is None else np.ascontiguousarray(seed, np.int16)
		mh, mw = _mask_size(lm, rm)
		sh, sw = sd.shape if sd is not None else (0, 0)
		disp = np.zeros((h-6, w-6), np.int16); cost = np.zeros((h-6, w-6), np.uint16)
		ptr = lambda a: a.ctypes.data if a is not None else None
		rc = self._lib.b200mvs_sgm_match_tsgm(self._ctx, lg.ctypes.data, lc.ctypes.data, rg.ctypes.data, rcol.ctypes.data, w, h,
			ptr(lm), ptr(rm), mw, mh, ptr(sd), sw, sh, int(minResolution), int(nSpeckleSize), int(subpixelSteps), C.byref(self.prm),
			disp.ctypes.data, cost.ctypes.data, C.byref(self.stats))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_match_tsgm")
		return disp, cost

	def Disparity2RangeMap(self, disparityMap, maskMap, minNumDisp: int, minNumDispInvalid: int):
		"""SemiGlobalMatcher::Disparity2RangeMap on CUDA tensors (int16 coarse map, uint8 fine mask) ->
		(PixelMap as (n, 16) uint8 records, numCosts, maxNumDisp).  Synchronises the stream."""
		import torch
		h, w = disparityMap.shape
		mh, mw = maskMap.shape
		px = torch.empty((mh*mw, 16), dtype=torch.uint8, device=disparityMap.device)
		nc = C.c_uint64(); mx = C.c_int()
		rc = self._lib.b200mvs_sgm_range_map_device(self._ctx, disparityMap.data_ptr(), w, h, maskMap.data_ptr(), mw, mh, int(minNumDisp),
			int(minNumDispInvalid), px.data_ptr(), C.byref(nc), C.byref(mx), C.c_void_p(_stream_handle(disparityMap.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_range_map_device")
		return px, int(nc.value), int(mx.value)

	def FlipDirection(self, l2r):
		"""SemiGlobalMatcher::FlipDirection: int16 CUDA tensor -> the right-to-left map."""
		import torch
		h, w = l2r.shape
		r2l = torch.empty_like(l2r)
		rc = self._lib.b200mvs_sgm_flip_direction_device(self._ctx, l2r.data_ptr(), r2l.data_ptr(), w, h, C.c_void_p(_stream_handle(l2r.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_flip_direction_device")
		return r2l

	def FilterSpeckles(self, disparityMap, newVal: int = NO_DISP, maxSpeckleSize: int = 100, maxDiff: int = 5):
		"""cv::filterSpeckles on an int16 CUDA tensor, in place."""
		h, w = disparityMap.shape
		rc = self._lib.b200mvs_sgm_filter_speckles_device(self._ctx, disparityMap.data_ptr(), w, h, int(newVal), int(maxSpeckleSize), int(maxDiff),
			C.c_void_p(_stream_handle(disparityMap.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_filter_speckles_device")
		return disparityMap

	def ExtractMask(self, disparityMap, maskMap, thValid: int = 3):
		"""SemiGlobalMatcher::ExtractMask on CUDA tensors; maskMap (uint8) in place."""
		h, w = disparityMap.shape
		rc = self._lib.b200mvs_sgm_extract_mask_device(self._ctx, disparityMap.data_ptr(), maskMap.data_ptr(), w, h, int(thValid),
			C.c_void_p(_stream_handle(disparityMap.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_extract_mask_device")
		return maskMap

	def UpscaleMask(self, maskMap, width2: int, height2: int):
		"""SemiGlobalMatcher::UpscaleMask: uint8 CUDA tensor -> mask of (height2, width2)."""
		import torch
		h, w = maskMap.shape
		out = torch.empty((height2, width2), dtype=torch.uint8, device=maskMap.device)
		rc = self._lib.b200mvs_sgm_upscale_mask_device(self._ctx, maskMap.data_ptr(), w, h, out.data_ptr(), int(width2), int(height2),
			C.c_void_p(_stream_handle(maskMap.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_sgm_upscale_mask_device")
		return out

	def ResizeAreaBGR8(self, image, factor: int):
		"""cv::resize(image, Size(), 1/factor, 1/factor, INTER_AREA) of a uint8 (H, W, 3) CUDA tensor, integer factor."""
		import torch
		h, w = image.shape[:2]
		out = torch.empty((int(round(h/factor)), int(round(w/factor)), 3), dtype=torch.uint8, device=image.device)
		rc = self._lib.b200mvs_resize_area_bgr8_device(self._ctx, image.data_ptr(), w, h, int(factor), out.data_ptr(),
			C.c_void_p(_stream_handle(image.device)))
		_lib.check(self._lib, self._ctx, rc, "b200mvs_resize_area_bgr8_device")
		return out


@dataclasses.dataclass
class PointCloud:
	"""MVS::PointCloud as FuseDepthMaps fills it: points, pointViews, pointWeights, colors, normals."""
	points: np.ndarray            # (n, 3) float32
	pointViews: list              # per point: ascending image IDs (np.uint32 arrays)
	pointWeights: list            # per point: float32 weights, parallel to pointViews
	colors: object = None         # (n, 3) uint8
	normals: object = None        # (n, 3) float32
	projs: list = None            # per point: (k, 2) uint16 pixel coordinates of its views
	nDepths: int = 0


def FuseDepthMaps(views, nMinViewsFuse: int = 2, fDepthDiffThreshold: float = 0.01, fNormalDiffThreshold: float = 25.0,
		bEstimateColor: bool = True, bEstimateNormal: bool = True) -> PointCloud:
	"""DepthMapsData::FuseDepthMaps (libs/MVS/SceneDensify.cpp:1372-1646) through b200mvs_fuse_depth_maps (host arrays, host code:
	the sequential greedy order is the specification).  views[i] (index = image ID): dict with depth (h, w) float32 — MODIFIED in
	place like the reference's depth-maps (depths behind an accepted point are zeroed) — or None, normal (h, w, 3) / conf (h, w) /
	color (h, w, 3) uint8 or None, K R C, neighbors (image IDs, best first) and n_scene_neighbors (the connection score)."""
	lib = _lib.load()
	n = len(views)
	arr = (_lib.FuseView*n)()
	keep = []
	for i, v in enumerate(views):
		o = arr[i]
		d = v.get("depth")
		if d is not None:
			if not (isinstance(d, np.ndarray) and d.dtype == np.float32 and d.flags.c_contiguous and d.flags.writeable):
				raise ValueError("views[%d].depth must be a writeable C-contiguous float32 array (it is modified in place)" % i)
			o.height, o.width = d.shape
			o.depth = d.ctypes.data
			for key, dt, shape in (("normal", np.float32, d.shape+(3,)), ("conf", np.float32, d.shape), ("color", np.uint8, d.shape+(3,))):
				a = v.get(key)
				if a is not None:
					a = np.ascontiguousarray(a, dt)
					if a.shape != shape:
						raise ValueError("views[%d].%s has shape %s, expected %s" % (i, key, a.shape, shape))
					keep.append(a); setattr(o, key, a.ctypes.data)
		for name in ("K", "R", "C"):
			getattr(o, name)[:] = list(np.asarray(v[name], np.float64).ravel())
		nb = np.ascontiguousarray(v.get("neighbors", []), np.uint32)
		keep.append(nb)
		o.neighbors = nb.ctypes.data if nb.size else None
		o.nNeighbors = int(nb.size)
		o.nSceneNeighbors = int(v.get("n_scene_neighbors", nb.size))
	prm = _lib.FuseParams(int(nMinViewsFuse), float(fDepthDiffThreshold), float(fNormalDiffThreshold), int(bool(bEstimateColor)), int(bool(bEstimateNormal)))
	cloud = C.c_void_p()
	rc = lib.b200mvs_fuse_depth_maps(arr, n, C.byref(prm), C.byref(cloud))
	if rc:
		raise _lib.B200MVSError("b200mvs_fuse_depth_maps failed with status %d (bad view description)" % rc)
	try:
		m = int(lib.b200mvs_pointcloud_size(cloud))
		def take(fn, count, dt):
			p = fn(cloud)
			return np.ctypeslib.as_array(p, shape=(count,)).astype(dt, copy=True) if (count and p) else None
		off = take(lib.b200mvs_pointcloud_view_offsets, m+1, np.uint32)
		total = int(off[-1]) if off is not None else 0
		pts = take(lib.b200mvs_pointcloud_points, 3*m, np.float32)
		vs = take(lib.b200mvs_pointcloud_views, total, np.uint32); ws = take(lib.b200mvs_pointcloud_weights, total, np.float32)
		pj = take(lib.b200mvs_pointcloud_projs, 2*total, np.uint16)
		nr = take(lib.b200mvs_pointcloud_normals, 3*m, np.float32); cl = take(lib.b200mvs_pointcloud_colors, 3*m, np.uint8)
		return PointCloud(points=pts.reshape(-1, 3) if pts is not None else np.zeros((0, 3), np.float32),
			pointViews=[vs[off[i]:off[i+1]] for i in range(m)], pointWeights=[ws[off[i]:off[i+1]] for i in range(m)],
			colors=None if cl is None else cl.reshape(-1, 3), normals=None if nr is None else nr.reshape(-1, 3),
			projs=[pj[2*off[i]:2*off[i+1]].reshape(-1, 2) for i in range(m)], nDepths=int(lib.b200mvs_pointcloud_depths(cloud)))
	finally:
		lib.b200mvs_pointcloud_free(cloud)
