"""The PatchMatch sweep kernel with its patch weights in tensor memory (TMEM, 128 columns per CTA; run with -m gpu).

Its variants must agree bit for bit, and it must share the GPU with the tensor-core cost kernel of the SGM matcher, which
allocates all 512 columns of an SM: on two streams their CTAs share SMs, so an allocation may wait for the other kernel's CTAs
to release theirs.  The maps must come out exactly as when the two run one after the other.
"""
import numpy as np
import pytest
import torch

from openmvs_b200 import synth

pytestmark = pytest.mark.gpu


def _dev(a):
	return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("w,h", [(203, 151), (640, 360)])
def test_sweep_variants_agree(w, h):
	"""The instantiations and fill paths of the sweep kernel give the same maps: weights filled from the TMA tile or from global
	memory (noTMA), 4 CTAs per SM (all 512 TMEM columns of an SM taken), scalar taps.  203 x 151 leaves partial warps and CTAs at
	the right and bottom edges and carries an ignore-mask: lanes without a pixel to update inside warps that have one."""
	if not torch.cuda.is_available():
		pytest.skip("no CUDA device")
	from openmvs_b200.depth_estimator import OPTDENSE, Camera, ViewData, DepthData, PatchMatchB200
	saved = {k: getattr(OPTDENSE, k) for k in dir(OPTDENSE) if k[0] in "nf" and not callable(getattr(OPTDENSE, k))}
	dev = torch.device("cuda:0")
	pm = PatchMatchB200(0)
	try:
		OPTDENSE.nSubResolutionLevels = 0; OPTDENSE.nEstimationGeometricIters = 0; OPTDENSE.nEstimationIters = 3
		sc = synth.make_scene(w, h, 4, step_deg=5.0, device=dev)
		views = [sc.views[1]]+[sc.views[i] for i in sc.neighbors(1, 3)]
		imgs = [ViewData(torch.as_tensor(v.image, device=dev), Camera(v.K, v.R, v.C)) for v in views]
		if w == 203:
			mask = np.ones((h, w), np.uint8)
			mask[20:60, 33:91] = 0
			mask[100:, 150:] = 0
			pm.SetIgnoreMask(mask)

		def run(**dbg):
			pm.SetDebug(**dbg)
			dd = DepthData(imgs, sc.dmin, sc.dmax)
			pm.EstimateDepthMap(dd)
			return dd, int(pm.stats.tma_active)

		ref, tma = run()
		assert tma == 1
		assert (ref.depthMap > 0).float().mean().item() > 0.5
		for dbg in ({"noTMA": 1}, {"sweepFourCtas": 1}, {"scalarTaps": 1}):
			dd, _ = run(**dbg)
			for name in ("depthMap", "normalMap", "confMap", "viewsMap"):
				assert torch.equal(getattr(ref, name), getattr(dd, name)), (dbg, name)
	finally:
		for k, v in saved.items():
			setattr(OPTDENSE, k, v)
		pm.SetDebug()
		pm.SetIgnoreMask(None)
		pm.Release()


def test_sweep_and_sgm_tensor_core_cost_concurrently():
	if not torch.cuda.is_available():
		pytest.skip("no CUDA device")
	from openmvs_b200.depth_estimator import OPTDENSE, Camera, ViewData, DepthData, PatchMatchB200, SemiGlobalMatcher
	saved = {k: getattr(OPTDENSE, k) for k in dir(OPTDENSE) if k[0] in "nf" and not callable(getattr(OPTDENSE, k))}
	dev = torch.device("cuda:0")
	pm = PatchMatchB200(0)
	sgm = SemiGlobalMatcher()
	try:
		OPTDENSE.nSubResolutionLevels = 0; OPTDENSE.nEstimationGeometricIters = 0; OPTDENSE.nEstimationIters = 4
		sc = synth.make_scene(960, 540, 6, step_deg=4.0, device=dev)
		r = 2
		views = [sc.views[r]]+[sc.views[i] for i in sc.neighbors(r, 5)]
		imgs = [ViewData(torch.as_tensor(v.image, device=dev), Camera(v.K, v.R, v.C)) for v in views]
		lg, lc, rg, _ = synth.make_stereo_pair(1920, 1080, d0=40.0, amp=25.0)
		px, n = synth.sgm_pixel_map(1920, 1080, 0, 128)
		sgm_args = (_dev(lg), _dev(lc), _dev(rg), torch.from_numpy(px.view(np.uint8).reshape(-1, 16).copy()).cuda(), n)
		sgm.SetDebug(sgmCost=2)   # the tensor-core cost kernel (tcgen05, 512 TMEM columns per CTA)

		def pm_run():
			dd = DepthData(imgs, sc.dmin, sc.dmax)
			pm.EstimateDepthMap(dd, sync=False)
			return dd

		# one after the other
		dd0 = pm_run()
		torch.cuda.synchronize()
		ref = sgm.MatchDevice(*sgm_args)
		torch.cuda.synchronize()

		# concurrently: PatchMatch on one stream, several SGM matches on another
		s_pm, s_sgm = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
		s_pm.wait_stream(torch.cuda.current_stream(dev)); s_sgm.wait_stream(torch.cuda.current_stream(dev))
		with torch.cuda.stream(s_pm):
			dd1 = pm_run()
		outs = []
		with torch.cuda.stream(s_sgm):
			for _ in range(4):
				outs.append(sgm.MatchDevice(*sgm_args, sync=False))
		torch.cuda.synchronize()

		for name in ("depthMap", "normalMap", "confMap", "viewsMap"):
			assert torch.equal(getattr(dd0, name), getattr(dd1, name)), name
		assert (dd0.depthMap > 0).float().mean().item() > 0.5
		for gd, gc in outs:
			assert torch.equal(gd, ref[0]) and torch.equal(gc, ref[1])
	finally:
		for k, v in saved.items():
			setattr(OPTDENSE, k, v)
		sgm.SetDebug()
		sgm.Release()
		pm.Release()
