"""Coarse-to-fine (tSGM) matching on the device (b200mvs_sgm_match_tsgm_device and its building blocks) against the CPU oracle
(oracle/tsgm_oracle.cpp), OpenCV and the analytic disparity of synthetic pairs."""
import ctypes as C

import numpy as np
import pytest

from tsgm_common import NO_DISP, pair, sparse_seed, accuracy

torch = pytest.importorskip("torch")
cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sgm():
	if not torch.cuda.is_available():
		pytest.skip("no CUDA device")
	from openmvs_b200.depth_estimator import SemiGlobalMatcher
	from oracle import tsgm_oracle as O
	m = SemiGlobalMatcher()
	yield m, O
	m.Release()


def _dev(a):
	return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _maps(rng, h, w, kind):
	if kind == "dense":
		d = (rng.randint(-6, 7, (h, w)) + np.arange(w)//3).astype(np.int16)
		d[rng.rand(h, w) < 0.1] = NO_DISP
	elif kind == "sparse":
		d = np.full((h, w), NO_DISP, np.int16)
		m = rng.rand(h, w) < 0.03
		d[m] = rng.randint(-60, 120, int(m.sum()))
	elif kind == "wide":
		d = rng.randint(-100, 100, (h, w)).astype(np.int16)
	else:
		d = np.full((h, w), NO_DISP, np.int16)
	return d


@pytest.mark.parametrize("kind", ["dense", "sparse", "wide", "empty"])
def test_range_map_bit_exact(sgm, kind):
	m, O = sgm
	rng = np.random.RandomState(len(kind))
	for h, w in ((9, 13), (129, 234), (84, 154)):
		D = _maps(rng, h, w, kind)
		for mnd, mndi, border in ((11, 33, True), (5, 7, False)):
			M = np.full((2*h+6+rng.randint(0, 3), 2*w+6+rng.randint(0, 3)), 255, np.uint8)
			if border:
				M[:, :5] = 0; M[-3:, :] = 0; M[rng.rand(*M.shape) < 0.05] = 0
			want, n, mx = O.sgm_range_map(D, M, mnd, mndi)
			px, n_d, mx_d = m.Disparity2RangeMap(_dev(D), _dev(M), mnd, mndi)
			assert (n_d, mx_d) == (n, mx)
			got = px.cpu().numpy().view(want.dtype).ravel()
			for f in ("idx", "dmin", "dmax"):
				assert np.array_equal(got[f], want[f]), f


def test_flip_speckles_extract_upscale_bit_exact(sgm):
	m, O = sgm
	rng = np.random.RandomState(5)
	for h, w in ((7, 11), (129, 234), (354, 634)):
		for kind in ("dense", "sparse", "empty"):
			D = _maps(rng, h, w, kind)
			D[rng.rand(h, w) < 0.3] = rng.randint(-3, 4)
			assert np.array_equal(m.FlipDirection(_dev(D)).cpu().numpy(), O.sgm_flip_direction(D))
			for size, diff in ((100, 5), (4, 1)):
				assert np.array_equal(m.FilterSpeckles(_dev(D), NO_DISP, size, diff).cpu().numpy(), O.filter_speckles(D, NO_DISP, size, diff))
			M = np.full((h, w), 255, np.uint8); M[rng.rand(h, w) < 0.1] = 0
			assert np.array_equal(m.ExtractMask(_dev(D), _dev(M), 3).cpu().numpy(), O.sgm_extract_mask(D, M, 3))
			for w2, h2 in ((2*w+6, 2*h+6), (2*w+3, 2*h+4)):
				assert np.array_equal(m.UpscaleMask(_dev(M), w2, h2).cpu().numpy(), O.sgm_upscale_mask(M, w2, h2))
	# a structured map with large regions: OpenCV's own filterSpeckles
	ys, xs = np.mgrid[0:300, 0:500]
	img = (xs//7 + 9*(ys//11)).astype(np.int16)
	img[(xs*3+ys) % 13 == 0] = NO_DISP
	ref = img.copy(); cv2.filterSpeckles(ref, NO_DISP, 100, 5)
	assert np.array_equal(m.FilterSpeckles(_dev(img)).cpu().numpy(), ref)


@pytest.mark.parametrize("factor", [2, 4, 8])
def test_bgr_area_resize_matches_opencv(sgm, factor):
	m, _ = sgm
	rng = np.random.RandomState(factor)
	for h, w in ((1080, 1920), (37, 53), (361, 641)):
		img = rng.randint(0, 256, (h, w, 3)).astype(np.uint8)
		ref = cv2.resize(img, None, fx=1.0/factor, fy=1.0/factor, interpolation=cv2.INTER_AREA)
		assert np.array_equal(m.ResizeAreaBGR8(_dev(img), factor).cpu().numpy(), ref)


def _compare(d, want, gt):
	vd, vw = d != NO_DISP, want != NO_DISP
	assert (vd != vw).mean() < 0.02
	both = vd & vw
	assert (np.abs(d.astype(np.int32)-want.astype(np.int32))[both] > 1).mean() < 0.02
	cov, acc = accuracy(d, gt)
	cov_o, acc_o = accuracy(want, gt)
	assert abs(cov-cov_o) <= 0.01 and abs(acc-acc_o) <= 0.01, ((cov, acc), (cov_o, acc_o))
	return cov, acc


@pytest.mark.parametrize("size", [(640, 360), (1280, 720)])
@pytest.mark.parametrize("seeded", [False, True])
def test_level_loop_matches_oracle(sgm, size, seeded):
	m, O = sgm
	w, h = size
	lg, lc, rg, rc, gt = pair(w, h)
	L, sw, sh = m.TsgmLevels(w, h)
	assert (L, sw, sh) == O.sgm_tsgm_levels(w, h)
	sd = sparse_seed(gt, L, sw, sh) if seeded else None
	want, wcost = O.sgm_match_tsgm(lg, lc, rg, rc, seed=sd)
	d, cost = m.MatchPyramidDevice(_dev(lg), _dev(lc), _dev(rg), _dev(rc), seed=None if sd is None else _dev(sd))
	d = d.cpu().numpy()
	cov, acc = _compare(d, want, gt)
	assert cov > 0.88 and acc > 0.88
	assert m.stats.levels == L
	# the host form computes the same integers
	hd, hcost = m.MatchPyramid(lg, lc, rg, rc, seed=sd)
	assert np.array_equal(hd, d) and np.array_equal(hcost.view(np.int16), cost.cpu().numpy())


def test_masks_follow_the_oracle(sgm):
	m, O = sgm
	w, h = 640, 360
	lg, lc, rg, rc, gt = pair(w, h)
	lm = np.full((h, w), 255, np.uint8); rm = lm.copy()
	lm[:, :40] = 0; rm[:, -25:] = 0; lm[100:140, 300:360] = 0
	want, _ = O.sgm_match_tsgm(lg, lc, rg, rc, lm, rm)
	d, _ = m.MatchPyramidDevice(_dev(lg), _dev(lc), _dev(rg), _dev(rc), _dev(lm), _dev(rm))
	d = d.cpu().numpy()
	assert (d[:, :34] == NO_DISP).all()
	_compare(d, want, gt)


def test_disparity_span_beyond_256(sgm):
	"""d from 10 to 290 px: more than the 256 disparities one global range can hold, matched from a sparse seed"""
	m, O = sgm
	w, h = 1280, 720
	lg, lc, rg, rc, gt = pair(w, h, d0=150.0, amp=140.0)
	L, sw, sh = m.TsgmLevels(w, h)
	sd = sparse_seed(gt, L, sw, sh)
	want, _ = O.sgm_match_tsgm(lg, lc, rg, rc, seed=sd)
	d, _ = m.MatchPyramidDevice(_dev(lg), _dev(lc), _dev(rg), _dev(rc), seed=_dev(sd))
	_compare(d.cpu().numpy(), want, gt)
	from openmvs_b200 import lib
	with pytest.raises(lib.B200MVSError):
		m.MatchPairDevice(_dev(lg), _dev(lc), _dev(rg), _dev(rc), -300, 0)


def test_wrong_seed_or_mask_sizes_are_argument_errors(sgm):
	m, _ = sgm
	w, h = 640, 360
	lg, lc, rg, rc, gt = pair(w, h)
	L, sw, sh = m.TsgmLevels(w, h)
	t = [_dev(a) for a in (lg, lc, rg, rc)]
	out = [torch.empty((h-6, w-6), dtype=torch.int16, device="cuda") for _ in range(2)]
	seed = torch.full((sh, sw+1), NO_DISP, dtype=torch.int16, device="cuda")
	mask = torch.full((h, w), 255, dtype=torch.uint8, device="cuda")
	dll = m._lib
	def call(mk, mw, mh, sd, ssw, ssh):
		return dll.b200mvs_sgm_match_tsgm_device(m._ctx, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), w, h,
			mk, mk, mw, mh, sd, ssw, ssh, 320, 100, 4, None, out[0].data_ptr(), out[1].data_ptr(), None, None)
	assert call(None, 0, 0, seed.data_ptr(), sw+1, sh) == 1
	assert call(None, 0, 0, seed.data_ptr(), sw, sh+1) == 1
	assert call(mask.data_ptr(), w-1, h, None, 0, 0) == 1
	assert call(mask.data_ptr(), w, h+2, None, 0, 0) == 1
	assert call(mask.data_ptr(), w, h, None, 0, 0) == 0
	torch.cuda.synchronize()
	with pytest.raises(ValueError):
		m.MatchPyramidDevice(*t, leftMask=mask, rightMask=mask[:, 1:])
