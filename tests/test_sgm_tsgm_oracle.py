"""CPU oracle of the coarse-to-fine (tSGM) level loop (oracle/tsgm_oracle.cpp) against OpenCV and against independent pure-Python
transcriptions of the reference functions (libs/MVS/SemiGlobalMatcher.cpp:1350-1444, 1518-1575, 1630-1690), and the whole loop
against the analytic disparity of synthetic pairs."""
import numpy as np
import pytest

from oracle import tsgm_oracle as O
from tsgm_common import NO_DISP, pair, sparse_seed, accuracy

cv2 = pytest.importorskip("cv2")


# ---- pure-Python transcriptions of the reference ----
def py_median(v):
	v = sorted(v)
	n = len(v)
	if n % 2:
		return v[n//2]
	s = v[n//2-1] + v[n//2]
	return int(s/2)  # C division truncates toward zero


def i16(x):
	return int(np.int16(np.int64(x)))


def py_range_map(D, M, minNumDisp, minNumDispInvalid):
	dh, dw = D.shape
	mh, mw = M.shape
	recs = [None]*(mw*mh)
	numCosts = 0
	maxNumDisp = 0
	for r in range(dh):
		r2 = 0 if r == 0 else r*2+3
		offset = r2*mw
		c2e = 3
		c2 = 0
		for c in range(dw):
			if M[r*2+3, 3+2*c] == 0:
				lo = hi = NO_DISP; num = 0
			else:
				bInvalid = D[r, c] == NO_DISP
				hw = 20 if bInvalid else 3
				disps = [int(D[y, x]) for y in range(r-hw, r+hw+1) for x in range(c-hw, c+hw+1)
					if 0 <= x < dw and 0 <= y < dh and D[y, x] != NO_DISP]
				if len(disps) < 3:
					hi = min(i16(dw*2//3), minNumDispInvalid); lo = -hi; num = hi-lo
				else:
					disp = i16(i16(py_median(disps))*2)
					mn, mx = min(disps), max(disps)
					num = i16((mx-mn)*2)
					if num < minNumDisp:
						num = minNumDisp
						lo = i16(disp-int(num/2)); hi = i16(disp+int((num+1)/2))
					else:
						M_ = 64 if bInvalid else 32
						if num > M_:
							lo = i16(disp-int((M_*(disp-mn*2)+1)/num)); hi = i16(disp+int((M_*(mx*2+1-disp)+1)/num)); num = hi-lo
						else:
							lo = i16(disp-int(num/2)); hi = i16(disp+int((num+1)/2))
				maxNumDisp = max(maxNumDisp, num)
			c2e += 2
			while c2 < c2e:
				recs[offset+c2] = (numCosts, lo, hi); numCosts += num; c2 += 1
		while c2e < mw:
			_, lo_, hi_ = recs[offset+c2e-1]
			recs[offset+c2e] = (numCosts, lo_, hi_); numCosts += hi_-lo_; c2e += 1
		end = (mh if r+1 == dh else r*2+5)*mw
		for o in range(offset+mw, end, mw):
			for c2 in range(mw):
				_, lo_, hi_ = recs[offset+c2]
				recs[o+c2] = (numCosts, lo_, hi_); numCosts += hi_-lo_
	return recs, numCosts, maxNumDisp


def py_flip(l2r):
	h, w = l2r.shape
	out = np.full_like(l2r, NO_DISP)
	for r in range(h):
		for c in range(w):
			d = int(l2r[r, c])
			if d == NO_DISP:
				continue
			for x in range(max(c+d-1, 0), min(c+d+2, w)):
				out[r, x] = i16(-d)
	return out


def py_extract_mask(D, M, th=3):
	M = M.copy()
	h, w = D.shape
	for cols in (range(w), range(w-1, -1, -1)):
		for r in range(h):
			n = 0
			for c in cols:
				if M[r, c] == 0:
					continue
				M[r, c] = 0
				if D[r, c] == NO_DISP:
					continue
				n += 1
				if n >= th:
					break
	return M


def py_upscale_mask(M, w2, h2):
	out = np.zeros((h2, w2), np.uint8)
	h, w = M.shape
	for r in range(h):
		for c in range(w):
			for i in range(2):
				for j in range(2):
					y, x = r*2+3+i, c*2+3+j
					if x < w2 and y < h2:
						out[y, x] = M[r, c]
	return out


# ---- small maps: dense, sparse seed, all NO_DISP; masks with invalid borders; odd sizes ----
def small_map(kind, h, w, rng):
	if kind == "dense":
		d = (rng.randint(-6, 7, (h, w)) + np.arange(w)//3).astype(np.int16)
		d[rng.rand(h, w) < 0.1] = NO_DISP
	elif kind == "sparse":
		d = np.full((h, w), NO_DISP, np.int16)
		m = rng.rand(h, w) < 0.04
		d[m] = rng.randint(-40, 80, int(m.sum()))
	elif kind == "wide":
		d = rng.randint(-100, 100, (h, w)).astype(np.int16)
	else:
		d = np.full((h, w), NO_DISP, np.int16)
	return d


def small_mask(h, w, rng, border=True):
	m = np.full((h, w), 255, np.uint8)
	if border:
		m[:, :rng.randint(1, 9)] = 0; m[-rng.randint(1, 6):, :] = 0
		m[rng.rand(h, w) < 0.05] = 0
	return m


@pytest.mark.parametrize("kind", ["dense", "sparse", "wide", "empty"])
@pytest.mark.parametrize("size", [(9, 13), (24, 31)])
def test_range_map_matches_reference_transcription(kind, size):
	rng = np.random.RandomState(hash((kind, size)) & 0xFFFF)
	h, w = size
	D = small_map(kind, h, w, rng)
	for first, border in ((True, True), (False, False)):
		M = small_mask(2*h+2+rng.randint(0, 3), 2*w+4+rng.randint(0, 3), rng, border)
		mnd, mndi = (11, 33) if first else (5, 7)
		px, n, mx = O.sgm_range_map(D, M, mnd, mndi)
		recs, n_ref, mx_ref = py_range_map(D, M, mnd, mndi)
		assert n == n_ref and mx == mx_ref
		assert [tuple(int(v) for v in (p["idx"], p["dmin"], p["dmax"])) for p in px] == recs


@pytest.mark.parametrize("size", [(7, 11), (20, 33)])
def test_flip_extract_upscale_match_reference_transcriptions(size):
	rng = np.random.RandomState(size[0]*100+size[1])
	h, w = size
	for kind in ("dense", "sparse", "empty"):
		D = small_map(kind, h, w, rng)
		D[rng.rand(h, w) < 0.3] = rng.randint(-3, 4)  # overlapping writes
		assert np.array_equal(O.sgm_flip_direction(D), py_flip(D))
		M = small_mask(h, w, rng)
		assert np.array_equal(O.sgm_extract_mask(D, M, 3), py_extract_mask(D, M, 3))
		for w2, h2 in ((2*w+6, 2*h+6), (2*w+3, 2*h+4), (2*w+9, 2*h+5)):
			assert np.array_equal(O.sgm_upscale_mask(M, w2, h2), py_upscale_mask(M, w2, h2))


@pytest.mark.parametrize("kind", ["random", "structured"])
def test_filter_speckles_matches_opencv(kind):
	rng = np.random.RandomState(3 if kind == "random" else 4)
	for t in range(12):
		h, w = rng.randint(8, 90), rng.randint(8, 90)
		if kind == "random":
			img = rng.randint(-12, 12, (h, w)).astype(np.int16)
			img[rng.rand(h, w) < 0.3] = NO_DISP
		else:
			ys, xs = np.mgrid[0:h, 0:w]
			img = (xs//5 + 7*(ys//9)).astype(np.int16)
			img[(xs*3+ys) % 11 == 0] = NO_DISP
			img[rng.rand(h, w) < 0.02] = rng.randint(-200, 200)
		for size, diff in ((100, 5), (7, 1), (30, 0)):
			ref = img.copy()
			cv2.filterSpeckles(ref, NO_DISP, size, diff)
			assert np.array_equal(O.filter_speckles(img, NO_DISP, size, diff), ref), (t, size, diff)


@pytest.mark.parametrize("factor", [2, 4, 8])
def test_area_resize_u8_matches_opencv(factor):
	rng = np.random.RandomState(factor)
	for h, w in ((64, 96), (37, 53), (81, 129), (270, 481)):
		for shape in ((h, w, 3), (h, w)):
			img = rng.randint(0, 256, shape).astype(np.uint8)
			ref = cv2.resize(img, None, fx=1.0/factor, fy=1.0/factor, interpolation=cv2.INTER_AREA)
			assert np.array_equal(O.resize_area_u8(img, factor), ref), (h, w, shape)


def test_levels_and_seed_size():
	assert O.sgm_tsgm_levels(1920, 1080) == (3, 234, 129)
	assert O.sgm_tsgm_levels(1280, 720) == (3, 154, 84)
	assert O.sgm_tsgm_levels(640, 360) == (2, 154, 84)
	assert O.sgm_tsgm_levels(320, 240) == (2, 74, 54)


# coverage / share within 0.5 px the oracle's loop reaches (recorded: 320x240 0.907 / 0.903, 640x360 0.954 / 0.951, without and
# with a 3 % seed); the GPU loop is held to these within one point
@pytest.mark.parametrize("size,seeded", [((320, 240), False), ((320, 240), True), ((640, 360), True)])
def test_oracle_level_loop_reaches_analytic_disparity(size, seeded):
	w, h = size
	lg, lc, rg, rc, gt = pair(w, h)
	L, sw, sh = O.sgm_tsgm_levels(w, h)
	sd = sparse_seed(gt, L, sw, sh) if seeded else None
	disp, cost = O.sgm_match_tsgm(lg, lc, rg, rc, seed=sd)
	cov, acc = accuracy(disp, gt)
	assert cov > 0.88 and acc > 0.88, (cov, acc)
	assert (cost[disp != NO_DISP] < 65535).all()
