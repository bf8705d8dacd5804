"""Shared inputs of the coarse-to-fine SGM tests: synthetic pairs and sparse seeds from the analytic disparity."""
import numpy as np

from openmvs_b200 import synth

NO_DISP = 32767


def pair(width, height, d0=12.0, amp=6.0):
	"""-> left gray, left BGR, right gray, right BGR, ground-truth disparity (full resolution)"""
	lg, lc, rg, gt, rc = synth.make_stereo_pair(width, height, d0=d0, amp=amp, right_color=True)
	return lg, lc, rg, rc, gt


def sparse_seed(gt, levels, seed_w, seed_h, frac=0.03, seed=1):
	"""int16 seed at half the coarsest scale (1 / 2^levels of the full resolution): a `frac` share of its pixels carry the rounded
	analytic disparity at that scale, the rest NO_DISP"""
	rng = np.random.RandomState(seed)
	f = 2**levels
	h, w = gt.shape
	ys, xs = np.mgrid[0:seed_h, 0:seed_w]
	X = np.clip(np.rint((xs+3+0.5)*f-0.5).astype(int), 0, w-1)
	Y = np.clip(np.rint((ys+3+0.5)*f-0.5).astype(int), 0, h-1)
	sd = np.full((seed_h, seed_w), NO_DISP, np.int16)
	m = rng.rand(seed_h, seed_w) < frac
	sd[m] = np.rint(gt[Y, X]/f).astype(np.int16)[m]
	return sd


def accuracy(disp, gt, steps=4):
	"""(coverage, share of the valid region within 0.5 px of the analytic disparity) of a refined disparity map"""
	g = gt[3:-3, 3:-3]
	valid = disp != NO_DISP
	err = np.abs(disp.astype(np.float64)/steps - g)
	return float(valid.mean()), float((valid & (err <= 0.5)).mean())
