"""Coarse-to-fine (tSGM) matching of one 1920x1080 synthetic pair on the GPU (SemiGlobalMatcher.MatchPyramidDevice, three levels
1/4, 1/2, 1, 3 % sparse seed), alternated with the one-range matcher MatchPairDevice at D = 128 on the same pair.

Records, as JSON in <out>/tsgm_profile.json:
  * device name and power limit (read in this run);
  * ms per pair of both matchers (CUDA events around each call, profiler off, calls alternated);
  * per level: device span and summed kernel time (torch.profiler trace of one extra call), the px*d of the right and left match
    (cost-volume sizes of the oracle's loop on the same pair: its ranges equal the engine's on all but a few % of pixels) and
    G px*d/s over the level's span;
  * kernel launches (b200mvs_stats) and host synchronisations of one call (cudaStreamSynchronize / blocking copies in the trace);
  * the bytes of the largest ragged match: 17 B per px*d allocated (u8 costs, the u16 path costs of eight directions that run side
    by side) against the algorithmic 11 B per px*d count of DESIGN.md;
  * the oracle's level loop on the CPU (wall time).
Needs a GPU: there is no CPU fall-back.  Usage: python scripts/profile_tsgm.py --out DIR [--reps 10]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from openmvs_b200.depth_estimator import SemiGlobalMatcher  # noqa: E402
from tsgm_common import pair, sparse_seed, accuracy  # noqa: E402


def device_info():
	name = torch.cuda.get_device_name(0)
	try:
		q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
			capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
	except Exception as e:  # the number is reported without it, and says so
		q = "nvidia-smi unavailable: %s" % e
	return {"torch_device_name": name, "nvidia_smi": q}


def level_split(events):
	"""kernel events of one MatchPyramidDevice call (time order) -> per level [first start, last end, summed kernel us]; a level begins
	at its first pyramid resize or mask upscale after the previous level's FlipDirection"""
	levels = []
	flip_seen = True
	for name, t0, dur in events:
		marker = "resize_area" in name or "upscale_mask" in name or "resize_nearest_u8" in name or "fill_i16" in name
		if marker and flip_seen:
			levels.append([t0, t0+dur, 0.0])
			flip_seen = False
		if not levels:
			levels.append([t0, t0+dur, 0.0])
		if "flip_scatter" in name:
			flip_seen = True
		lv = levels[-1]
		lv[1] = max(lv[1], t0+dur)
		lv[2] += dur
	return levels


def main():
	ap = argparse.ArgumentParser()
	ap.add_argument("--out", required=True, help="directory for tsgm_profile.json")
	ap.add_argument("--reps", type=int, default=10)
	ap.add_argument("--no-oracle", action="store_true")
	a = ap.parse_args()
	if not torch.cuda.is_available():
		raise SystemExit("profile_tsgm.py needs a CUDA device")
	os.makedirs(a.out, exist_ok=True)
	res = {"device": device_info()}
	W, H = 1920, 1080
	lg, lc, rg, rc, gt = pair(W, H)
	m = SemiGlobalMatcher()
	L, sw, sh = m.TsgmLevels(W, H)
	sd = sparse_seed(gt, L, sw, sh)
	t = [torch.from_numpy(x).cuda() for x in (lg, lc, rg, rc, sd)]
	res["pair"] = {"width": W, "height": H, "levels": L, "seed": [sw, sh], "seed_fraction": float((sd != 32767).mean())}

	def tsgm():
		return m.MatchPyramidDevice(t[0], t[1], t[2], t[3], seed=t[4], sync=False)

	def one_range():
		return m.MatchPairDevice(t[0], t[1], t[2], t[3], -128, 0)

	for _ in range(3):
		tsgm(); one_range()
	torch.cuda.synchronize()
	ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
	ms_t, ms_p = [], []
	for _ in range(a.reps):
		ev[0].record(); d, c = tsgm(); ev[1].record()
		ev[2].record(); one_range(); ev[3].record()
		torch.cuda.synchronize()
		ms_t.append(ev[0].elapsed_time(ev[1])); ms_p.append(ev[2].elapsed_time(ev[3]))
	d, c = tsgm()
	torch.cuda.synchronize()
	cov, acc = accuracy(d.cpu().numpy(), gt)
	res["tsgm_ms"] = {"median": float(np.median(ms_t)), "min": float(np.min(ms_t)), "max": float(np.max(ms_t)), "all": ms_t}
	res["match_pair_D128_ms"] = {"median": float(np.median(ms_p)), "min": float(np.min(ms_p)), "max": float(np.max(ms_p)), "all": ms_p}
	res["tsgm_quality"] = {"coverage": cov, "within_0.5px": acc}

	# one call with stats: launches; one call under the profiler: per-level spans, host synchronisations
	m.MatchPyramidDevice(t[0], t[1], t[2], t[3], seed=t[4], sync=True)
	res["kernel_launches"] = int(m.stats.kernel_launches)
	from torch.profiler import profile, ProfilerActivity
	with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
		tsgm()
		torch.cuda.synchronize()
	kern, syncs = [], 0
	for e in prof.events():
		if e.device_type.name == "CUDA" and e.name and "Memcpy" not in e.name and "Memset" not in e.name:
			kern.append((e.name, e.time_range.start, e.time_range.end-e.time_range.start))
		elif e.name in ("cudaStreamSynchronize", "cudaDeviceSynchronize", "cudaMemcpy"):
			syncs += 1
	kern.sort(key=lambda k: k[1])
	spans = level_split(kern)
	# torch.cuda.synchronize() above is one of the counted synchronisations
	res["host_synchronisations"] = syncs-1
	res["launches_in_trace"] = len(kern)

	t0 = time.time()
	if a.no_oracle:
		vols = None
	else:
		from oracle import tsgm_oracle as O
		od, _, vols = O.sgm_match_tsgm(lg, lc, rg, rc, seed=sd, level_costs=True)
		res["oracle_cpu_s"] = time.time()-t0
		res["oracle_quality"] = dict(zip(("coverage", "within_0.5px"), accuracy(od, gt)))
	res["levels"] = []
	for k, (s0, s1, ksum) in enumerate(spans):
		lv = {"level": k, "scale": 1.0/2**(L-1-k) if k < L else None, "span_ms": (s1-s0)/1e3, "kernel_ms": ksum/1e3}
		if vols and k < len(vols):
			lv["pxd_right"], lv["pxd_left"] = vols[k]
			lv["Gpxd_per_s"] = (vols[k][0]+vols[k][1])/((s1-s0)*1e-6)/1e9
		res["levels"].append(lv)
	if vols:
		big = max(max(v) for v in vols)
		res["ragged_volume"] = {"largest_pxd": big, "bytes_allocated": 17*big, "bytes_11B_per_pxd": 11*big}
	json.dump(res, open(os.path.join(a.out, "tsgm_profile.json"), "w"), indent=1)
	print(json.dumps(res, indent=1))


if __name__ == "__main__":
	main()
