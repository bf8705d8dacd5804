#!/usr/bin/env python
"""bench.py — Mpix/s of depth+normal estimation (BASELINE.json metric).

Default workload (config.workload "C2"): BASELINE.json configs[1] — a 12-image synthetic scene at 1920x1080, every image
used once as reference view with its 9 nearest neighbours, PatchMatch 6 iterations, single scale, no geometric pass
(SURVEY.md §8(d) C2).  One step = the 12 DepthMapsData::EstimateDepthMap calls of that scene on one GPU.  With N GPUs every
rank estimates its OWN 12-view scene (seed 1234 + rank: distinct images per rank; weak scaling, reference views are
independent, no data-path collective) and the maps are gathered on rank 0 over NCCL inside the timed region.

  value      device-resident throughput: images already in HBM, reference views alternating between two contexts on two
             CUDA streams (joined back into the timing stream), CUDA events, barrier + synchronize on both sides, max over
             ranks.
  e2e        the same work through the reference-facing call with HOST buffers (pinned): b200mvs_estimate_async +
             b200mvs_sync on two contexts used alternately, so that the copies of one reference view overlap the kernels of
             the other; per reference view the H2D copy of its 10 images + initial maps and the D2H read of
             depth/normal/conf/views are inside the timed region; with N > 1 the NCCL gather of the ranks' maps as well.
  roofline   dominant kernel (pm_sweep_kernel, one red-black half-sweep), timed live with CUDA events on its launch stream;
             algorithmic bytes per launch = (20 B plane+cost read for every pixel + 20 B written for the active half +
             4(N+1) B of images) per pixel (DESIGN.md §5).
  sgm        (N = 1, rank 0) BASELINE configs[2]: one SemiGlobalMatcher::Match of a 1920x1080 pair — fixed range D = 128
             (the non-tSGM branch) and one tSGM-like ragged case — timed live: ms per Match and per stage, G px.d/s, fraction of
             the HBM roofline on SURVEY §8(d)'s 11 B/(px.d), the CPU oracle on a bounded band beside it.
  cpu_baseline / --impl reference
             the reference algorithm (oracle, zig-zag schedule, all host threads) on a bounded sample: a full-width band of
             one reference view, same N and iteration count; CPU model, affinity size and cgroup quota recorded.

Other workloads (secondary lines, same JSON contract; the driver runs the default):
  --workload c4   BASELINE configs[3]: 200 distinct 1920x1080 views (images replicated on every GPU), reference views dealt
                  round-robin over the ranks — strong scaling; NCCL gather of the maps inside the timed region.
  --workload c5   BASELINE configs[4]: 50 views 4032x3024, pass 1 + ONE geometric-consistency pass: per step every rank
                  estimates its views, all-gathers the depth-maps (ncclAllGather, timed separately with CUDA events),
                  re-estimates them with the neighbours' depth-maps, and rank 0 gathers the result.

--dump-outputs DIR
  after the timed steps, rank 0 writes the maps the timed path returned for its reference views in the last step, at one fixed,
  seeded sample of pixels (the same for every view, 32 MB of data at most): DIR/depth.npy [V, P], normal.npy [V, P, 3],
  conf.npy [V, P] and views.npy [V, P, 4], float32.  The scene is seeded, so two builds given the same arguments can be compared
  output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

# the tree the benchmark runs from may be read-only: nothing is written into it
sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
	sys.path.insert(0, ROOT)

W, H, N_VIEWS, N_NEIGH, ITERS = 1920, 1080, 12, 9, 6
METRIC = "Mpix/sec depth+normal (1920x1080, 9 neighbours)"


def parse():
	ap = argparse.ArgumentParser()
	ap.add_argument("--gpus", type=int, default=1)
	ap.add_argument("--steps", type=int, default=3)
	ap.add_argument("--warmup", type=int, default=3)
	ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
	ap.add_argument("--workload", default="c2", choices=["c2", "c4", "c5"])
	ap.add_argument("--views", type=int, default=0, help="c4 / c5: number of views of the scene (default 200 / 50)")
	ap.add_argument("--cpu-band", type=int, default=0, help="rows of the CPU sample band (0: auto)")
	ap.add_argument("--no-cpu-baseline", action="store_true")
	ap.add_argument("--no-sgm", action="store_true")
	ap.add_argument("--small", action="store_true", help="developer mode: 640x360 scene")
	ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's maps to DIR/*.npy")
	args = ap.parse_args()
	if args.steps < 1:
		ap.error("--steps must be at least 1")
	if args.dump_outputs and args.impl == "reference":
		ap.error("--dump-outputs writes the engine's maps: not with --impl reference")
	return args


DUMP_BYTES = 32_000_000


def dump_outputs(directory, stack, views):
	"""DIR/<map>.npy of the maps `stack` holds for `views`, at a fixed, seeded sample of pixels (sorted, the same for every
	view) sized to keep the four files within DUMP_BYTES."""
	import torch
	hw = stack.h*stack.w
	n = min(hw, DUMP_BYTES//(len(views)*9*4))   # 9 floats per pixel: depth, normal, conf, 4 view ids
	idx = torch.from_numpy(np.sort(np.random.RandomState(0).choice(hw, n, replace=False))).to(stack.depth.device)
	slots = torch.tensor([stack.slot(v) for v in views], device=stack.depth.device)
	os.makedirs(directory, exist_ok=True)
	for name, t, c in (("depth", stack.depth, 1), ("normal", stack.normal, 3), ("conf", stack.conf, 1), ("views", stack.views, 4)):
		a = t.view(t.shape[0], hw, c)[:, idx][slots].float().cpu().numpy()
		np.save(os.path.join(directory, name+".npy"), a[..., 0] if c == 1 else a)


class ClockSampler:
	"""nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
	Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

	def __init__(self, index: int):
		self.index = index
		self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
		self.p = None

	def start(self):
		try:
			self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu="+self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
				stdout=self.f, stderr=subprocess.DEVNULL)
		except Exception:
			self.p = None

	def stop(self):
		if self.p is not None:
			self.p.terminate()
			try:
				self.p.wait(5)
			except Exception:
				self.p.kill()
		self.f.flush(); self.f.seek(0)
		sm, mx, reasons = [], [], set()
		for line in self.f.read().splitlines():
			c = [x.strip() for x in line.split(",")]
			if len(c) < 9:
				continue
			try:
				sm.append(float(c[1])); mx.append(float(c[2]))
			except ValueError:
				continue
			for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
				if val.lower().startswith("active"):
					reasons.add(name)
		try:
			os.unlink(self.f.name)
		except OSError:
			pass
		if not sm:
			return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
		busy = [s for s in sm if s > 0.5*max(sm)] or sm
		return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def host_info(threads):
	"""what the CPU arm ran on: model, logical CPUs, affinity size, cgroup quota (a 5.5x box-to-box spread was seen in round 1)"""
	info = {"threads_used": threads, "nproc": os.cpu_count()}
	try:
		for line in open("/proc/cpuinfo"):
			if line.startswith("model name"):
				info["cpu_model"] = line.split(":", 1)[1].strip(); break
	except Exception:
		pass
	try:
		info["affinity"] = len(os.sched_getaffinity(0))
	except Exception:
		pass
	for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
		try:
			info["cgroup_cpu_max"] = open(path).read().strip(); break
		except Exception:
			pass
	try:
		info["loadavg_1m"] = float(open("/proc/loadavg").read().split()[0])
	except Exception:
		pass
	return info


def build_scene(device, w, h, n_views=N_VIEWS, seed=1234, gt_views=None):
	from openmvs_b200 import synth
	return synth.make_scene(w, h, n_views, seed=seed, step_deg=4.0, device=device, gt_views=gt_views)


def cpu_sample(scene, w, h, band_rows, threads):
	"""The reference algorithm on a bounded sample: reference view 5, rows [y0, y0+band) as a cropped pinhole view (principal
	point shifted), full neighbour images, N and iterations as in the GPU workload; the throughput build of the oracle
	(-O3 -march=native).  Returns (Mpix/s, seconds, description, valid fraction)."""
	from oracle import oracle as O
	from openmvs_b200 import synth
	ref = 5
	nb = scene.neighbors(ref, N_NEIGH)
	v = scene.views[ref]
	y0 = (h-band_rows)//2
	K = v.K.copy(); K[1, 2] -= y0
	crop = synth.View(np.ascontiguousarray(v.image[y0:y0+band_rows]), K, v.R, v.C, v.depth_gt[y0:y0+band_rows], v.normal_gt[y0:y0+band_rows])
	views = [crop]+[scene.views[i] for i in nb]
	prm = O.default_params(schedule=0, nEstimationIters=ITERS, nSubResolutionLevels=0, nEstimationGeometricIters=0, threads=threads)
	fast = hasattr(O, "use_fast_build") and O.use_fast_build(True)
	try:
		t = time.perf_counter()
		d, n, c = O.pm_estimate(views, prm, scene.dmin, scene.dmax)
		dt = time.perf_counter()-t
	finally:
		if fast:
			O.use_fast_build(False)
	mpix = w*band_rows/1e6/dt
	desc = "oracle ZZ schedule (reference algorithm restated, %s build), ref view %d rows %d..%d (%dx%d band), %d neighbours, %d iters, %d threads" % (
		"-O3 -march=native" if fast else "-O2 parity", ref, y0, y0+band_rows, w, band_rows, N_NEIGH, ITERS, threads)
	return mpix, dt, desc, float((d > 0).mean())


def sgm_block(dev, peak, threads):
	"""BASELINE configs[2]: SemiGlobalMatcher::Match of one 1920x1080 pair, timed live (CUDA events of the C-ABI on its stream)."""
	import torch
	from openmvs_b200 import synth
	from openmvs_b200.depth_estimator import SemiGlobalMatcher
	w, h, D = 1920, 1080, 128
	lg, lc, rg, d = synth.make_stereo_pair(w, h, d0=40.0, amp=25.0)
	todev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
	pxd = lambda px: torch.from_numpy(px.view(np.uint8).reshape(-1, 16).copy()).to(dev)
	m = SemiGlobalMatcher(device=dev.index or 0)
	out = {"workload": "C3: 1920x1080 rectified pair, valid region 1914x1074, WZNCC 7x7 cost + 8-path aggregation + WTA per Match"}
	L, C3, R = todev(lg), todev(lc), todev(rg)

	def run(px, n, reps=5):
		P = pxd(px)
		costs = torch.zeros(n, dtype=torch.uint8, device=dev); accums = torch.zeros(n, dtype=torch.int16, device=dev)
		res = {}
		for name, st in (("cost", 1), ("aggregate", 2), ("wta", 4), ("match", 7)):
			ms = []
			for rep in range(2+reps):
				disp, cost = m.MatchDevice(L, C3, R, P, n, stages=st, costs=costs, accums=accums)
				if rep >= 2:
					ms.append(m.stats.ms_device)
			res["ms_"+name] = float(np.median(ms))
		res["kernel_launches"] = int(m.stats.kernel_launches)
		return res, disp

	px, n = synth.sgm_pixel_map(w, h, 0, D)
	fixed, disp = run(px, n)
	gt = d[3:-3, 3:-3]
	fixed["px_d"] = int(n)
	fixed["gpxd_per_s"] = n/fixed["ms_match"]/1e6
	fixed["within_1px_of_ground_truth"] = float((np.abs(disp.cpu().numpy()-gt)[8:-8, 8:-140] <= 1).mean())
	ach = 11.0*n/(fixed["ms_match"]*1e-3)/1e9
	fixed["roofline"] = {"bound": "hbm", "algorithmic_bytes_per_px_d": 11, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach/peak, "traffic": None}
	tf = os.path.join(ROOT, "profiles", "sgm_traffic.json")
	if os.path.exists(tf):
		try:
			t = json.load(open(tf))
			fixed["roofline"]["traffic"] = t.get("dram_bytes_per_match"); fixed["roofline"]["traffic_source"] = t.get("source")
		except Exception:
			pass
	# host API (H2D of the images + pixel map, D2H of the maps inside the call)
	m.Match(lg, lc, rg, px, n)   # warm-up: the host path's staging buffers are allocated on first use
	t0 = time.perf_counter(); m.Match(lg, lc, rg, px, n); m.Match(lg, lc, rg, px, n); fixed["ms_host_api"] = (time.perf_counter()-t0)*500
	out["fixed_range_D128"] = fixed
	# the unit the reference works in: a PAIR (right->left match, left->right match with mirrored ranges, cross-check, sub-pixel
	# refinement; SemiGlobalMatcher.cpp:643-725), the two matches on two contexts / streams
	try:
		lg2, lc2, rg2, d2, rc2 = synth.make_stereo_pair(w, h, d0=40.0, amp=25.0, right_color=True)
		RC = todev(rc2)
		ms = []
		for rep in range(5):
			e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
			torch.cuda.synchronize(dev); e0.record()
			ld, rd = m.MatchPairDevice(L, C3, R, RC, -D, 0)
			e1.record(); torch.cuda.synchronize(dev)
			if rep >= 2:
				ms.append(e0.elapsed_time(e1))
		out["pair_D128"] = {"ms_pair": float(np.median(ms)), "gpxd_per_s": 2*n/float(np.median(ms))/1e6,
			"left_within_1px_of_ground_truth": float((np.abs(ld.cpu().numpy()/4.0-gt)[8:-8, 8:-140] <= 1).mean())}
	except Exception as e:
		out["pair_D128"] = {"error": repr(e)}
	# tSGM-like ragged ranges around the true disparity (per-pixel [dmin, dmax), 10..48 wide), 3 % invalid pixels
	rng = np.random.RandomState(3)
	base = np.rint(gt).astype(np.int16)
	lo = base-rng.randint(2, 9, gt.shape).astype(np.int16); hi = base+rng.randint(8, 40, gt.shape).astype(np.int16)
	pxr, nr = synth.sgm_pixel_map(w, h, lo, hi, rng.rand(*gt.shape) < 0.03)
	ragged, _ = run(pxr, nr, reps=3)
	ragged["px_d"] = int(nr); ragged["gpxd_per_s"] = nr/ragged["ms_match"]/1e6
	ach = 11.0*nr/(ragged["ms_match"]*1e-3)/1e9
	ragged["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach/peak, "traffic": None}
	out["tsgm_ragged"] = ragged
	m.Release()
	# CPU oracle beside it: a band of 54 rows (48 valid rows) of the same pair, fixed range, single thread (the restatement is scalar)
	try:
		from oracle import oracle as O
		bh = 54
		y0 = (h-bh)//2
		pxb, nb = synth.sgm_pixel_map(w, bh, 0, D)
		t0 = time.perf_counter()
		O.sgm_match(lg[y0:y0+bh], lc[y0:y0+bh], rg[y0:y0+bh], pxb, nb)
		dt = time.perf_counter()-t0
		out["cpu_baseline"] = {"value": nb/dt/1e9, "unit": "G px.d/s", "cores": 1, "kind": "port", "seconds": dt,
			"sample": "oracle SGM (cost + 8 paths + WTA), %dx%d band of the same pair, D=%d, 1 thread" % (w, bh, D)}
	except Exception as e:  # the checker is optional here
		out["cpu_baseline"] = {"error": str(e)}
	return out


def main():
	args = parse()
	w, h = (640, 360) if args.small else (W, H)
	rank = int(os.environ.get("RANK", "0"))
	world = int(os.environ.get("WORLD_SIZE", "1"))
	local_rank = int(os.environ.get("LOCAL_RANK", "0"))
	try:
		threads = len(os.sched_getaffinity(0)) or 1
	except Exception:
		threads = os.cpu_count() or 1
	# a cgroup CPU quota below the affinity size (seen on the GPU boxes: 128 logical CPUs, quota 16) makes more threads than the
	# quota only fight for the same CPU time: the CPU arm uses the quota, and reports it
	try:
		q, per = open("/sys/fs/cgroup/cpu.max").read().split()
		if q != "max":
			threads = max(1, min(threads, int(round(int(q)/int(per)))))
	except Exception:
		pass

	if args.impl == "reference":
		# the reference's own CPU implementation of the path: the oracle port (the reference cannot be compiled in this image,
		# DESIGN.md §3).  Rank 0 only.
		if rank != 0:
			return 0
		scene = build_scene(None if args.small else _maybe_cuda(), w, h)
		band = args.cpu_band or max(24, min(h, int(round(h*0.25*threads/8.0))))
		for _ in range(args.warmup and 1):
			cpu_sample(scene, w, h, 16, threads)
		t_total, px_total, valid = 0.0, 0.0, 0.0
		for _ in range(args.steps):
			mp, dt, desc, valid = cpu_sample(scene, w, h, band, threads)
			t_total += dt; px_total += w*band/1e6
		val = px_total/t_total
		out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps,
			"warmup": args.warmup, "ms_per_step": 1e3*t_total/args.steps, "higher_is_better": True, "scaling": "weak",
			"vs_baseline": None, "dtype": "f32", "data": "synthetic",
			"config": {"workload": "C2: 12x1920x1080, 9 neighbours, PatchMatch 6 iters, single scale (bounded CPU sample per step)", "sample": desc},
			"cpu_baseline": {"value": val, "unit": "Mpix/s", "cores": threads, "kind": "port", "sample": desc, "host": host_info(threads)},
			"e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
		print(json.dumps(out))
		return 0

	import torch
	import torch.distributed as dist
	from openmvs_b200 import multi_gpu
	from openmvs_b200.depth_estimator import OPTDENSE, Camera, ViewData, DepthData, PatchMatchB200

	if not torch.cuda.is_available():
		raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
	torch.cuda.set_device(local_rank)
	dev = torch.device("cuda", local_rank)
	if world > 1:
		dist.init_process_group("nccl", device_id=dev)

	OPTDENSE.nSubResolutionLevels = 0; OPTDENSE.nEstimationGeometricIters = 0
	OPTDENSE.nEstimationIters = ITERS; OPTDENSE.nRandomIters = 6; OPTDENSE.nSweepsPerIter = 0; OPTDENSE.nPropagation = 4
	N_SWEEPS, N_REFINE = OPTDENSE.schedule()
	peaks = {}
	try:
		peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
	except Exception:
		pass
	peak = float(peaks.get("hbm_gbs", 6650.0))

	if args.workload != "c2":
		rc = run_scene_workload(args, dev, rank, world, local_rank, peak)
		if world > 1:
			dist.destroy_process_group()
		return rc

	# distinct images per rank: rank r estimates the 12-view scene with seed 1234 + r
	scene = build_scene(dev, w, h, seed=1234+rank)
	nbrs = [scene.neighbors(r, N_NEIGH) for r in range(N_VIEWS)]
	pm = PatchMatchB200(local_rank)
	cams = [Camera(v.K, v.R, v.C) for v in scene.views]
	# device-resident copies and pinned host copies of the images
	d_imgs = [torch.from_numpy(v.image).to(dev) for v in scene.views]
	h_imgs = []
	for v in scene.views:
		t = torch.empty((h, w), dtype=torch.float32, pin_memory=True)
		t.copy_(torch.from_numpy(v.image))
		h_imgs.append(t.numpy())
	# per-reference-view in/out maps: slices of this rank's preallocated stacks (the gather takes the stacks as they are)
	stack = multi_gpu.ViewStack(N_VIEWS*world, h, w, dev)
	mine = stack.mine                                  # global view ids of this rank; local view r <-> mine[r]
	d_maps = [stack.maps(v) for v in mine]
	pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()
	h_maps = [dict(depth=pin((h, w), torch.float32), normal=pin((h, w, 3), torch.float32), conf=pin((h, w), torch.float32),
		views=pin((h, w, 4), torch.uint8)) for _ in range(N_VIEWS)]
	launches = [0]

	pm2 = PatchMatchB200(local_rank)
	pms = [pm, pm2]
	streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]

	def step_resident():
		# reference views alternate between two contexts on two CUDA streams, so that the ramp-down of one
		# view's kernels overlaps the start of the next view's (same two-context scheme as the e2e path)
		main = torch.cuda.current_stream(dev)
		for st in streams:
			st.wait_stream(main)
		for r in range(N_VIEWS):
			k = r & 1
			with torch.cuda.stream(streams[k]):
				m = d_maps[r]
				m["depth"].zero_(); m["normal"].zero_()  # depth 0 => random initialisation on device
				dd = DepthData([ViewData(d_imgs[r], cams[r])]+[ViewData(d_imgs[i], cams[i]) for i in nbrs[r]], scene.dmin, scene.dmax,
					depthMap=m["depth"], normalMap=m["normal"], confMap=m["conf"], viewsMap=m["views"])
				pms[k].EstimateDepthMap(dd, sync=False)
			launches[0] += 1+1+N_SWEEPS*2+1
		for st in streams:
			main.wait_stream(st)
		if world > 1:
			stack.gather(dst=0)  # final gather of depth+normal+conf of every rank's views on rank 0 (NCCL), no staging copies

	def step_e2e():
		# two contexts used alternately (b200mvs_estimate_async / b200mvs_sync): the H2D/D2H copies of one
		# reference view overlap the kernels of the other, like the reference's two worker threads around the seam
		h2d = d2h = 0
		busy = [False, False]
		for r in range(N_VIEWS):
			k = r & 1
			if busy[k]:
				pms[k].Wait(); h2d += pms[k].stats.bytes_h2d; d2h += pms[k].stats.bytes_d2h
			m = h_maps[r]
			m["depth"][:] = 0  # depth 0 => random initialisation (the normal is ignored then)
			dd = DepthData([ViewData(h_imgs[r], cams[r])]+[ViewData(h_imgs[i], cams[i]) for i in nbrs[r]], scene.dmin, scene.dmax,
				depthMap=m["depth"], normalMap=m["normal"], confMap=m["conf"], viewsMap=m["views"])
			pms[k].EstimateDepthMap(dd, sync=False)
			busy[k] = True
		for k in range(2):
			if busy[k]:
				pms[k].Wait(); h2d += pms[k].stats.bytes_h2d; d2h += pms[k].stats.bytes_d2h
		if world > 1:
			# the hand-over of a multi-GPU run: every rank's maps (host buffers) go back to the device stacks of the previous
			# resident step's layout and are gathered on rank 0 — the collective is part of the end-to-end number
			for r in range(N_VIEWS):
				for key in ("depth", "normal", "conf"):
					d_maps[r][key].copy_(torch.from_numpy(h_maps[r][key]), non_blocking=True)
			stack.gather(dst=0)
		return h2d, d2h

	def timed(fn, steps, warmup):
		for _ in range(warmup):
			fn()
		torch.cuda.synchronize()
		if world > 1: dist.barrier()
		torch.cuda.synchronize()
		e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
		e0.record()
		ret = None
		for _ in range(steps):
			ret = fn()
		e1.record()
		torch.cuda.synchronize()
		if world > 1: dist.barrier()
		ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
		if world > 1: dist.all_reduce(ms, op=dist.ReduceOp.MAX)
		return float(ms.item()), ret

	sampler = ClockSampler(local_rank)
	if rank == 0 and not os.environ.get("BENCH_NO_SMI"): sampler.start()
	launches[0] = 0
	ms_res, _ = timed(step_resident, args.steps, args.warmup)
	n_launch = launches[0]*args.steps//(args.steps+args.warmup)
	clocks = sampler.stop() if rank == 0 else None
	if args.dump_outputs and rank == 0:
		dump_outputs(args.dump_outputs, stack, mine)
	ms_e2e, (h2d, d2h) = timed(step_e2e, args.steps, max(1, args.warmup//3))
	mpix_step = N_VIEWS*w*h/1e6*world
	value = mpix_step/(ms_res/args.steps/1e3)
	e2e = mpix_step/(ms_e2e/args.steps/1e3)

	# ---- roofline of the dominant kernel: one red-black half-sweep, timed live --------------------
	# CUDA events are recorded by the engine around every pm_sweep_kernel launch of one more (untimed)
	# resident EstimateDepthMap call, on the stream the kernels are launched on (b200mvs_stats)
	r = 5
	m = d_maps[r]
	m["depth"].zero_(); m["normal"].zero_()
	dd = DepthData([ViewData(d_imgs[r], cams[r])]+[ViewData(d_imgs[i], cams[i]) for i in nbrs[r]], scene.dmin, scene.dmax,
		depthMap=m["depth"], normalMap=m["normal"], confMap=m["conf"], viewsMap=m["views"])
	pm.EstimateDepthMap(dd, sync=True)
	k_ms = pm.stats.ms_sweep_kernels/max(1, pm.stats.sweep_launches)
	sweep_share = pm.stats.ms_sweep_kernels/max(1e-9, pm.stats.ms_device)
	bytes_launch = w*h*(20+10+4*(N_NEIGH+1))
	achieved = bytes_launch/(k_ms*1e-3)/1e9
	roof = {"kernel": "pm_sweep_kernel<1, 0, 3> (packed taps, photometric, 3 CTAs/SM: one red-black half-sweep)", "bound": "hbm", "achieved": achieved, "peak": peak,
		"unit": "GB/s", "frac": achieved/peak, "traffic": None, "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650",
		"launch_ms": k_ms, "launches_timed": int(pm.stats.sweep_launches), "share_of_step": sweep_share, "algorithmic_bytes_per_launch": bytes_launch,
		"secondary": {"bound": "issue / L1 data pipe (gather stencil, AI ~ 280 flop/B): see the committed ncu capture",
			"hypotheses_per_pixel_and_sweep_upper_bound": 4+N_REFINE}}
	# the honest bound of this kernel is the L1 LSU data pipe / instruction issue: the committed ncu capture of THIS kernel
	# (the file names the kernel it was taken on; the numbers are quoted only when it is the shipped instantiation)
	ncu_file = os.path.join(ROOT, "profiles", "ncu_pm_sweep.txt")
	try:
		lines = open(ncu_file).read().splitlines()
		if lines and "pm_sweep_kernel<1, 0, 3>" in lines[0].replace("(bool)", "").replace("(int)", ""):
			roof["secondary"]["ncu_capture"] = "profiles/ncu_pm_sweep.txt"
			for line in lines:
				if line.startswith("l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed"):
					roof["secondary"]["l1_lsu_data_pipe_pct_of_peak_ncu"] = float(line.split()[1])
				if line.startswith("smsp__issue_active.avg.pct_of_peak_sustained_active"):
					roof["secondary"]["issue_slots_busy_pct_ncu"] = float(line.split()[1])
				if line.startswith("dram__bytes_read.sum"):
					rd = float(line.split()[1])*1e6
				if line.startswith("dram__bytes_write.sum"):
					roof["traffic"] = rd+float(line.split()[1])*1e6
	except Exception:
		pass

	if rank == 0:
		cpu = None
		if not args.no_cpu_baseline:
			band = args.cpu_band or max(24, min(h, int(round(h*0.25*threads/8.0))))
			mp, dt, desc, _ = cpu_sample(scene, w, h, band, threads)
			cpu = {"value": mp, "unit": "Mpix/s", "cores": threads, "kind": "port", "sample": desc, "seconds": dt, "host": host_info(threads)}
		sgm = None
		if world == 1 and not args.no_sgm and not args.small:
			try:
				sgm = sgm_block(dev, peak, threads)
			except Exception as e:
				sgm = {"error": repr(e)}
		out = {"metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
			"ms_per_step": ms_res/args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
			"data": "synthetic",
			"config": {"workload": "C2: 12x1920x1080 synthetic scene, 9 neighbours, PatchMatch 6 iters, single scale" if not args.small else "dev 12x640x360",
				"views_per_gpu_per_step": N_VIEWS, "neighbours": N_NEIGH, "iters": ITERS,
				"schedule": "red-black, %d sweeps for %d reference iterations; per sweep <= 4 propagation candidates (lowest-cost pixel at distance 1/3/5 per direction, unchanged directions skipped) + %d refinement tries" % (N_SWEEPS, ITERS, N_REFINE),
				"parallelism": "per-reference-view shards, %d GPU(s), distinct scene per rank, NCCL gather of the maps (%.2f GB to rank 0 per step)" % (world, (world-1)*stack.bytes_gather()/1e9),
				"l2": "no flush: a step streams %.2f GB of distinct images+maps (> 126 MB L2)" % ((N_VIEWS*w*h*(4+24+20))/1e9)},
			"clocks": clocks,
			"e2e": {"value": e2e, "unit": "Mpix/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e/args.steps,
				"includes_gather": world > 1},
			"gpu_launches": int(n_launch), "roofline": roof, "cpu_baseline": cpu, "sgm": sgm}
		print(json.dumps(out))
	if world > 1:
		dist.destroy_process_group()
	return 0


def run_scene_workload(args, dev, rank, world, local_rank, peak):
	"""c4 / c5: one scene sharded over the ranks (strong scaling), images replicated on every GPU."""
	import torch
	import torch.distributed as dist
	from openmvs_b200 import multi_gpu
	from openmvs_b200.depth_estimator import OPTDENSE, Camera, ViewData, DepthData, PatchMatchB200
	c5 = args.workload == "c5"
	w, h = (4032, 3024) if c5 else (1920, 1080)
	if args.small:
		w, h = w//4, h//4
	n_views = args.views or (50 if c5 else 200)
	n_neigh = N_NEIGH if not c5 else 8
	OPTDENSE.nEstimationGeometricIters = 1 if c5 else 0   # pass 1 keeps with the x1.333 threshold when a geometric pass follows
	# ground truth only for the two views of this rank whose accuracy is reported (200 x 1080p of it would be 6.6 GB of host memory per rank)
	# (two views from the middle of the shard: the corner views of a 200-view camera grid look at the surface so obliquely that part
	# of it leaves the scene's depth range [dmin, dmax], which says nothing about the engine)
	mine_all = multi_gpu.shard_views(n_views, rank, world)
	sampled = mine_all[len(mine_all)//2:len(mine_all)//2+2]
	scene = build_scene(dev, w, h, n_views=n_views, gt_views=set(sampled))
	nbrs = [scene.neighbors(r, n_neigh) for r in range(n_views)]
	cams = [Camera(v.K, v.R, v.C) for v in scene.views]
	imgs = [torch.from_numpy(v.image).to(dev) for v in scene.views]
	scene_gt = None
	stack = multi_gpu.ViewStack(n_views, h, w, dev)
	pms = [PatchMatchB200(local_rank), PatchMatchB200(local_rank)]
	streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
	ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
	coll_ms = []
	T, _ = OPTDENSE.schedule(False); S, _ = OPTDENSE.schedule(True)
	launches = [0]

	def estimate_all(geo):
		main = torch.cuda.current_stream(dev)
		for st in streams:
			st.wait_stream(main)
		for k, v in enumerate(stack.mine):
			with torch.cuda.stream(streams[k & 1]):
				m = stack.maps(v)
				views = [ViewData(imgs[v], cams[v])]
				for i in nbrs[v]:
					vd = ViewData(imgs[i], cams[i])
					if geo >= 0:
						vd.depthMap = stack.depth_of(i); vd.cameraDepthMap = cams[i]
					views.append(vd)
				if geo < 0:
					m["depth"].zero_(); m["normal"].zero_()
				dd = DepthData(views, scene.dmin, scene.dmax, depthMap=m["depth"], normalMap=m["normal"], confMap=m["conf"], viewsMap=m["views"])
				pms[k & 1].EstimateDepthMap(dd, nGeometricIter=geo, sync=False)
			launches[0] += 3+2*(T if geo < 0 else S)
		for st in streams:
			main.wait_stream(st)

	def step():
		estimate_all(-1)
		if c5:
			ev[0].record()
			stack.all_gather_depth()          # the one exchange a geometric pass needs (SceneDensify.cpp:380-394 reloads .dmap files)
			ev[1].record()
			estimate_all(0)
		stack.gather(dst=0)
		if c5:
			torch.cuda.synchronize()
			coll_ms.append(ev[0].elapsed_time(ev[1]))

	for _ in range(args.warmup):
		step()
	torch.cuda.synchronize()
	if world > 1: dist.barrier()
	torch.cuda.synchronize()
	sampler = ClockSampler(local_rank)
	if rank == 0: sampler.start()
	del coll_ms[:]; launches[0] = 0
	e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
	e0.record()
	for _ in range(args.steps):
		step()
	e1.record()
	torch.cuda.synchronize()
	if world > 1: dist.barrier()
	ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
	if world > 1: dist.all_reduce(ms, op=dist.ReduceOp.MAX)
	clocks = sampler.stop() if rank == 0 else None
	if args.dump_outputs and rank == 0:
		dump_outputs(args.dump_outputs, stack, stack.mine)
	ms_step = float(ms.item())/args.steps
	passes = 2 if c5 else 1
	value = n_views*w*h/1e6/(ms_step/1e3)
	# quality of this rank's views against the analytic ground truth (a bench number without it proves nothing)
	acc = []
	for v in sampled:
		gd = stack.maps(v)["depth"].cpu().numpy(); gt = scene.views[v].depth_gt; mm = gd > 0
		# accuracy over the pixels whose true depth lies inside the search range [dmin, dmax) (oblique views of the large camera grid
		# see parts of the surface beyond it; no estimator can return those depths)
		inr = mm & (gt >= scene.dmin) & (gt < scene.dmax)
		acc.append((float(mm.mean()), float((np.abs(gd-gt)[inr]/gt[inr] < 1e-3).mean()), float(inr.sum()/max(1, mm.sum()))))
	if rank == 0:
		cfg = {"workload": ("C5: %d views %dx%d, 8 neighbours, pass 1 (6 iters) + 1 geometric-consistency pass with the depth all-gather" if c5 else
			"C4: %d views %dx%d, 9 neighbours, PatchMatch 6 iters, sharded per reference view") % (n_views, w, h),
			"parallelism": "reference views round-robin over %d GPU(s), images replicated, NCCL gather of the maps to rank 0" % world,
			"views_sampled_valid__within_1e-3_of_ground_truth__fraction_with_true_depth_in_range": acc}
		out = {"metric": "Mpix/sec depth+normal (%dx%d, %d neighbours%s)" % (w, h, n_neigh, ", incl. one geometric pass" if c5 else ""), "value": value, "unit": "Mpix/s",
			"n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
			"vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks, "gpu_launches": int(launches[0]),
			"passes_per_view": passes}
		if c5 and world > 1:
			cm = float(np.median(coll_ms)) if coll_ms else None
			out["collective"] = {"name": "ncclAllGather of the depth-maps before the geometric pass", "ms": cm, "bytes": stack.bytes_all_gather(),
				"GB_per_s": (stack.bytes_all_gather()/1e9/(cm/1e3)) if cm else None}
		print(json.dumps(out))
	return 0


def _maybe_cuda():
	try:
		import torch
		if torch.cuda.is_available():
			return torch.device("cuda", 0)
	except Exception:
		pass
	return None


if __name__ == "__main__":
	sys.exit(main())
