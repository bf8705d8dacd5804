""".dmap writer/reader: byte layout of HeaderDepthDataRaw (libs/MVS/Interface.h:773-792), round trip,
and our files as the reference's own Python reader scripts/python/MvsUtils.py:loadDMAP read them (stored fixture)."""
import os
import struct

import numpy as np
import pytest

from openmvs_b200 import dmap_io


def _sample(rng, h=12, w=17):
	depth = rng.rand(h, w).astype(np.float32)*5+1; depth[rng.rand(h, w) < 0.2] = 0
	normal = rng.randn(h, w, 3).astype(np.float32)
	conf = rng.rand(h, w).astype(np.float32)
	views = rng.randint(0, 255, (h, w, 4)).astype(np.uint8)
	K = np.array([[500.0, 0, 8.0], [0, 500.0, 5.5], [0, 0, 1]]); R = np.linalg.qr(rng.randn(3, 3))[0]; C = rng.randn(3)
	return depth, normal, conf, views, K, R, C


def test_byte_layout_and_round_trip(tmp_path):
	rng = np.random.RandomState(0)
	depth, normal, conf, views, K, R, C = _sample(rng)
	p = str(tmp_path/"depth0000.dmap")
	assert dmap_io.ExportDepthDataRaw(p, str(tmp_path/"images"/"00000.jpg"), [3, 1, 4], (34, 24), K, R, C, 0.5, 9.5, depth, normal, conf, views)
	raw = open(p, "rb").read()
	# HeaderDepthDataRaw: u16 name 'DR', u8 type, u8 padding, 4 x u32, 2 x f32 = 28 bytes
	assert raw[:2] == b"DR" and raw[2] == 15 and raw[3] == 0
	assert struct.unpack("<IIIIff", raw[4:28]) == (34, 24, 17, 12, 0.5, 9.5)
	n, = struct.unpack("<H", raw[28:30]); assert raw[30:30+n] == b"images/00000.jpg"
	o = 30+n
	assert struct.unpack("<IIII", raw[o:o+16]) == (3, 3, 1, 4)
	o += 16
	assert np.array_equal(np.frombuffer(raw[o:o+72], np.float64), K.ravel()); o += 72+72+24
	assert np.array_equal(np.frombuffer(raw[o:o+4*12*17], np.float32), depth.ravel())
	assert len(raw) == o+12*17*(4+12+4+4)
	d = dmap_io.ImportDepthDataRaw(p)
	assert np.array_equal(d["depthMap"], depth) and np.array_equal(d["normalMap"], normal) and np.array_equal(d["confMap"], conf) and np.array_equal(d["viewsMap"], views)
	assert d["imageSize"] == (34, 24) and list(d["IDs"]) == [3, 1, 4] and np.array_equal(d["R"], R) and d["dMin"] == 0.5
	# optional maps and the flags argument
	dmap_io.ExportDepthDataRaw(p, str(tmp_path/"x.jpg"), [0, 1], (17, 12), K, R, C, 1, 2, depth, confMap=conf)
	d = dmap_io.ImportDepthDataRaw(p)
	assert d["normalMap"] is None and d["viewsMap"] is None and np.array_equal(d["confMap"], conf)
	assert dmap_io.ImportDepthDataRaw(p, flags=1)["confMap"] is None
	with pytest.raises(ValueError):
		dmap_io.ExportDepthDataRaw(p, "x.jpg", [0], (17, 12), K, R, C, 1, 2, depth)


def write_reader_case(directory):
	"""The file whose reading by the reference's reader is stored in tests/golden/dmap_reference_reader.npz."""
	rng = np.random.RandomState(1)
	depth, normal, conf, views, K, R, C = _sample(rng)
	p = os.path.join(str(directory), "depth0001.dmap")
	dmap_io.ExportDepthDataRaw(p, os.path.join(str(directory), "img.jpg"), [7, 2, 5, 9], (17, 12), K, R, C, 0.25, 7.5, depth, normal, conf, views)
	return p, (depth, normal, conf, views, K, R, C)


def test_reference_reader_reads_our_files(tmp_path):
	"""What the writer produces, read by the reference's own reader MvsUtils.py:loadDMAP (scripts/python of the reference).  The
	reader's result on this file is stored in tests/golden/dmap_reference_reader.npz (tests/golden/make_reference_goldens.py):
	the writer must still produce that file byte for byte, and what the reader read from it must be what was written."""
	p, (depth, normal, conf, views, K, R, C) = write_reader_case(tmp_path)
	d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dmap_reference_reader.npz"))
	assert open(p, "rb").read() == d["dmap"].tobytes()
	assert d["depth_width"] == 17 and d["depth_height"] == 12 and d["reference_view_id"] == 7 and list(d["neighbor_view_ids"]) == [2, 5, 9]
	assert np.array_equal(d["depth_map"], depth) and np.array_equal(d["normal_map"], normal)
	assert np.array_equal(d["confidence_map"], conf) and np.array_equal(d["views_map"], views)
	assert np.array_equal(d["K"], K) and np.array_equal(d["R"], R) and np.array_equal(d["C"], C)
	assert d["depth_min"] == np.float32(0.25) and d["file_name"] == "img.jpg"


def test_async_writer_host_arrays_and_errors(tmp_path):
	"""AsyncDepthDataWriter: files submitted from host arrays equal the synchronous writer's byte for byte, the queue is bounded,
	an unwritable path surfaces in flush()."""
	rng = np.random.RandomState(1)
	samples = [_sample(rng) for _ in range(7)]
	with dmap_io.AsyncDepthDataWriter(max_pending=2) as wr:
		for i, (depth, normal, conf, views, K, R, C) in enumerate(samples):
			wr.submit(str(tmp_path/("a%02d.dmap" % i)), str(tmp_path/"img.jpg"), [i, i+1], (17, 12), K, R, C, 0.5, 9.5, depth, normal, conf, views)
			depth[:] = -1   # submit() snapshots host arrays: reuse is allowed at once
		wr.flush()
		assert wr.files_written == 7
	rng = np.random.RandomState(1)
	for i in range(7):
		depth, normal, conf, views, K, R, C = _sample(rng)
		d = dmap_io.ImportDepthDataRaw(str(tmp_path/("a%02d.dmap" % i)))
		assert np.array_equal(d["depthMap"], depth) and np.array_equal(d["normalMap"], normal) and np.array_equal(d["viewsMap"], views) and list(d["IDs"]) == [i, i+1]
	wr = dmap_io.AsyncDepthDataWriter()
	depth, normal, conf, views, K, R, C = samples[0]
	wr.submit(str(tmp_path/"no_such_dir"/"x.dmap"), "img.jpg", [0, 1], (17, 12), K, R, C, 1, 2, depth)
	with pytest.raises(RuntimeError):
		wr.flush()
	wr.close()


@pytest.mark.gpu
def test_async_writer_device_maps_overlap_and_equal_sync(tmp_path):
	"""Device-resident maps: submit() returns before the file exists, later writes to the same tensors on the producing stream
	do not leak into the file, and the file equals the synchronous export of the maps as they were at submit time."""
	import torch
	if not torch.cuda.is_available():
		pytest.skip("no CUDA device")
	rng = np.random.RandomState(2)
	h, w = 1080, 1920
	depth = torch.from_numpy((rng.rand(h, w).astype(np.float32)*5+1)).cuda()
	normal = torch.from_numpy(rng.randn(h, w, 3).astype(np.float32)).cuda()
	conf = torch.from_numpy(rng.rand(h, w).astype(np.float32)).cuda()
	views = torch.from_numpy(rng.randint(0, 255, (h, w, 4)).astype(np.uint8)).cuda()
	K = np.array([[1700.0, 0, 959.5], [0, 1700.0, 539.5], [0, 0, 1]]); R = np.eye(3); C = np.zeros(3)
	want = [t.cpu().numpy().copy() for t in (depth, normal, conf, views)]
	with dmap_io.AsyncDepthDataWriter(max_pending=3) as wr:
		for i in range(3):
			wr.submit(str(tmp_path/("d%d.dmap" % i)), str(tmp_path/"img.jpg"), [0, 1, 2], (w, h), K, R, C, 0.5, 9.5, depth, normal, conf, views)
		# overwrite on the producing stream right after the submits: ordered after the copies
		depth.zero_(); normal.zero_()
		wr.flush()
	for i in range(3):
		d = dmap_io.ImportDepthDataRaw(str(tmp_path/("d%d.dmap" % i)))
		assert np.array_equal(d["depthMap"], want[0]) and np.array_equal(d["normalMap"], want[1])
		assert np.array_equal(d["confMap"], want[2]) and np.array_equal(d["viewsMap"], want[3])
