"""Generates the two fixtures through which tests compare with the reference (cdcseacave/openMVS) without needing its tree:

  reference_line_counts.json    every .cpp/.h/.inl/.cu/.txt/.yml file of the reference and its number of lines, against which
                                tests/test_citations.py resolves the `path:line` citations of this repository;
  dmap_reference_reader.npz     a .dmap file written by openmvs_b200.dmap_io and what the reference's own Python reader
                                (scripts/python/MvsUtils.py:loadDMAP) read from it, for tests/test_dmap_io.py.

Run from the repository root with the reference checkout as argument:
  python tests/golden/make_reference_goldens.py path/to/openMVS
"""
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
REF = os.path.abspath(sys.argv[1])

counts = {}
for dp, dn, fn in os.walk(REF):
	dn[:] = [d for d in dn if d != ".git"]
	for f in fn:
		if f.endswith((".cpp", ".h", ".inl", ".cu", ".txt", ".yml")):
			full = os.path.join(dp, f)
			counts[os.path.relpath(full, REF)] = sum(1 for _ in open(full, errors="replace"))
with open(os.path.join(HERE, "reference_line_counts.json"), "w") as f:
	json.dump(counts, f, indent=0, sort_keys=True)
	f.write("\n")

sys.path.insert(0, os.path.join(REF, "scripts", "python"))
from MvsUtils import loadDMAP  # noqa: E402
from test_dmap_io import write_reader_case  # noqa: E402

with tempfile.TemporaryDirectory() as tmp:
	p, _ = write_reader_case(tmp)
	d = loadDMAP(p)
	raw = np.frombuffer(open(p, "rb").read(), np.uint8)
keys = ("image_width", "image_height", "depth_width", "depth_height", "depth_min", "depth_max", "reference_view_id", "neighbor_view_ids",
	"K", "R", "C", "depth_map", "normal_map", "confidence_map", "views_map")
np.savez_compressed(os.path.join(HERE, "dmap_reference_reader.npz"), dmap=raw, file_name=np.array(d["file_name"]),
	**{k: np.asarray(d[k]) for k in keys})
print("%d reference files indexed; .dmap of %d bytes read back by loadDMAP" % (len(counts), raw.size))
