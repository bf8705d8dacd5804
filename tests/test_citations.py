"""Every `path:line` citation of the reference in the sources, headers and docs points at an existing file and line range of
the reference.  The reference's files and their line counts are stored in tests/golden/reference_line_counts.json
(tests/golden/make_reference_goldens.py)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINE_COUNTS = os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")
# full paths (libs/MVS/DepthMap.cpp:465-564) and bare file names (DepthMap.cpp:465-564; resolved through the reference tree)
PAT = re.compile(r"(?<![A-Za-z0-9_/.-])((?:(?:libs|apps|scripts|docs|build)/)?[A-Za-z0-9_./+-]*[A-Za-z0-9_+-]+\.(?:cpp|h|inl|cu|txt|yml))`?:(\d+)(?:-(\d+))?")
OWN = ("pm_kernels.cu", "capi.cu", "sgm_kernels.cu", "filter_kernels.cu", "resize_kernels.cu", "b200mvs.h", "oracle.h", "pm_oracle.cpp",
	"sgm_oracle.cpp", "filter_oracle.cpp", "adapter_main.cpp", "sgm_step_main.cu")


def _files():
	for dp, dn, fn in os.walk(ROOT):
		dn[:] = [d for d in dn if d not in (".git", "gpurun_out", "__pycache__", ".pytest_cache", "profiles")]
		for f in fn:
			if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp", ".md")) and f not in ("SURVEY.md", "PAPERS.md", "SNIPPETS.md"):
				yield os.path.join(dp, f)


def test_reference_citations_resolve():
	lengths = json.load(open(LINE_COUNTS))
	index = {}
	for rel in lengths:
		index.setdefault(os.path.basename(rel), []).append(rel)
	bad = []
	n = 0
	for path in _files():
		for m in PAT.finditer(open(path, errors="replace").read()):
			rel, a, b = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
			if os.path.basename(rel) in OWN:
				continue  # a citation of this repo's own files
			if "/" not in rel:
				cands = index.get(rel, [])
				if len(cands) != 1:
					if not cands: bad.append("%s cites %s: no such file in the reference" % (os.path.relpath(path, ROOT), rel))
					continue  # ambiguous bare names (CMakeLists.txt) are not checked
				rel = cands[0]
			n += 1
			if rel not in lengths or not (1 <= a <= b <= lengths[rel]):
				bad.append("%s cites %s:%d-%d (%s)" % (os.path.relpath(path, ROOT), rel, a, b, "%d lines" % lengths[rel] if rel in lengths else "missing file"))
	assert n > 200
	assert not bad, "\n".join(bad[:20])
