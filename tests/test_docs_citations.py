"""CPU: every `path:line[-line]` citation of the reference in the C ABI header, the C++ mirror, DESIGN.md and INTEGRATION.md names a
file that exists in the reference tree and a line range inside it.  The tree's source files and their line counts are committed
(tests/golden/reference_files.json, written by tests/golden/make_golden.py --only-files)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILES = os.path.join(ROOT, "tests", "golden", "reference_files.json")
DOCS = ["include/nvbio_b200.h", "DESIGN.md", "INTEGRATION.md", "oracle/nvb_oracle.c", "oracle/ref_shim.cpp",
        "oracle/ref_cuda_bench.cu", "oracle/orc.py", "oracle/cpu_pipeline.py",
        "nvbio_b200/csrc/common.cuh", "nvbio_b200/csrc/fm_core.cuh", "nvbio_b200/csrc/fm_kernels.cu", "nvbio_b200/csrc/gotoh_core.cuh",
        "nvbio_b200/csrc/gotoh_full_core.cuh", "nvbio_b200/csrc/gotoh_kernels.cu", "nvbio_b200/csrc/sa_build.cu", "nvbio_b200/csrc/pipeline.cu",
        "nvbio_b200/fmindex.py", "nvbio_b200/aln.py", "nvbio_b200/pipeline.py", "nvbio_b200/strings.py", "nvbio_b200/io.py", "nvbio_b200/dist.py",
        "bench.py", "README.md", "profiles/README.md"]
CITE = re.compile(r"([A-Za-z0-9_\-./]+\.(?:h|cu|cpp|cuh|cmake|md|txt)):(\d+)(?:-(\d+))?")


def test_reference_citations_resolve():
    with open(FILES) as f:
        n_lines = json.load(f)                                  # path in the reference tree -> number of lines
    idx = {}
    for p in n_lines:
        idx.setdefault(os.path.basename(p), []).append(p)
    bad, checked = [], 0
    for doc in DOCS:
        text = open(os.path.join(ROOT, doc), errors="ignore").read()
        for m in CITE.finditer(text):
            path, lo, hi = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            base = os.path.basename(path)
            if base not in idx:
                if path.startswith(("tests/", "profiles/", "nvbio_b200/", "oracle/", "tools/", "include/")):
                    continue                                  # a citation of this repo, not of the reference
                bad.append((doc, m.group(0), "no such file in the reference")); continue
            cands = [p for p in idx[base] if p.endswith(path)] or idx[base]
            ok = False
            for p in cands:
                if lo <= hi <= n_lines[p]:
                    ok = True
            checked += 1
            if not ok:
                bad.append((doc, m.group(0), "line range outside the file"))
    assert checked > 100
    assert not bad, bad[:20]
