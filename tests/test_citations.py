"""Every `file:line` citation into the reference tree (C-ABI header, oracle, CUDA sources, host mirror, docs) must
point at an existing file and lines inside it.  The reference's file list and line counts are stored in
tests/golden/reference_index.json (tests/golden/make_reference_index.py regenerates it from a bigsnpr checkout)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INDEX = os.path.join(ROOT, "tests", "golden", "reference_index.json")
CITE = re.compile(r"\b((?:src|R|tests/testthat|inst/extdata)/[A-Za-z0-9_./-]+\.(?:cpp|h|R|ld|rds|bed))(?::(\d+)(?:-(\d+))?)?")

FILES = ["include/bsgpu.h", "oracle/bsg_oracle.c", "oracle/ref.py", "bigsnpr_b200/api.py", "bigsnpr_b200/dist.py",
         "r_shim/bigsnpr_shim.c", "INTEGRATION.md", "DESIGN.md"] + [
    os.path.join("bigsnpr_b200/csrc", f) for f in sorted(os.listdir(os.path.join(ROOT, "bigsnpr_b200", "csrc")))
    if f.endswith((".cu", ".cuh"))] + [os.path.join("tests", f) for f in sorted(os.listdir(os.path.join(ROOT, "tests")))
                                        if f.endswith(".py") and f != "test_citations.py"]


def test_reference_citations_resolve():
    nlines = json.load(open(INDEX))["files"]
    bad, total = [], 0
    for rel in FILES:
        text = open(os.path.join(ROOT, rel), errors="replace").read()
        for m in CITE.finditer(text):
            path, a, b = m.group(1), m.group(2), m.group(3)
            total += 1
            if path not in nlines:
                bad.append((rel, m.group(0), "no such file"))
                continue
            if a is None:
                continue
            lo, hi = int(a), int(b or a)
            if not (1 <= lo <= hi <= nlines[path]):
                bad.append((rel, m.group(0), "file has %d lines" % nlines[path]))
    assert total > 200, total
    assert not bad, bad[:20]
