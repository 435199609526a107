"""Regenerates tests/golden/reference_index.json from a checkout of the reference (bigsnpr) sources:

    python tests/golden/make_reference_index.py <path to the bigsnpr checkout>

  files         every file under src/, R/, tests/testthat/ and inst/extdata/ that a `file:line` citation can name
                (.cpp .h .R .ld .rds .bed), with its number of lines -- what tests/test_citations.py resolves against
  call_methods  name -> arity of each entry of the reference's R_CallMethodDef table (src/RcppExports.cpp) -- what
                tests/test_abi.py compares the R shim's table with

Only names and counts are stored, no source text, so the tests run without the reference checkout.
"""
import json
import os
import re
import sys

DIRS = ("src", "R", "tests/testthat", "inst/extdata")
EXTS = (".cpp", ".h", ".R", ".ld", ".rds", ".bed")
CALL_DEF = re.compile(r'\{"(_bigsnpr_\w+)",\s*\(DL_FUNC\)\s*&\w+,\s*(\d+)\}')


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    ref = sys.argv[1]
    files = {}
    for d in DIRS:
        for dp, _, fns in os.walk(os.path.join(ref, d)):
            for fn in fns:
                if fn.endswith(EXTS):
                    full = os.path.join(dp, fn)
                    with open(full, "rb") as f:
                        files[os.path.relpath(full, ref)] = sum(1 for _ in f)
    calls = {m.group(1): int(m.group(2))
             for m in CALL_DEF.finditer(open(os.path.join(ref, "src", "RcppExports.cpp")).read())}
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_index.json")
    with open(out, "w") as f:
        json.dump({"files": dict(sorted(files.items())), "call_methods": dict(sorted(calls.items()))}, f, indent=1)
        f.write("\n")
    print("wrote", out, len(files), "files,", len(calls), "call methods")


if __name__ == "__main__":
    sys.exit(main())
