#!/usr/bin/env python
"""Writes tests/golden/ref_results.json: what the UNMODIFIED reference computes for the tests that compare with it through
golden_util.reference() (digests of taps and message lists, small values), so that those tests also run where the
reference was not compiled.  Needs oracle/_ref/libaisref.so (`make -C oracle ref` next to the reference sources).

Run:  python tests/golden/make_ref_results.py
Every such test asks golden_util.reference() before it creates an engine, so this records the GPU tests' cases on a
machine without a GPU too (their engines then fail, which is expected here; only the recorded results are kept).
"""
import json
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS, os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
import __graft_entry__  # noqa: E402
import golden_util as G  # noqa: E402
import oracle as O  # noqa: E402

FILES = ["test_oracle_port_vs_ref.py", "test_egress.py", "test_gpu_matrix.py", "test_gpu_parity.py"]


def main():
    if not O.have_ref():
        sys.exit("oracle/_ref/libaisref.so missing: build it with `make -C oracle ref` next to the reference sources")
    __graft_entry__.build()  # before collection: test_egress.py skips when libaisgpu.so is missing
    G.RECORD = {}
    pytest.main([os.path.join(TESTS, f) for f in FILES] + ["-q", "-p", "no:cacheprovider"])
    with open(G.REF_RESULTS, "w") as f:
        json.dump(G.RECORD, f, indent=1, sort_keys=True)
        f.write("\n")
    print("%d cases -> %s" % (len(G.RECORD), G.REF_RESULTS))


if __name__ == "__main__":
    main()
