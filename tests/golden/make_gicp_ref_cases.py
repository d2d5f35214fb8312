"""Generates tests/golden/gicp_fastgicp_cases.npz: the REFERENCE's own tracker (fast_gicp's unmodified sources + its
pybind11 module, oracle/_ref/fast_gicp, built by `make -C oracle ref` where the reference tree is present) on every call
sequence of tests/gicp_cases.py that tests/test_gicp_reference.py compares against.  CPU only:
    python tests/golden/make_gicp_ref_cases.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import ref_gicp  # noqa: E402
from tests import gicp_cases as cases  # noqa: E402
from tests.refdigest import save  # noqa: E402
from tests.test_gicp_reference import UNUSED_KW  # noqa: E402


def main():
    make = ref_gicp.FastGICP
    out = {}
    cases.store(out, "c1", cases.c1(make))
    for P in (100000, 300000):
        cases.store(out, f"tracker_c3_{P}", cases.tracker_c3(make, P=P))
    cases.store(out, "kitti", cases.kitti(make))
    for name, kw in UNUSED_KW.items():
        cases.store(out, f"unused_{name}", cases.unused_bindings(make, **kw))
    cases.store(out, "duplicates", cases.duplicates_and_outliers(make))
    save(cases.REF_CASES, out)
    print("wrote", cases.REF_CASES, os.path.getsize(cases.REF_CASES), "bytes")


if __name__ == "__main__":
    main()
