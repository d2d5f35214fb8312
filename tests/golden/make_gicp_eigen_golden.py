"""Generates tests/golden/gicp_eigen_calls.npz: the outputs of the reference's vendored Eigen (oracle/_ref/libref_gicp_eigen.so,
built by `make -C oracle ref` where the reference tree is present) for every call the Eigen tests of
tests/test_gicp_oracle.py make, per test and in call order, plus Eigen's linearisation summed over the correspondences of
linearize_case().  The tests run against the real build while recording, so their assertions are checked too.  CPU only:
    python tests/golden/make_gicp_eigen_golden.py"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import test_gicp_oracle as T  # noqa: E402


def main():
    lib = C.CDLL(T.EIG)
    out = {}
    for test in (T.test_svd_and_quaternion_match_eigen, T.test_quaternion_of_reflection_matches_eigen,
                 T.test_ldlt_and_so3_exp_match_eigen, T.test_covariance_pipeline_matches_eigen, T.test_cov_from_qs_quirk_matches_eigen):
        rec = T.EigenRecorder(lib)
        test(rec)
        out.update(rec.arrays(test.__name__ + "/"))
    r, pose, corr, sqd, src, tgt, _ = T.linearize_case()
    H, b, e = T.eigen_linearize(lib, r, pose, corr, src, tgt)
    out.update({"linearize.H": H, "linearize.b": b, "linearize.e": np.float64(e)})
    out = {k: v for k, v in out.items() if v.size}
    np.savez_compressed(T.EIG_CALLS, **out)
    print("wrote", T.EIG_CALLS, os.path.getsize(T.EIG_CALLS), "bytes")


if __name__ == "__main__":
    main()
