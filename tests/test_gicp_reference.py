"""GICP parity against the REFERENCE ITSELF: fast_gicp's unmodified sources + its own pybind11 module, compiled against
the vendored Eigen and oracle/pcl_shim (oracle/Makefile).  Its results on every case below are stored in
tests/golden/gicp_fastgicp_cases.npz (tests/golden/make_gicp_ref_cases.py), so the comparison needs no build of it.

  * CPU (`-m "not gpu"`): the oracle restatement (oracle/gicp_oracle.cpp) is pinned to the real fast_gicp on C1, on
    the C3 tracker shape (12 416-point frames vs a Gaussian-map target from (q, s), estimated-pose seeding) and on the
    reference's KITTI fixture, and to golden vectors of the real fast_gicp committed under tests/golden/.
  * GPU (`-m gpu`): the CUDA tracker (pygicp drop-in, through the C ABI) against the real fast_gicp on the same cases.
Bars: neighbour indices, squared distances and the float32 rotation/scale exports bit-exact; pose within 1e-6;
final 6x6 normal equations within 1e-9 relative."""
import os

import numpy as np
import pytest

from tests import gicp_cases as cases
from oracle import ref_gicp

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "gicp_fastgicp_ref.npz")
needs_ref = pytest.mark.skipif(not ref_gicp.available(), reason="oracle/_ref/fast_gicp not built (needs the reference tree)")
UNUSED_KW = {"k20": dict(), "k10": dict(k=10), "knn-radius-0.05": dict(max_knn=0.05)}


def _oracle():
    from oracle import gicp_oracle as G

    return G.FastGICP()


def _cuda():
    import pygicp

    return pygicp.FastGICP()


# ------------------------------------------------------------------------------------------------- CPU: oracle pin
def test_oracle_matches_fast_gicp_c1():
    cases.compare_stored(cases.c1(_oracle), "c1")


def test_oracle_matches_fast_gicp_tracker_c3_shape():
    # 100k-Gaussian target keeps the CPU suite short; the GPU test runs the full 300k
    a = cases.tracker_c3(_oracle, P=100000)
    cases.compare_stored(a, "tracker_c3_100000")
    assert np.abs(a["pose3"] - a["gt_last"]).max() < 2e-2


def test_oracle_matches_fast_gicp_kitti():
    a = cases.kitti(_oracle)
    b, _ = cases.compare_stored(a, "kitti")
    pose, rel = b["pose"].astype(np.float64), a["relative"]
    assert np.linalg.norm(pose[:3, 3] - rel[:3, 3]) < 0.05  # the reference's own acceptance bound (gicp_test.cpp:55-56)
    dR = pose[:3, :3] @ rel[:3, :3].T
    assert np.degrees(np.arccos(min(1.0, (np.trace(dR) - 1) / 2))) < 1.0


def test_oracle_matches_fast_gicp_golden():
    """Golden vectors produced by the real fast_gicp build (tests/golden/make_gicp_ref_golden.py): the pin that travels."""
    g = np.load(GOLD)
    a = cases.c1(_oracle, n=4000)
    ref = {k[len("c1_"):]: g[k] for k in g.files if k.startswith("c1_")}
    cases.compare({k: a[k] for k in ref}, ref)
    a = cases.tracker_c3(_oracle, P=20000, frames=(1, 2), keyframe_at=1)
    ref = {k[len("trk_"):]: g[k] for k in g.files if k.startswith("trk_")}
    cases.compare({k: a[k] for k in ref}, ref)


@pytest.mark.parametrize("kw", list(UNUSED_KW.values()), ids=list(UNUSED_KW))
def test_oracle_matches_fast_gicp_on_the_bindings_the_slam_never_calls(kw):
    """withz covariances + z values, set_correspondence_randomness, a finite k-NN radius, get_fitness_score and
    swap_source_and_target (main.cpp:169,172,203,205,228,246-253): the oracle the CUDA path is tested against
    (tests/test_gicp_gpu.py::test_unused_by_slam_bindings_match_oracle) is itself pinned to the real fast_gicp here."""
    name = next(k for k, v in UNUSED_KW.items() if v == kw)
    b = cases.unused_bindings(_oracle, **kw)
    a, gold = cases.stored(f"unused_{name}")
    for k in ("tgt_rots", "tgt_scales_z", "src_rots", "src_scales", "corr", "sqd", "corr_swapped", "sqd_swapped"):
        assert gold.equal(f"unused_{name}/{k}", b[k]) and b[k].dtype.str == str(gold.z[f"unused_{name}/{k}.dtype"]), k
    assert np.array_equal(a["pose"], b["pose"]) and np.array_equal(a["pose_swapped"], b["pose_swapped"])
    assert np.abs(a["H"] - b["H"]).max() <= 1e-12 * np.abs(a["H"]).max()
    # getFitnessScore lives in PCL's Registration base class (here: oracle/pcl_shim): float transform of the cloud, 1-NN
    assert np.allclose(a["fitness"], b["fitness"], rtol=2e-6, atol=0)


def test_oracle_matches_fast_gicp_with_duplicates_and_outliers():
    """Ties (duplicated points in both clouds) and source points with no correspondence within max_corr (-1 rows)."""
    b = cases.duplicates_and_outliers(_oracle)
    a, _ = cases.compare_stored(b, "duplicates")
    assert (b["corr"][:50] == -1).all() and np.array_equal(a["pose"], b["pose"])


@needs_ref
def test_reference_module_is_the_reference():
    """The loaded module is the pybind11 module of main.cpp (its class list), not this repo's drop-in."""
    m = ref_gicp.load()
    assert {"FastGICP", "FastVGICP", "LsqRegistration", "align_points", "downsample"} <= set(dir(m))
    assert ref_gicp.path().startswith(os.path.join(os.path.dirname(HERE), "oracle", "_ref"))
    assert m.FastGICP is not __import__("pygicp").FastGICP


# ------------------------------------------------------------------------------------------------- GPU: product pin
@pytest.mark.gpu
def test_cuda_matches_fast_gicp_c1(cuda):
    a = cases.c1(_cuda)
    cases.compare_stored(a, "c1")
    assert np.abs(a["pose"] - a["T_gt"]).max() < 1e-3


@pytest.mark.gpu
def test_cuda_matches_fast_gicp_tracker_c3(cuda):
    """Full C3 tracker shape: 12 416-point frames against the 300k-Gaussian target."""
    a = cases.tracker_c3(_cuda)
    cases.compare_stored(a, "tracker_c3_300000")
    assert np.abs(a["pose3"] - a["gt_last"]).max() < 2e-2


@pytest.mark.gpu
def test_cuda_matches_fast_gicp_kitti(cuda):
    cases.compare_stored(cases.kitti(_cuda), "kitti")


@pytest.mark.gpu
def test_cuda_matches_fast_gicp_golden(cuda):
    g = np.load(GOLD)
    a = cases.c1(_cuda, n=4000)
    ref = {k[len("c1_"):]: g[k] for k in g.files if k.startswith("c1_")}
    cases.compare({k: a[k] for k in ref}, ref)
