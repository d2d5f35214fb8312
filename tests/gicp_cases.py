"""Call sequences shared by the GICP parity tests.  Every case takes a `make()` factory returning an object with the
pygicp.FastGICP interface (this repo's CUDA drop-in, the CPU oracle, or the reference's own pybind11 module:
oracle/ref_gicp.py) and returns a dict of numpy results to compare.  The reference's results are stored in
tests/golden/gicp_fastgicp_cases.npz (tests/golden/make_gicp_ref_cases.py)."""
import os

import numpy as np

from gs_icp_slam_b200 import synthetic as S
from tests.refdigest import Golden, record

HERE = os.path.dirname(os.path.abspath(__file__))
REF_CASES = os.path.join(HERE, "golden", "gicp_fastgicp_cases.npz")
EXACT = ("corr", "sqd", "tgt_rots", "src_rots", "tgt_scales", "src_scales", "rots_kf", "scales_kf")


def _params(r, max_corr):
    r.set_max_correspondence_distance(max_corr)
    r.set_max_knn_distance(99999)
    return r


def _filter_all(n):
    return np.arange(1, n + 1, dtype=np.int32)


def c1(make, n=10000):
    """BASELINE config C1: two n-point clouds, known SE(3), identity guess; the tracker's calls
    (calculate_target_covariance_with_filter + lazy source covariances inside align)."""
    tgt, src, T = S.gicp_pair(n, n)
    r = _params(make(), 0.05)
    r.set_input_target(tgt)
    r.set_target_filter(len(tgt), _filter_all(len(tgt)))
    r.calculate_target_covariance_with_filter()
    out = dict(T_gt=np.asarray(T), tgt_rots=np.array(r.get_target_rotationsq()), tgt_scales=np.array(r.get_target_scales()))
    r.set_input_source(src)
    r.set_source_filter(len(src), _filter_all(len(src)))
    out["pose"] = np.array(r.align(np.eye(4, dtype=np.float32)))
    c, d = r.get_source_correspondence()
    out.update(corr=np.array(c), sqd=np.array(d), src_rots=np.array(r.get_source_rotationsq()),
               src_scales=np.array(r.get_source_scales()), H=np.array(r.get_final_hessian()))
    return out


def tracker_c3(make, P=300000, frames=(1, 2, 3), keyframe_at=2):
    """BASELINE config C3 tracker shape: 12 416-point frames (97 x 128, mp_Tracker.py:394-413) with the trackable-subset
    filter, registered against a P-Gaussian map target installed through set_target_covariances_fromqs
    (mp_Tracker.py:284-289), seeded with the previous ESTIMATED pose (mp_Tracker.py:199); at `keyframe_at` the source
    rotations/scales are read back and the target is refreshed from (q, s) again."""
    cam = S.TUM
    g = S.gaussian_map(P, 3)
    r = _params(make(), 0.03)
    r.set_input_target(g["means3D"].astype(np.float64))
    r.set_target_covariances_fromqs(g["rotations"].reshape(-1), g["scales"].reshape(-1))
    pose = S.trajectory_pose(frames[0] - 1, 200).astype(np.float32)
    out = {}
    for f in frames:
        pts, tr = S.tracker_cloud(S.raycast_depth(S.trajectory_pose(f, 200), cam)[0], cam)
        r.set_input_source(pts)
        r.set_source_filter(len(tr), S.trackable_filter(len(pts), tr))
        pose = np.array(r.align(pose))
        c, d = r.get_source_correspondence()
        out[f"pose{f}"], out[f"corr{f}"], out[f"sqd{f}"] = pose, np.array(c), np.array(d)
        out[f"H{f}"] = np.array(r.get_final_hessian())
        if f == keyframe_at:
            out["rots_kf"], out["scales_kf"] = np.array(r.get_source_rotationsq()), np.array(r.get_source_scales())
            r.set_input_target(g["means3D"].astype(np.float64))
            r.set_target_covariances_fromqs(g["rotations"].reshape(-1), g["scales"].reshape(-1))
    out["gt_last"] = S.trajectory_pose(frames[-1], 200)
    return out


def kitti(make):
    """The reference's only acceptance fixture (FG/src/test/gicp_test.cpp:147-201): the KITTI pair + relative.txt."""
    k = np.load(os.path.join(HERE, "golden", "gicp_kitti_pair.npz"))
    r = make()
    r.set_max_knn_distance(99999)
    r.set_input_target(k["target"])
    r.set_input_source(k["source"])
    # the lazy source covariances go through calculate_source_covariances_with_filter (fgi:230): without a filter the
    # reference reads an empty vector and an uninitialised count, so the all-trackable filter is set explicitly
    r.set_source_filter(len(k["source"]), _filter_all(len(k["source"])))
    out = dict(pose=np.array(r.align(np.eye(4, dtype=np.float32))), relative=k["relative"])
    c, d = r.get_source_correspondence()
    out.update(corr=np.array(c), sqd=np.array(d), tgt_rots=np.array(r.get_target_rotationsq()),
               src_rots=np.array(r.get_source_rotationsq()), tgt_scales=np.array(r.get_target_scales()),
               src_scales=np.array(r.get_source_scales()), H=np.array(r.get_final_hessian()))
    return out


def compare(a, b, exact_prefixes=EXACT, pose_tol=1e-6, h_rtol=1e-9):
    """Parity bars (BASELINE.json north_star): indices / squared distances / float32 exports bit-exact, pose SE(3)
    within 1e-6, fp64 normal equations within h_rtol of their largest entry."""
    for k in a:
        if k in ("T_gt", "relative", "gt_last"):
            continue
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape and x.dtype == y.dtype, (k, x.shape, y.shape, x.dtype, y.dtype)
        if k.startswith("pose"):
            assert np.abs(x.astype(np.float64) - y.astype(np.float64)).max() <= pose_tol, k
        elif k.startswith("H"):
            assert np.abs(x - y).max() <= h_rtol * np.abs(y).max(), (k, np.abs(x - y).max() / np.abs(y).max())
        elif k.startswith(exact_prefixes):
            assert np.array_equal(x, y), (k, int((x != y).sum()), x.size)
        else:
            raise AssertionError(f"unclassified key {k}")


def unused_bindings(make, n_t=4000, n_s=3000, k=20, max_knn=99999.0):
    """The FastGICP bindings the SLAM scripts never call (FG/src/python/main.cpp:169,172,203,205,228,246-253): z values +
    calculate_target_covariance_withz, set_correspondence_randomness, a finite set_max_knn_distance, get_fitness_score,
    swap_source_and_target."""
    tgt, src, T = S.gicp_pair(n_t, n_s, 40, 41)
    z = np.random.default_rng(5).uniform(0.2, 3.0, size=len(tgt)).astype(np.float32)
    r = _params(make(), 0.05)
    r.set_correspondence_randomness(k)
    r.set_max_knn_distance(max_knn)
    r.set_input_target(tgt)
    r.set_target_z_values(z)
    r.calculate_target_covariance_withz()
    out = dict(tgt_rots=np.array(r.get_target_rotationsq()), tgt_scales_z=np.array(r.get_target_scales()))
    r.set_input_source(src)
    r.set_source_filter(len(src), _filter_all(len(src)))
    out["pose"] = np.array(r.align(np.eye(4, dtype=np.float32)))
    c, d = r.get_source_correspondence()
    out.update(corr=np.array(c), sqd=np.array(d), src_rots=np.array(r.get_source_rotationsq()), src_scales=np.array(r.get_source_scales()),
               H=np.array(r.get_final_hessian()))
    out["fitness"] = np.array([r.get_fitness_score(x) for x in (1e-4, 0.01, 1e9)])
    r.swap_source_and_target()
    # after the swap the former target (with its withz covariances) is the source: the filter must cover it
    r.set_source_filter(len(tgt), _filter_all(len(tgt)))
    r.set_target_filter(len(src), _filter_all(len(src)))
    out["pose_swapped"] = np.array(r.align(np.eye(4, dtype=np.float32)))
    c, d = r.get_source_correspondence()
    out.update(corr_swapped=np.array(c), sqd_swapped=np.array(d))
    return out


def duplicates_and_outliers(make):
    """Duplicated target points (k-NN / 1-NN ties resolved by the lowest index) and 50 source points 40 m outside the target
    (no correspondence within max_corr: -1 rows), through the tracker's call sequence."""
    tgt = S.sample_surface(3000, 30, 0.001)[0]
    tgt[5] = tgt[6]
    tgt[100] = tgt[2000]
    src = S.sample_surface(500, 31, 0.001)[0]
    src[:50] += 40.0
    src[60] = src[61]
    r = _params(make(), 0.1)
    r.set_input_target(tgt)
    r.set_target_filter(len(tgt), _filter_all(len(tgt)))
    r.calculate_target_covariance_with_filter()
    r.set_input_source(src)
    r.set_source_filter(len(src), _filter_all(len(src)))
    out = dict(pose=np.array(r.align(np.eye(4, dtype=np.float32))))
    c, d = r.get_source_correspondence()
    out.update(corr=np.array(c), sqd=np.array(d), tgt_rots=np.array(r.get_target_rotationsq()), tgt_scales=np.array(r.get_target_scales()),
               src_rots=np.array(r.get_source_rotationsq()), src_scales=np.array(r.get_source_scales()), H=np.array(r.get_final_hessian()))
    return out


def store(out, case, res):
    """Adds a case's results to the dict `out`: the bit-exact outputs as records (tests/refdigest.py), the rest in full."""
    for k, v in res.items():
        v = np.asarray(v)
        if k.startswith(EXACT):
            record(out, f"{case}/{k}", v, sample=False)
        else:
            out[f"{case}/{k}"] = v


def stored(case, gold=None):
    """(the fully stored results of `case`, the Golden reader) from tests/golden/gicp_fastgicp_cases.npz."""
    gold = gold or Golden(REF_CASES)
    pre = case + "/"
    return {k[len(pre):]: v for k, v in gold.z.items() if k.startswith(pre) and "." not in k[len(pre):]}, gold


def compare_stored(a, case, gold=None, **kw):
    """compare(a, reference results of `case`): bit-exact outputs through their records, dtype included."""
    full, gold = stored(case, gold)
    compare({k: a[k] for k in a if k in full}, full, **kw)
    for k in a:
        if k in full or k in ("T_gt", "relative", "gt_last"):
            continue
        assert k.startswith(kw.get("exact_prefixes", EXACT)), f"unclassified key {k}"
        x = np.asarray(a[k])
        assert x.dtype.str == str(gold.z[f"{case}/{k}.dtype"]) and gold.equal(f"{case}/{k}", x), k
    return full, gold
