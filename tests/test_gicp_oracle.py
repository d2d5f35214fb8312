"""CPU tests: the GICP oracle (oracle/gicp_oracle.cpp) against
  * the reference's vendored Eigen (oracle/_ref/libref_gicp_eigen.so: JacobiSVD, Quaterniond, inverse, LDLT), through its
    outputs on these inputs stored in tests/golden/gicp_eigen_calls.npz (tests/golden/make_gicp_eigen_golden.py),
  * brute-force numpy k-NN,
  * the committed golden vectors (tests/golden/gicp_*.npz), incl. the reference's own acceptance fixture
    (KITTI pair + relative.txt, bound 0.05 m / 1 deg: submodules/fast_gicp/src/test/gicp_test.cpp:147-201)."""
import ctypes as C
import os

import numpy as np
import pytest

from gs_icp_slam_b200 import synthetic as S
from oracle import gicp_oracle as G

HERE = os.path.dirname(os.path.abspath(__file__))
EIG = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libref_gicp_eigen.so")
EIG_CALLS = os.path.join(HERE, "golden", "gicp_eigen_calls.npz")
# output arguments of the libref_gicp_eigen.so functions the tests call: (argument position, dtype, element count)
EIG_OUT = {"eig_svd3": [(1, "f8", 9), (2, "f8", 3), (3, "f8", 9)], "eig_quat_from_matrix": [(1, "f8", 4)],
           "eig_ldlt_solve6": [(2, "f8", 6)], "eig_so3_exp": [(1, "f8", 9)],
           "eig_cov_pipeline": [(2, "f4", 4), (3, "f4", 3), (4, "f8", 9)], "eig_cov_from_qs": [(2, "f8", 9)]}


class EigenRecorder:
    """Calls the Eigen build and keeps the outputs of every call, in call order (tests/golden/make_gicp_eigen_golden.py)."""

    def __init__(self, lib):
        self.lib, self.calls = lib, {k: [] for k in EIG_OUT}

    def __getattr__(self, name):
        def call(*args):
            getattr(self.lib, name)(*args)
            self.calls[name].append([np.ctypeslib.as_array(C.cast(args[i].value, C.POINTER(C.c_double if t == "f8" else C.c_float)),
                                                           (n,)).copy() for i, t, n in EIG_OUT[name]])
        return call

    def arrays(self, prefix):
        return {f"{prefix}{name}.{i}": np.array([c[j] for c in calls]).reshape(len(calls), n)
                for name, calls in self.calls.items() for j, (i, t, n) in enumerate(EIG_OUT[name])}


class EigenReplay:
    """Stands in for the Eigen build: each call writes the outputs the build produced for the same call of the same test."""

    def __init__(self, arrays, prefix):
        self.arrays, self.next = {k[len(prefix):]: v for k, v in arrays.items() if k.startswith(prefix)}, {k: 0 for k in EIG_OUT}

    def __getattr__(self, name):
        def call(*args):
            k = self.next[name]
            self.next[name] += 1
            for i, t, n in EIG_OUT[name]:
                a = np.ascontiguousarray(self.arrays[f"{name}.{i}"][k], dtype=t)
                C.memmove(args[i].value, a.ctypes.data, a.nbytes)
        return call


@pytest.fixture()
def eig(request):
    return EigenReplay(dict(np.load(EIG_CALLS)), request.function.__name__ + "/")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _sym_psd(rng, n):
    out = []
    for i in range(n):
        A = rng.normal(size=(3, 3)) * 10.0 ** rng.uniform(-4, 1)
        M = A @ A.T
        if i % 7 == 0:  # rank-deficient (planar neighbourhood)
            M = np.outer(A[:, 0], A[:, 0]) + np.outer(A[:, 1], A[:, 1])
        if i % 11 == 0:
            M = np.diag(np.abs(rng.normal(size=3)))
        out.append(M)
    return out


def test_svd_and_quaternion_match_eigen(eig):
    rng = np.random.default_rng(0)
    L = G.lib()
    for M in _sym_psd(rng, 300) + [np.zeros((3, 3)), np.eye(3)]:
        M = np.ascontiguousarray(M)
        U, Sg, V = np.empty((3, 3)), np.empty(3), np.empty((3, 3))
        Ue, Se, Ve = np.empty((3, 3)), np.empty(3), np.empty((3, 3))
        L.go_svd3(_p(M), _p(U), _p(Sg), _p(V))
        eig.eig_svd3(_p(M), _p(Ue), _p(Se), _p(Ve))
        scale = max(np.abs(M).max(), 1e-300)
        assert np.allclose(Sg, Se, rtol=0, atol=1e-13 * scale)
        # U is only unique up to rotations inside (near-)degenerate singular subspaces: compare where it is
        gaps = np.abs(np.diff(Se)) / max(Se[0], 1e-300)
        if gaps.min(initial=1.0) > 1e-6 and Se[2] / max(Se[0], 1e-300) > 1e-9:
            assert np.allclose(U, Ue, atol=1e-9) and np.allclose(V, Ve, atol=1e-9)
            q, qe = np.empty(4), np.empty(4)
            L.go_quat_from_matrix(_p(U), _p(q))
            eig.eig_quat_from_matrix(_p(Ue), _p(qe))
            assert np.allclose(q, qe, atol=1e-9)
        assert np.allclose(U @ np.diag(Sg) @ V.T, M, atol=1e-12 * scale)


def test_quaternion_of_reflection_matches_eigen(eig):
    """det(U) = -1 inputs (column swaps in the SVD): Shoemake's formula applied to a non-rotation."""
    rng = np.random.default_rng(1)
    L = G.lib()
    for _ in range(100):
        Q, _r = np.linalg.qr(rng.normal(size=(3, 3)))
        if np.linalg.det(Q) > 0:
            Q[:, 2] *= -1
        Q = np.ascontiguousarray(Q)
        q, qe = np.empty(4), np.empty(4)
        L.go_quat_from_matrix(_p(Q), _p(q))
        eig.eig_quat_from_matrix(_p(Q), _p(qe))
        assert np.allclose(q, qe, atol=1e-12, equal_nan=True)


def test_ldlt_and_so3_exp_match_eigen(eig):
    rng = np.random.default_rng(2)
    L = G.lib()
    for i in range(100):
        A = rng.normal(size=(6, 8))
        H = np.ascontiguousarray(A @ A.T * 10.0 ** rng.uniform(-2, 4) + (1e-9 if i % 3 else 1.0) * np.eye(6))
        b = rng.normal(size=6)
        x, xe = np.empty(6), np.empty(6)
        L.go_ldlt_solve6(_p(H), _p(b), _p(x))
        eig.eig_ldlt_solve6(_p(H), _p(b), _p(xe))
        assert np.allclose(x, xe, rtol=1e-9, atol=1e-12 * np.abs(xe).max())
    for i in range(100):
        w = rng.normal(size=3) * (1e-6 if i % 4 == 0 else 0.5)
        R, Re = np.empty((3, 3)), np.empty((3, 3))
        L.go_so3_exp(_p(w), _p(R))
        eig.eig_so3_exp(_p(w), _p(Re))
        assert np.allclose(R, Re, atol=1e-15)


def _brute_knn(pts32, k):
    d = ((pts32[:, None, :] - pts32[None, :, :]) ** 2).astype(np.float32)
    d2 = (d[..., 0] + d[..., 1]) + d[..., 2]
    idx = np.lexsort((np.broadcast_to(np.arange(len(pts32)), d2.shape), d2), axis=1)[:, :k]
    return idx, np.take_along_axis(d2, idx, 1)


def test_kdtree_knn_is_exact():
    pts = S.sample_surface(1500, 3, 0.002)[0].astype(np.float32)
    pts[10] = pts[11]  # coincident points: tie broken by index
    idx, d2 = G.knn(pts, 10)
    bidx, bd2 = _brute_knn(pts, 10)
    assert np.array_equal(idx, bidx)
    assert np.array_equal(d2, bd2)


def test_covariance_pipeline_matches_eigen(eig):
    pts = S.sample_surface(800, 4, 0.002)[0]
    r = G.FastGICP()
    r.set_max_knn_distance(99999)
    r.set_input_target(pts)
    r.calculate_target_covariance_with_filter()  # no filter set: every point trackable
    rots, scales, covs = r.get_target_rotationsq().reshape(-1, 4), r.get_target_scales().reshape(-1, 3), r.get_target_covariances()
    p32 = pts.astype(np.float32)
    idx, _ = _brute_knn(p32, 10)
    for i in range(0, 800, 7):
        nb = p32[idx[i]].astype(np.float64)
        c = nb - nb.mean(0)
        Cm = np.ascontiguousarray(c.T @ c / 10.0)
        q, s, out = np.empty(4, np.float32), np.empty(3, np.float32), np.empty((3, 3))
        eig.eig_cov_pipeline(_p(Cm), 0, _p(q), _p(s), _p(out))
        assert np.allclose(scales[i], s, rtol=1e-5)
        assert np.allclose(covs[i], out, rtol=1e-7, atol=1e-9)
        if s[1] > 1e-3 * s[0] and abs(s[0] - s[1]) > 1e-3 * s[0] and abs(s[1] - s[2]) > 1e-3 * s[0]:
            assert np.allclose(rots[i], q, atol=1e-4)


def test_cov_from_qs_quirk_matches_eigen(eig):
    rng = np.random.default_rng(5)
    n = 64
    q = rng.normal(size=(n, 4)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    s = np.exp(rng.normal(-3, 1, size=(n, 3))).astype(np.float32)
    s[0] = [0.01, 0.02, 0.03]  # sv1 < 1e-3 branch
    pts = rng.normal(size=(n, 3))
    r = G.FastGICP()
    r.set_input_target(pts)
    r.set_target_covariances_fromqs(q.flatten(), s.flatten())
    covs = r.get_target_covariances()
    for i in range(n):
        out = np.empty((3, 3))
        eig.eig_cov_from_qs(_p(q[i].copy()), _p(s[i].copy()), _p(out))
        assert np.allclose(covs[i], out, rtol=1e-10, atol=1e-14)


def eigen_linearize(lib, r, pose, corr, src, tgt):
    """Eigen's per-point Mahalanobis matrix and linearisation summed over the correspondences: (H, b, error)."""
    s32, t32 = src.astype(np.float32), tgt.astype(np.float32)
    ca, cb = r.get_source_covariances(), r.get_target_covariances()
    He, be, ee = np.zeros((6, 6)), np.zeros(6), 0.0
    for i in range(len(src)):
        j = corr[i]
        if j < 0:
            continue
        M, Hi, bi, ei = np.empty((3, 3)), np.empty((6, 6)), np.empty(6), C.c_double(0)
        lib.eig_mahalanobis(_p(np.ascontiguousarray(ca[i])), _p(np.ascontiguousarray(cb[j])), _p(pose), _p(M))
        lib.eig_linearize_point(_p(pose), _p(s32[i].copy()), _p(t32[j].copy()), _p(M), _p(Hi), _p(bi), C.byref(ei))
        He += Hi
        be += bi
        ee += ei.value
    return He, be, ee


def linearize_case():
    """The oracle's linearisation on a perturbed pose: (oracle, pose, correspondences, squared distances, source, target)."""
    tgt, src, T = S.gicp_pair(600, 400, 8, 9, 0.002)
    r = G.FastGICP()
    r.set_max_correspondence_distance(0.5)
    r.set_max_knn_distance(99999)
    r.set_input_target(tgt)
    r.calculate_target_covariance_with_filter()
    r.set_input_source(src)
    r.calculate_source_covariance()
    pose = np.ascontiguousarray(T + 1e-3 * np.random.default_rng(1).normal(size=(4, 4)) * np.array([[1, 1, 1, 1]] * 3 + [[0, 0, 0, 0]]))
    H, b, err = r.linearize(pose)
    corr, sqd = r.get_source_correspondence()
    return r, pose, corr, sqd, src, tgt, (H, b, err)


def test_linearize_matches_eigen_per_point():
    r, pose, corr, sqd, src, tgt, (H, b, err) = linearize_case()
    # correspondences: brute force with the same fp32 transform
    Pf = pose.astype(np.float32)
    s32, t32 = src.astype(np.float32), tgt.astype(np.float32)
    # (c0 x + c1 y) + (c2 z + c3): the order Eigen's packet product evaluates trans_f * getVector4fMap() (fgi:260), pinned
    # against the reference build in tests/test_gicp_reference.py
    tp = (Pf[:3, 0] * s32[:, [0]] + Pf[:3, 1] * s32[:, [1]]) + (Pf[:3, 2] * s32[:, [2]] + Pf[:3, 3])
    d = (tp[:, None, :] - t32[None, :, :]).astype(np.float32) ** 2
    d2 = (d[..., 0] + d[..., 1]) + d[..., 2]
    assert np.array_equal(corr, np.where(d2.min(1) < 0.25, d2.argmin(1), -1))
    assert np.array_equal(sqd, d2.min(1))
    He, be, ee = (np.load(EIG_CALLS)[k] for k in ("linearize.H", "linearize.b", "linearize.e"))
    assert np.allclose(H, He, rtol=1e-9, atol=1e-9 * np.abs(He).max())
    assert np.allclose(b, be, rtol=1e-9, atol=1e-9 * np.abs(be).max())
    assert abs(err - ee) <= 1e-9 * abs(ee)
    assert abs(r.compute_error(pose) - err) <= 1e-12 * abs(err)


def test_golden_c1_and_reference_fixture():
    g = np.load(os.path.join(HERE, "golden", "gicp_c1.npz"))
    tgt, src, T = S.gicp_pair(10000, 10000)
    r = G.FastGICP()
    r.set_max_correspondence_distance(0.05)
    r.set_max_knn_distance(99999)
    r.set_input_target(tgt)
    r.calculate_target_covariance_with_filter()
    r.set_input_source(src)
    pose = r.align(np.eye(4))
    assert np.array_equal(pose, g["oracle_pose"])  # deterministic restatement
    assert r.last_iterations == int(g["iterations"])
    corr, sqd = r.get_source_correspondence()
    assert np.array_equal(corr[:512], g["corr_head"]) and np.array_equal(sqd[:512], g["sqd_head"])
    assert np.abs(pose - T).max() < 1e-3  # BASELINE config C1: pose RMSE check against ground truth

    k = np.load(os.path.join(HERE, "golden", "gicp_kitti_pair.npz"))
    r = G.FastGICP()
    r.set_max_knn_distance(99999)
    r.set_input_target(k["target"])
    r.set_input_source(k["source"])
    pose = r.align(np.eye(4)).astype(np.float64)
    rel = k["relative"]
    assert r.has_converged()
    assert np.linalg.norm(pose[:3, 3] - rel[:3, 3]) < 0.05  # gicp_test.cpp:148
    dR = pose[:3, :3] @ rel[:3, :3].T
    assert np.degrees(np.arccos(min(1.0, (np.trace(dR) - 1) / 2))) < 1.0  # gicp_test.cpp:149
    assert np.array_equal(pose.astype(np.float32), k["oracle_pose"])


def test_oracle_withz_swap_fitness():
    """Bindings unused by the SLAM (main.cpp:169,172,228,246-253) restated in the oracle: consistency checks against numpy."""
    from oracle import gicp_oracle as G

    tgt, src, T = S.gicp_pair(1500, 1200)
    z = np.random.default_rng(2).uniform(0.2, 3.0, size=len(tgt)).astype(np.float32)
    a, b = G.FastGICP(), G.FastGICP()
    for r in (a, b):
        r.set_max_correspondence_distance(0.05)
        r.set_max_knn_distance(99999)
        r.set_input_target(tgt)
    a.calculate_target_covariance()
    b.set_target_z_values(z)
    b.calculate_target_covariance_withz()
    zz = np.maximum(1.0, z.astype(np.float64) ** 1.5 * 2.0).astype(np.float32)
    assert np.array_equal(a.get_target_rotationsq(), b.get_target_rotationsq())
    assert np.allclose(b.get_target_scales().reshape(-1, 3), a.get_target_scales().reshape(-1, 3) / zz[:, None], rtol=2e-7, atol=0)
    assert np.array_equal(a.get_target_covariances(), b.get_target_covariances())
    a.set_input_source(src)
    pose = a.align(np.eye(4)).astype(np.float32)
    moved = (src.astype(np.float32) @ pose[:3, :3].T + pose[:3, 3]).astype(np.float32)
    d2 = ((moved[:, None, :].astype(np.float64) - tgt.astype(np.float32)[None].astype(np.float64)) ** 2).sum(-1).min(1)
    for rng in (1e-4, 1e9):
        sel = d2 <= rng
        assert abs(a.get_fitness_score(rng) - d2[sel].mean()) <= 1e-4 * d2[sel].mean()  # the tree measures distances in float32
    assert a.get_fitness_score(-1.0) == np.finfo(np.float64).max
    a.swap_source_and_target()
    assert a.source_size() == len(tgt) and a.target_size() == len(src)
    back = a.align(np.eye(4)).astype(np.float64)
    assert np.abs(back @ pose.astype(np.float64) - np.eye(4)).max() < 5e-3
