"""GPU parity of the GICP tracker: pygicp.FastGICP (CUDA, through the C ABI) vs the CPU oracle
(oracle/gicp_oracle.cpp) on the same seeded inputs.  Bars (BASELINE.json north_star): correspondence
indices and squared distances bit-exact; pose SE(3) within 1e-6; fp64 quantities to 1e-10 relative."""
import os

import numpy as np
import pytest

from gs_icp_slam_b200 import synthetic as S

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _pair(n_t, n_s, **kw):
    import pygicp
    from oracle import gicp_oracle as G

    tgt, src, T = S.gicp_pair(n_t, n_s, **kw)
    regs = []
    for cls in (pygicp.FastGICP, G.FastGICP):
        r = cls()
        r.set_max_correspondence_distance(0.05)
        r.set_max_knn_distance(99999)
        regs.append(r)
    return tgt, src, T, regs[0], regs[1]


def _close(a, b, rtol=1e-10):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() <= rtol * max(np.abs(b).max(), 1e-300)


def test_c1_align_matches_oracle(cuda):
    """BASELINE config C1: two 10k-point clouds, known SE(3)."""
    tgt, src, T, g, o = _pair(10000, 10000)
    for r in (g, o):
        r.set_input_target(tgt)
        r.calculate_target_covariance_with_filter()
    assert np.array_equal(g.get_target_rotationsq(), o.get_target_rotationsq())
    assert np.array_equal(g.get_target_scales(), o.get_target_scales())
    assert _close(g.get_target_covariances(), o.get_target_covariances(), 1e-12)
    for r in (g, o):
        r.set_input_source(src)
    pg, po = g.align(np.eye(4)), o.align(np.eye(4))
    assert g.last_iterations == o.last_iterations
    assert g.has_converged() and o.has_converged()
    assert np.abs(pg.astype(np.float64) - po).max() <= 1e-6
    assert np.abs(pg - T).max() < 1e-3
    cg, dg = g.get_source_correspondence()
    co, do = o.get_source_correspondence()
    assert cg.dtype == np.int32 and dg.dtype == np.float32 and pg.dtype == np.float32
    assert np.array_equal(cg, co)
    assert np.array_equal(dg, do)
    assert np.array_equal(g.get_source_rotationsq(), o.get_source_rotationsq())
    assert np.array_equal(g.get_source_scales(), o.get_source_scales())
    gold = np.load(os.path.join(HERE, "golden", "gicp_c1.npz"))
    assert np.abs(pg.astype(np.float64) - gold["oracle_pose"]).max() <= 1e-6
    assert np.array_equal(cg[:512], gold["corr_head"])


def test_linearize_and_error_match_oracle(cuda):
    tgt, src, T, g, o = _pair(20000, 5000, seed_t=20, seed_s=21)
    pose = np.array(T)
    pose[:3, 3] += [0.004, -0.003, 0.002]
    for r in (g, o):
        r.set_input_target(tgt)
        r.calculate_target_covariance()
        r.set_input_source(src)
        r.calculate_source_covariance()
    Hg, bg, eg = g.linearize(pose)
    Ho, bo, eo = o.linearize(pose)
    assert _close(Hg, Ho, 1e-10) and _close(bg, bo, 1e-10) and abs(eg - eo) <= 1e-10 * abs(eo)
    assert np.allclose(Hg, Hg.T)
    pose2 = np.array(pose)
    pose2[:3, 3] += 1e-3
    assert abs(g.compute_error(pose2) - o.compute_error(pose2)) <= 1e-10 * abs(o.compute_error(pose2))
    cg, dg = g.get_source_correspondence()
    co, do = o.get_source_correspondence()
    assert np.array_equal(cg, co) and np.array_equal(dg, do)
    assert (cg < 0).any() and (cg >= 0).any()  # both matched and rejected points are exercised


def test_tracker_call_sequence(cuda):
    """The exact call sequence of mp_Tracker.py:157-167,191-199,231,256-263,287-288 on synthetic RGB-D frames."""
    import pygicp
    from oracle import gicp_oracle as G

    cam = S.TUM
    poses = [S.trajectory_pose(i, 200) for i in range(3)]
    clouds = [S.tracker_cloud(S.raycast_depth(p, cam)[0], cam) for p in poses]
    regs = [pygicp.FastGICP(), G.FastGICP()]
    out = []
    for r in regs:
        r.set_max_correspondence_distance(0.03)
        r.set_max_knn_distance(99999)
        pts0, tr0 = clouds[0]
        world0 = pts0 @ poses[0][:3, :3].T + poses[0][:3, 3]
        r.set_input_target(world0)
        r.set_target_filter(len(tr0), S.trackable_filter(len(pts0), tr0))
        r.calculate_target_covariance_with_filter()
        rots0, scales0 = r.get_target_rotationsq(), r.get_target_scales()
        res = dict(rots0=rots0, scales0=scales0)
        pose = poses[0].astype(np.float32)
        for f in (1, 2):
            pts, tr = clouds[f]
            r.set_input_source(pts)
            r.set_source_filter(len(tr), S.trackable_filter(len(pts), tr))
            pose = r.align(pose)
            corr, sqd = r.get_source_correspondence()
            res[f"pose{f}"], res[f"corr{f}"], res[f"sqd{f}"] = pose, corr, sqd
            res[f"rots{f}"], res[f"scales{f}"] = r.get_source_rotationsq(), r.get_source_scales()
            if f == 1:  # tracking keyframe: new target = all points so far, covariances from (q, s)
                world1 = pts @ pose[:3, :3].astype(np.float64).T + pose[:3, 3].astype(np.float64)
                tgt_pts = np.concatenate([world0, world1])
                q = np.concatenate([rots0.reshape(-1, 4), res["rots1"].reshape(-1, 4)])
                s = np.concatenate([scales0.reshape(-1, 3), res["scales1"].reshape(-1, 3)])
                r.set_input_target(tgt_pts)
                r.set_target_covariances_fromqs(q.flatten(), s.flatten())
        out.append(res)
    g, o = out
    assert len(g["rots0"]) == 4 * 12416 and len(g["scales0"]) == 3 * 12416
    for k in g:
        if k.startswith("pose"):
            assert np.abs(g[k].astype(np.float64) - o[k]).max() <= 1e-6, k
        else:
            assert np.array_equal(g[k], o[k]), k
    # tracking accuracy against the synthetic ground truth
    assert np.abs(g["pose2"] - poses[2]).max() < 1e-2


def test_reference_fixture_kitti_pair(cuda):
    import pygicp

    k = np.load(os.path.join(HERE, "golden", "gicp_kitti_pair.npz"))
    r = pygicp.FastGICP()
    r.set_max_knn_distance(99999)
    r.set_input_target(k["target"])
    r.set_input_source(k["source"])
    pose = r.align(np.eye(4)).astype(np.float64)
    rel = k["relative"]
    assert r.has_converged()
    assert np.linalg.norm(pose[:3, 3] - rel[:3, 3]) < 0.05
    dR = pose[:3, :3] @ rel[:3, :3].T
    assert np.degrees(np.arccos(min(1.0, (np.trace(dR) - 1) / 2))) < 1.0
    assert np.abs(pose - k["oracle_pose"]).max() <= 1e-6


def test_unused_by_slam_bindings_match_oracle(cuda):
    """The FastGICP bindings the SLAM scripts never call (main.cpp:169,172,228,246-253): withz covariances, z values,
    swap_source_and_target, get_fitness_score."""
    tgt, src, T, g, o = _pair(4000, 3000)
    z = np.random.default_rng(5).uniform(0.2, 3.0, size=len(tgt)).astype(np.float32)
    for r in (g, o):
        r.set_input_target(tgt)
        r.set_target_z_values(z)
        r.calculate_target_covariance_withz()
    assert np.array_equal(g.get_target_rotationsq(), o.get_target_rotationsq())
    sg, so = g.get_target_scales(), o.get_target_scales()
    assert np.allclose(sg, so, rtol=2e-7, atol=0)  # pow() may differ in the last place between libm and the device
    assert _close(g.get_target_covariances(), o.get_target_covariances(), 1e-12)
    for r in (g, o):
        r.set_input_source(src)
    pg, po = g.align(np.eye(4)), o.align(np.eye(4))
    assert np.abs(pg.astype(np.float64) - po).max() <= 1e-6
    for rng in (1e-4, 0.01, 1e9):
        fg, fo = g.get_fitness_score(rng), o.get_fitness_score(rng)
        assert abs(fg - fo) <= 1e-12 * max(abs(fo), 1e-300), (rng, fg, fo)
    assert g.get_fitness_score(-1.0) == o.get_fitness_score(-1.0) == np.finfo(np.float64).max
    # swapped roles: the inverse registration (covariances travel with their clouds)
    for r in (g, o):
        r.swap_source_and_target()
    assert g.source_size() == o.source_size() == len(tgt) and g.target_size() == o.target_size()
    pg2, po2 = g.align(np.eye(4)), o.align(np.eye(4))
    assert np.abs(pg2.astype(np.float64) - po2).max() <= 1e-6
    assert np.abs(pg2.astype(np.float64) @ pg.astype(np.float64) - np.eye(4)).max() < 5e-3
    cg, dg = g.get_source_correspondence()
    co, do = o.get_source_correspondence()
    assert np.array_equal(cg, co) and np.array_equal(dg, do)
    # withz without z values: an error, not an out-of-bounds read
    import pygicp

    r = pygicp.FastGICP()
    r.set_input_target(tgt)
    with pytest.raises(RuntimeError):
        r.calculate_target_covariance_withz()


def test_edge_cases(cuda):
    import pygicp
    from gs_icp_slam_b200._lib import GsicpError
    from oracle import gicp_oracle as G

    r = pygicp.FastGICP()
    with pytest.raises(GsicpError):
        r.align(np.eye(4))  # no clouds (pcl::Registration::align refuses without a target)
    # queries far outside the target (linear-scan fallback) and duplicated points (ties by index)
    tgt = S.sample_surface(3000, 30, 0.001)[0]
    tgt[5] = tgt[6]
    src = S.sample_surface(500, 31, 0.001)[0]
    src[:50] += 40.0
    res = []
    for cls in (pygicp.FastGICP, G.FastGICP):
        q = cls()
        q.set_max_correspondence_distance(0.1)
        q.set_max_knn_distance(99999)
        q.set_input_target(tgt)
        q.calculate_target_covariance()
        q.set_input_source(src)
        q.calculate_source_covariance()
        q.linearize(np.eye(4))
        res.append(q.get_source_correspondence())
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    assert (res[0][0][:50] == -1).all()
    # qs size mismatch: message + early return like the reference (main.cpp:241), no exception
    r = pygicp.FastGICP()
    r.set_input_target(tgt)
    r.set_target_covariances_fromqs(np.zeros(8, np.float32), np.zeros(9, np.float32))
    # pickling builds a fresh object (main.cpp:183-201)
    import pickle

    r2 = pickle.loads(pickle.dumps(r))
    assert isinstance(r2, pygicp.FastGICP) and r2.get_source_rotationsq().size == 0


def test_dist2_matches_bruteforce_and_reference(cuda):
    import torch
    from simple_knn._C import distCUDA2

    pts = S.sample_surface(4000, 40, 0.003)[0].astype(np.float32)
    pts[7] = pts[8]
    out = distCUDA2(torch.from_numpy(pts).to(cuda)).cpu().numpy()
    d = ((pts[:, None, :].astype(np.float64) - pts[None, :, :]) ** 2).sum(-1)
    np.fill_diagonal(d, np.inf)
    ref = np.sort(d, axis=1)[:, :3].mean(1)
    assert np.allclose(out, ref, rtol=2e-5, atol=1e-12)
    # against the reference's simple-knn on 200k points, through its recorded output (tests/golden/raster_ref_records.npz)
    from tests.refdigest import RASTER_RECORDS, Golden

    big = torch.from_numpy(S.sample_surface(200000, 41, 0.002)[0].astype(np.float32)).to(cuda)
    a, b, _ = Golden(RASTER_RECORDS).sample("dist2_200000/dist2", distCUDA2(big))
    assert np.allclose(a, b, rtol=2e-5, atol=1e-12)
    assert torch.isinf(distCUDA2(torch.zeros((2, 3), device=cuda))).all()  # fewer than 3 neighbours -> inf, like FLT_MAX sums


def test_device_lm_loop_matches_host_driven_loop(cuda):
    """align() runs the whole LM loop in one persistent kernel (align_lm_kernel); the host-driven loop (one launch + one
    wait per linearize / compute_error) is kept as the A-B reference: same iteration counts, poses to 1e-12, identical
    correspondences, final Hessian to 1e-12 relative — on C1 and on the tracker sequence shape."""
    import pygicp

    tgt, src, T = S.gicp_pair(10000, 10000)
    out = []
    for host in (False, True):
        r = pygicp.FastGICP()
        r.set_host_lm(host)
        r.set_max_correspondence_distance(0.05)
        r.set_max_knn_distance(99999)
        r.set_input_target(tgt)
        r.calculate_target_covariance_with_filter()
        res = []
        for guess in (np.eye(4), np.array(T) + 1e-3):
            r.set_input_source(src)
            p = r.align(guess.astype(np.float32))
            c, d = r.get_source_correspondence()
            res.append((p, r.last_iterations, r.has_converged(), c, d, r.get_final_hessian()))
        out.append(res)
    for a, b in zip(*out):
        assert a[1] == b[1] and a[2] == b[2]
        assert np.abs(a[0].astype(np.float64) - b[0]).max() <= 1e-12
        assert np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4])
        assert np.abs(a[5] - b[5]).max() <= 1e-12 * np.abs(b[5]).max()


def test_device_lm_loop_rejected_steps_and_iteration_cap(cuda):
    """A poor initial guess exercises rejected LM trials (lambda growth) and a capped iteration count, on both loops."""
    import pygicp

    tgt, src, T = S.gicp_pair(6000, 5000, 30, 31)
    bad = np.array(T)
    bad[:3, 3] += [0.12, -0.1, 0.08]
    out = []
    for host in (False, True):
        r = pygicp.FastGICP()
        r.set_host_lm(host)
        r.set_max_correspondence_distance(0.3)
        r.set_max_knn_distance(99999)
        r.set_max_iterations(7)
        r.set_input_target(tgt)
        r.calculate_target_covariance()
        r.set_input_source(src)
        p = r.align(bad.astype(np.float32))
        out.append((p, r.last_iterations, r.has_converged()))
    assert out[0][1] == out[1][1] and out[0][2] == out[1][2]
    assert np.abs(out[0][0].astype(np.float64) - out[1][0]).max() <= 1e-10
