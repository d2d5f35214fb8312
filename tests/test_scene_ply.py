"""N4 (SURVEY.md §8f): scene.ply written by gs_icp_slam_b200.map_table — byte layout, round trip, and byte-for-byte equality
with the reference's own GaussianModel.save_ply (scene/gaussian_model.py:619-636, imported unmodified from the installed copy
under oracle/_ref/gs_icp_slam; the `plyfile` package it calls is absent from this image and replaced by oracle/stubs/plyfile.py,
which only serialises the structured array the reference hands it).  The reference's output is stored as its size and SHA-256
in tests/golden/scene_ply_ref.json (tests/golden/make_scene_ply_golden.py)."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SLAM = os.path.join(ROOT, "oracle", "_ref", "gs_icp_slam")
GOLD = os.path.join(ROOT, "tests", "golden", "scene_ply_ref.json")


def _params(n, degree, seed=0):
    g = torch.Generator().manual_seed(seed)
    m = (degree + 1) ** 2
    r = lambda *s: torch.randn(*s, generator=g)
    return dict(xyz=r(n, 3), features_dc=r(n, 1, 3), features_rest=r(n, m - 1, 3), opacity=r(n, 1), scaling=r(n, 3), rotation=r(n, 4))


@pytest.mark.parametrize("n,degree", [(0, 0), (1, 0), (257, 0), (100, 3)])
def test_layout_and_round_trip(tmp_path, n, degree):
    from gs_icp_slam_b200.map_table import ply_attribute_names, read_scene_ply, write_scene_ply

    p = _params(n, degree)
    path = str(tmp_path / "sub" / "scene.ply")
    assert write_scene_ply(path, **p) == n
    blob = open(path, "rb").read()
    m = (degree + 1) ** 2
    names = ply_attribute_names(3, 3 * (m - 1))
    assert names[:6] == ["x", "y", "z", "nx", "ny", "nz"] and names[-8:] == ["opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3"]
    head = "ply\nformat binary_little_endian 1.0\nelement vertex %d\n" % n + "".join(f"property float {a}\n" for a in names) + "end_header\n"
    assert blob.startswith(head.encode())
    body = np.frombuffer(blob[len(head):], dtype="<f4").reshape(n, len(names))
    assert body.shape[1] == 17 + 3 * (m - 1) - 3 + 3
    if n:
        assert np.array_equal(body[:, :3], p["xyz"].numpy()) and not body[:, 3:6].any()
        # features are stored channel-major: f_rest_k = features_rest[:, k % (m-1), k // (m-1)]
        if m > 1:
            k = 5
            assert np.array_equal(body[:, 9 + k], p["features_rest"][:, k % (m - 1), k // (m - 1)].numpy())
    back = read_scene_ply(path, degree)
    for a, b in (("xyz", "xyz"), ("f_dc", "features_dc"), ("f_rest", "features_rest"), ("opacity", "opacity"), ("scaling", "scaling"),
                 ("rotation", "rotation")):
        assert back[a].shape == p[b].shape and torch.equal(back[a], p[b]), a
    with pytest.raises(ValueError):
        read_scene_ply(path, degree + 1)


def reference_save_ply(path, degree):
    """The reference's own GaussianModel.save_ply on the seeded parameters of the byte-equality test (needs its SLAM scripts
    installed under oracle/_ref/gs_icp_slam; used by tests/golden/make_scene_ply_golden.py)."""
    saved_path, saved_mods = list(sys.path), set(sys.modules)
    sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle", "stubs"), REF_SLAM]
    try:
        from scene.gaussian_model import GaussianModel  # the reference's class, unmodified

        p = _params(300, degree, seed=3)
        gm = GaussianModel(degree)
        gm._xyz, gm._features_dc, gm._features_rest = p["xyz"], p["features_dc"], p["features_rest"]
        gm._opacity, gm._scaling, gm._rotation = p["opacity"], p["scaling"], p["rotation"]
        gm.save_ply(path)
    finally:
        sys.path[:] = saved_path
        for k in list(sys.modules):
            if k not in saved_mods and k.split(".")[0] in ("scene", "utils", "arguments", "plyfile", "open3d", "rerun", "torchmetrics"):
                del sys.modules[k]


@pytest.mark.parametrize("degree", [0, 3])
def test_same_bytes_as_reference_save_ply(tmp_path, degree):
    """Byte-for-byte equality with the file the reference's save_ply writes, through its size and SHA-256
    (tests/golden/scene_ply_ref.json)."""
    from gs_icp_slam_b200.map_table import write_scene_ply

    ref = json.load(open(GOLD))[str(degree)]
    our_path = str(tmp_path / "ours" / "scene.ply")
    write_scene_ply(our_path, **_params(300, degree, seed=3))
    blob = open(our_path, "rb").read()
    assert len(blob) == ref["bytes"] and hashlib.sha256(blob).hexdigest() == ref["sha256"]
