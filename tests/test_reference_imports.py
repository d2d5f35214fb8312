"""Drop-in check at import level: the statements with which the reference's own SLAM modules import the packages this
repository replaces (tests/golden/reference_imports.json, found by parsing the reference's sources with
tests/golden/make_reference_imports_golden.py) bind OUR pygicp / diff_gaussian_rasterization / simple_knn, every name and
attribute they take from them exists, and the keyword names the reference's renderer passes exist on our classes."""
import importlib
import inspect
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPEC = os.path.join(ROOT, "tests", "golden", "reference_imports.json")


def test_reference_modules_bind_our_extensions():
    import diff_gaussian_rasterization as ours_dgr
    import pygicp as ours_gicp
    from simple_knn._C import distCUDA2 as ours_dist

    assert ours_gicp.__file__.startswith(ROOT) and ours_dgr.__file__.startswith(ROOT)
    spec = json.load(open(SPEC))
    # gaussian_renderer/__init__.py:14, scene/gaussian_model.py:20, mp_Tracker.py:15,53
    assert {"gaussian_renderer/__init__.py", "scene/gaussian_model.py", "mp_Tracker.py"} <= {k for k, v in spec.items() if v}
    for path, statements in spec.items():
        for st in statements:
            m = importlib.import_module(st["module"])
            assert os.path.abspath(m.__file__).startswith(ROOT), (path, st["module"], m.__file__)
            for name in st["names"] + st["attributes"]:
                assert hasattr(m, name), (path, st["module"], name)
    assert importlib.import_module("simple_knn._C").distCUDA2 is ours_dist
    # the keyword names the reference's renderer passes (gaussian_renderer/__init__.py:36-51,86-94) exist on our classes
    assert list(ours_dgr.GaussianRasterizationSettings._fields) == [
        "image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix", "sh_degree",
        "campos", "prefiltered", "debug"]
    assert list(inspect.signature(ours_dgr.GaussianRasterizer.__init__).parameters)[1:] == ["raster_settings"]
    assert list(inspect.signature(ours_dgr.GaussianRasterizer.forward).parameters)[1:] == [
        "means3D", "means2D", "opacities", "shs", "colors_precomp", "scales", "rotations", "cov3D_precomp"]
    # every FastGICP method the trackers call (mp_Tracker.py:53-308)
    for m in ("set_max_correspondence_distance", "set_max_knn_distance", "set_input_target", "set_input_source",
              "set_target_filter", "set_source_filter", "calculate_target_covariance_with_filter", "get_target_rotationsq",
              "get_target_scales", "get_source_rotationsq", "get_source_scales", "align", "get_source_correspondence",
              "set_target_covariances_fromqs"):
        assert callable(getattr(ours_gicp.FastGICP, m)), m
