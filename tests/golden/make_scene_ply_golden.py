"""Generates tests/golden/scene_ply_ref.json: size and SHA-256 of the scene.ply that the REFERENCE's own
GaussianModel.save_ply writes for the seeded parameters of tests/test_scene_ply.py (its SLAM scripts installed unmodified
under oracle/_ref/gs_icp_slam by `make -C oracle ref` where the reference tree is present).  CPU only:
    python tests/golden/make_scene_ply_golden.py"""
import hashlib
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import test_scene_ply as T  # noqa: E402


def main():
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for degree in (0, 3):
            path = os.path.join(d, str(degree), "scene.ply")
            T.reference_save_ply(path, degree)
            blob = open(path, "rb").read()
            out[str(degree)] = {"bytes": len(blob), "sha256": hashlib.sha256(blob).hexdigest()}
    json.dump(out, open(T.GOLD, "w"), indent=1, sort_keys=True)
    print("wrote", T.GOLD, out)


if __name__ == "__main__":
    main()
