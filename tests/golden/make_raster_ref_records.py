"""Generates tests/golden/raster_ref_records.npz: records (tests/refdigest.py) of the REFERENCE's own rasterizer and
simple-knn on the scenes of the GPU parity tests — its CUDA code compiled unmodified for sm_100a (oracle/_ref/libref_cuda.so)
and its PyTorch extension built through its own setup.py (oracle/_ref/site), both made by `make -C oracle ref` where the
reference tree is present.  Needs a GPU:
    python tests/golden/make_raster_ref_records.py [OUT.npz]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from gs_icp_slam_b200 import synthetic as S  # noqa: E402
from oracle import ref_cuda, ref_ext  # noqa: E402
from tests import test_raster_gpu as T  # noqa: E402
from tests.refdigest import RASTER_RECORDS, record, save  # noqa: E402
from tests.util import scene_tensors  # noqa: E402


def ref_raster(t, c, H, W, bg, degree=0, scale_modifier=1.0, colors=None, cov=None):
    shs = t["shs"] if colors is None else None
    sc, rot = (t["scales"], t["rotations"]) if cov is None else (None, None)
    return ref_cuda.RefRaster(bg, t["means3D"], shs, colors, t["opacities"].reshape(-1), sc, rot, cov, c["viewmatrix"],
                              c["projmatrix"], c["campos"], c["tanfovx"], c["tanfovy"], H, W, degree, scale_modifier=scale_modifier)


def put(out, k, ref, grads=None, names=T.GRADS, extra_rows=()):
    out[k + "num_rendered"] = np.int64(ref.num_rendered)
    pl, rg = ref.export()
    for name, x in (("radii", ref.radii), ("is_used", ref.is_used), ("point_list", pl), ("ranges", rg), ("color", ref.color),
                    ("depth", ref.depth)):
        record(out, k + name, x)
    if grads is not None:
        g = ref.backward(*grads)
        for name in names:
            record(out, k + "grad_" + name, g[name], extra_rows=extra_rows)
    ref.free()


def main():
    dev = torch.device("cuda:0")
    out = {}
    for P, (W, H), degree, seed in [(20000, (320, 240), 0, 2), (100000, (640, 480), 0, 3), (30000, (333, 211), 3, 5)]:
        t, c, bg, grads = T.fb_scene(dev, P, (W, H), degree, seed)
        put(out, f"fb_{P}_{W}x{H}_{degree}_{seed}/", ref_raster(t, c, H, W, bg, degree), grads)
    for active, sm, (W, H) in [(2, 0.7, (250, 190)), (1, 1.6, (96, 64)), (0, 1.0, (17, 33))]:
        t, c, bg, grads = T.options_scene(dev, active, (W, H))
        put(out, f"opt_{active}_{sm}_{W}x{H}/", ref_raster(t, c, H, W, bg, active, scale_modifier=sm), grads)
    t, c, a, bg, grads = T.degenerate_scene(dev)
    put(out, "degenerate/", ref_raster(t, c, 152, 200, bg), grads, extra_rows=a.cpu().numpy())
    t, c, colors, cov, bg, grads = T.precomputed_scene(dev)
    put(out, "precomputed/", ref_raster(t, c, 240, 320, bg, colors=colors, cov=cov), grads, names=T.GRADS[:5])
    for P in (9000, 40000):
        t, c, bg = T.crowded_scene(dev, P)
        put(out, f"crowded_{P}/", ref_raster(t, c, 120, 160, bg))
    ref_mod = ref_ext.diff_gaussian_rasterization()
    for P, (W, H), degree, seed in [(100000, (640, 480), 0, 3), (30000, (333, 211), 3, 5), (300000, (640, 480), 0, 3)]:
        t, c, bg, active, grads = T.autograd_scene(dev, P, (W, H), degree, seed)
        depth, color, radii, is_used, g1, g2 = T.autograd_run(ref_mod, t, c, bg, active, grads, H, W)
        k = f"ext_{P}_{W}x{H}_{degree}_{seed}/"
        for name, x in (("radii", radii), ("is_used", is_used), ("depth", depth), ("color", color)):
            record(out, k + name, x)
        for name, x in g1.items():
            record(out, k + "g1_" + name, x)
        for name, x in g2.items():
            record(out, k + "g2_" + name, x)
    # tests/test_full_size_gpu.py: C3 and C4 sizes, first of its two seeded upstream gradients
    for P, (W, H), scale in [(300000, (640, 480), 1.0), (1000000, (1280, 960), 2.0)]:
        g, cm, t, c, cam = scene_tensors(P, 3 if P == 300000 else 4, dev, size=(W, H), scale=scale)
        bg = torch.tensor([0.05, 0.1, 0.15], device=dev)
        gen = torch.Generator(device="cpu").manual_seed(1)
        g1c = torch.randn((3, H, W), generator=gen).to(dev)
        torch.randn((3, H, W), generator=gen)
        g1d = torch.randn((1, H, W), generator=gen).to(dev)
        put(out, f"full_{P}/", ref_raster(t, c, H, W, bg), (g1c, g1d))
    # tests/test_gicp_gpu.py::test_dist2_matches_bruteforce_and_reference
    big = torch.from_numpy(S.sample_surface(200000, 41, 0.002)[0].astype(np.float32)).to(dev)
    record(out, "dist2_200000/dist2", ref_cuda.ref_dist2(big))
    path = sys.argv[1] if len(sys.argv) > 1 else RASTER_RECORDS
    save(path, out)
    print("wrote", path, len(out), "entries,", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
