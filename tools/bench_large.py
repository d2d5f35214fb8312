"""GICP-only / rasterizer-only configs of bench.py (`--config c1|c4|c5`), one process per GPU under torchrun:
  C1: GICP align of two 10k-point clouds (the reference's own CPU-runnable case); `--impl reference` times the real
      fast_gicp (oracle/_ref, all host threads) on the same pair
  C4: 1280x960, 1M Gaussians, rasterizer fwd+bwd only, tiles sharded over the ranks (moments exchange inside backward)
  C5: GICP align on a 2M x 2M point pair, source points sharded (28-double normal equations exchanged per linearize)
Total work is fixed as N grows ("scaling": "strong").  A step = one raster fwd+bwd iteration (C4) / one align() (C5).
Same JSON contract as the default config: W warm-up steps, K steps timed with CUDA events between barriers, max over ranks.
    python bench.py --config c4 [--gpus N --steps K --warmup W]      (torchrun for N > 1)"""
import json
import os
import time

import numpy as np


def _timed(fn, steps, warmup, world, dev, torch, dist, flush):
    ts = []
    for i in range(warmup + steps):
        flush.fill_(i & 0xff)  # L2 flush between steps, outside the timed events
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i >= warmup:
            ts.append(e0.elapsed_time(e1))
    t = torch.tensor([float(np.sum(ts))], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), ts


_C1_WORKLOAD = ("C1: GICP align of a {n} x {n} point pair (seeds 0/1), identity guess, k-NN source covariances + LM loop, "
                "max_corr 0.05; target covariances precomputed outside the step")


def _c1_reference(args):
    """The reference's tracker on C1: fast_gicp itself (oracle/_ref/fast_gicp, unmodified sources, OpenMP on every host
    thread), same pair, same calls per step (set_input_source + set_source_filter + align with lazy source covariances)."""
    from gs_icp_slam_b200 import synthetic as S
    from oracle import ref_gicp

    if not ref_gicp.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/fast_gicp not built (make -C oracle ref needs /root/reference)"}))
        return
    n = args.gaussians
    tgt, src, T = S.gicp_pair(n, n)
    reg = ref_gicp.FastGICP()
    cores = os.cpu_count() or 1
    reg.set_num_threads(cores)
    reg.set_max_correspondence_distance(0.05)
    reg.set_max_knn_distance(99999)
    filt = np.arange(1, n + 1, dtype=np.int32)
    reg.set_input_target(tgt)
    reg.set_target_filter(n, filt)
    reg.calculate_target_covariance_with_filter()
    ts, pose = [], None
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        reg.set_input_source(src)
        reg.set_source_filter(n, filt)  # the SLAM's fast_gicp indexes its covariance table through the filter: always set
        pose = np.array(reg.align(np.eye(4, dtype=np.float32)))
        if i >= args.warmup:
            ts.append(time.perf_counter() - t0)
    v = len(ts) / float(np.sum(ts))
    print(json.dumps({"impl": "reference", "metric": "GICP align/sec (10k x 10k points)", "value": v, "unit": "aligns/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "f64 (GICP algebra on f32 points)", "data": "synthetic",
                      "config": {"workload": _C1_WORKLOAD.format(n=n)},
                      "cpu_baseline": {"value": v, "unit": "aligns/s", "cores": cores, "kind": "reference",
                                       "sample": f"{args.steps} full aligns of the same pair"},
                      "e2e": {"value": v, "unit": "aligns/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "pose_error_vs_ground_truth": float(np.abs(pose.astype(np.float64) - T).max())}))


def main(args, rank, local_rank, world):
    import torch

    from gs_icp_slam_b200 import _lib, sharding
    from gs_icp_slam_b200 import synthetic as S

    if args.impl == "reference" and args.config == "c1":
        if rank == 0:
            _c1_reference(args)
        return
    if args.impl == "reference":
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "the large configs have no reference arm: the reference's "
                              "rasterizer / fast_gicp are single-device (SURVEY §8e); see the default config"}))
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, args.warmup
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    group = sharding.ShardGroup(dev, world, rank) if world > 1 else None
    extra = {}
    if args.config == "c4":
        from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
        from gs_icp_slam_b200 import rasterizer as R

        W, H, P = 1280, 960, args.gaussians
        cam = dict(S.TUM)
        cam.update(W=W, H=H, fx=cam["fx"] * 2, fy=cam["fy"] * 2, cx=cam["cx"] * 2, cy=cam["cy"] * 2)
        g = S.gaussian_map(P, 4, scale=2.0)
        cm = S.camera_matrices(S.trajectory_pose(3, 20, scale=2.0), cam)
        t = {k: torch.from_numpy(v).to(dev).requires_grad_(True) for k, v in g.items()}
        c = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) else v) for k, v in cm.items()}
        m2 = torch.zeros_like(t["means3D"], requires_grad=True)
        gen = torch.Generator(device="cpu").manual_seed(5)
        gcol, gdep = torch.randn((3, H, W), generator=gen).to(dev), torch.randn((1, H, W), generator=gen).to(dev)
        if group is not None:
            group.attach_rasterizer()
        mask = sharding.tile_owner_mask(H, W, world, rank, dev)
        # BASELINE config C4: "fwd+bwd with dL_dcolor, dL_ddepth ~ N(0,1)" — each rank feeds the gradients of its own tiles
        gcol_own, gdep_own = (gcol * mask).contiguous(), (gdep * mask).contiguous()
        rs = GaussianRasterizationSettings(H, W, c["tanfovx"], c["tanfovy"], torch.zeros(3, device=dev), 1.0, c["viewmatrix"],
                                           c["projmatrix"], 0, c["campos"], False, False)
        info = {}

        def it():
            depth, color, radii, used = GaussianRasterizer(rs)(means3D=t["means3D"], means2D=m2, opacities=t["opacities"],
                                                               shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
            info["R"] = color.grad_fn.num_rendered
            torch.autograd.backward([color, depth], [gcol_own, gdep_own])
            for k in t:
                t[k].grad = None
            m2.grad = None

        metric, unit = "rasterizer fwd+bwd iterations/sec (1280x960, 1M Gaussians)", "iterations/s"
        workload = f"C4: 1280x960, {P} Gaussians (seed 4), rasterizer forward + backward with N(0,1) image gradients"
        step = it
        extra["tile_instances_this_rank"] = lambda: info.get("R")
    else:
        import pygicp

        n = args.gaussians
        c1 = args.config == "c1"
        tgt, src, T = S.gicp_pair(n, n) if c1 else S.gicp_pair(n, n, 6, 7, 0.001, scale=5.0)
        reg = pygicp.FastGICP()
        reg.set_max_correspondence_distance(0.05 if c1 else 0.25)
        reg.set_max_knn_distance(99999)
        if group is not None:
            group.attach_gicp(reg)
        reg.set_input_target(tgt)
        if c1:
            filt = np.arange(1, n + 1, dtype=np.int32)
            reg.set_target_filter(n, filt)
            reg.calculate_target_covariance_with_filter()
        else:
            reg.calculate_target_covariance()
        src_dev = torch.from_numpy(src.astype(np.float32)).to(dev)
        res = {}

        def it():
            reg.set_input_source(src_dev)   # new frame: source covariances are recomputed inside align (fgi:229-232)
            if c1:
                reg.set_source_filter(n, filt)
            res["pose"] = reg.align(np.eye(4, dtype=np.float32))

        metric, unit = ("GICP align/sec (10k x 10k points)" if c1 else "GICP align/sec (2M x 2M points)"), "aligns/s"
        workload = (_C1_WORKLOAD.format(n=n) if c1 else
                    f"C5: GICP align of a {n} x {n} point pair (seeds 6/7), k-NN source covariances + LM loop, max_corr 0.25")
        step = it
        extra["lm_iterations"] = lambda: reg.last_iterations
        extra["pose_error_vs_ground_truth"] = lambda: float(np.abs(res["pose"].astype(np.float64) - T).max())

    for _ in range(2):  # allocator / scratch growth, untimed
        step()
    l0 = _lib.launch_count() if hasattr(_lib, "launch_count") else 0
    t_ms, ts = _timed(step, K, Wm, world, dev, torch, dist, flush)
    launches = ((_lib.launch_count() - l0) * K) // (K + Wm) if hasattr(_lib, "launch_count") else 0
    _lib.prof_reset()
    _lib.prof_enable(True)
    for _ in range(min(K, 5)):
        step()
    torch.cuda.synchronize()
    _lib.prof_enable(False)
    kern = {k: {"ms_per_launch": v[0] / v[1], "launches_per_step": v[1] / min(K, 5)} for k, v in _lib.prof_read().items() if v[1]}
    if rank == 0:
        out = {"metric": metric, "value": K / (t_ms * 1e-3), "unit": unit, "n_gpus": world, "steps": K, "warmup": Wm,
               "ms_per_step": t_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f32 (rasterizer)" if args.config == "c4" else "f64 (GICP algebra on f32 points)", "data": "synthetic",
               "gpu_launches": int(launches),
               "config": {"workload": workload, "l2": "256 MiB write between steps, excluded from the per-step CUDA-event time"},
               "parallelism": "single GPU" if world == 1 else (f"{world} GPUs: " + ("screen tiles" if args.config == "c4" else "source points") +
                                                                " sharded, in-kernel exchange over peer memory"),
               "ms_p50_max": [float(np.median(ts)), float(np.max(ts))], "kernels": kern,
               "e2e": {"value": K / (t_ms * 1e-3), "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 64,
                       "note": "the public API call is what is timed; inputs are device tensors of the caller (the mapper's "
                               "parameters / the tracker's cloud), results (loss gradient tensors / 4x4 pose) stay where the API puts them"}}
        for k, f in extra.items():
            out[k] = f()
        print(json.dumps(out))
    if group is not None:
        group.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
