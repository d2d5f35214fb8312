"""Host side of the rasterizer: torch tensors in, C-ABI calls, torch tensors out.

Mirrors the three functions the reference's extension module exports
(submodules/diff-gaussian-rasterization/ext.cpp:15-19, rasterize_points.cu:35-227):
`rasterize_gaussians`, `rasterize_gaussians_backward`, `mark_visible` — same argument order,
same return tuples, same "empty tensor means not provided" convention.  PyTorch is used only
for device memory and the current stream; every kernel is ours (libgsicp_b200.so).
"""
import ctypes as C

import torch

from . import _lib
from ._lib import RasterArgs, check, lib

NUM_CHANNELS = 3

# Tile sharding for multi-GPU runs (SURVEY §8e): (count, index); set by gs_icp_slam_b200.sharding.
_tile_shard = (1, 0)


def set_tile_shard(count, index):
    global _tile_shard
    if count < 1 or not (0 <= index < count):
        raise ValueError("bad tile shard")
    _tile_shard = (int(count), int(index))


def set_comm(comm):
    """Multi-GPU: the library's own exchange group (gs_icp_slam_b200.sharding.ShardGroup) or None.  With tile sharding
    active, rasterize_gaussians_backward exchanges the render moments through the peers' device segments inside the call."""
    check(lib.gsicp_raster_set_comm(comm))


def _ptr(t):
    """Device pointer of a tensor, or None for the reference's 'not provided' empty tensor."""
    if t is None or t.numel() == 0:
        return None
    return t.data_ptr()


def _f32c(t, device):
    if t is None or t.numel() == 0:
        return None
    if t.device != device:
        raise ValueError(f"tensor on {t.device}, expected {device}")
    if t.dtype is torch.float32 and t.is_contiguous():
        return t
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class _Buffers:
    """The three resizable byte buffers (reference: resizeFunctional, rasterize_points.cu:27-33).  One instance per host
    thread, reused by every call: building a ctypes callback thunk costs more than the call it serves."""

    def __init__(self):
        self.device = None
        self.t = {}
        self.cbs = {key: _lib.ALLOC_FN(self._make(key)) for key in ("geom", "binning", "img")}

    def _make(self, key):
        def alloc(nbytes, _user):
            t = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            self.t[key] = t
            return t.data_ptr()

        return alloc

    def begin(self, device):
        self.device = device
        self.t = {}
        return self

    def cb(self, key):
        return self.cbs[key]


import threading  # noqa: E402

_tls = threading.local()


def _buffers(device):
    b = getattr(_tls, "buffers", None)
    if b is None:
        b = _tls.buffers = _Buffers()
    return b.begin(device)


class _on_device:
    """`with torch.cuda.device(dev)` only when dev is not already current (the context manager costs ~10 us)."""

    def __init__(self, dev):
        self.ctx = None if (dev.index is None or torch.cuda.current_device() == dev.index) else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def _arg(t, device):
    """(tensor to keep alive, device pointer) of an optional float32 input; (None, None) for the reference's 'not provided'
    empty tensor.  Fast path: float32 + contiguous tensors are passed through untouched."""
    if t is None:
        return None, None
    if t.dtype is not torch.float32 or not t.is_contiguous():
        if t.numel() == 0:
            return None, None
        t = t.float().contiguous()
    elif t.numel() == 0:
        return None, None
    if t.device != device:
        raise ValueError(f"tensor on {t.device}, expected {device}")
    return t, t.data_ptr()


def _args_struct():
    a = getattr(_tls, "args", None)
    if a is None:
        a = _tls.args = RasterArgs()
    return a


def _fill_args(a, P, D, M, H, W, tanx, tany, scale_mod, prefiltered, debug, ptrs):
    a.P, a.D, a.M, a.width, a.height = P, D, M, W, H
    a.tan_fovx, a.tan_fovy, a.scale_modifier = tanx, tany, scale_mod
    a.prefiltered, a.debug = int(bool(prefiltered)), int(bool(debug))
    (a.d_background, a.d_means3D, a.d_shs, a.d_colors_precomp, a.d_opacities, a.d_scales, a.d_rotations, a.d_cov3D_precomp,
     a.d_viewmatrix, a.d_projmatrix, a.d_campos) = ptrs
    a.tile_shard_count, a.tile_shard_index = _tile_shard
    return a


def rasterize_gaussians(background, means3D, colors, opacity, scales, rotations, scale_modifier, cov3D_precomp,
                        viewmatrix, projmatrix, tan_fovx, tan_fovy, image_height, image_width, sh, degree, campos,
                        prefiltered, debug):
    """_C.rasterize_gaussians (rasterize_points.cu:35-121).

    Returns (num_rendered, out_depth[1,H,W], out_color[3,H,W], radii[P] int32, is_used[P] bool,
    geomBuffer, binningBuffer, imgBuffer)."""
    if means3D.ndimension() != 2 or means3D.size(1) != 3:
        raise RuntimeError("means3D must have dimensions (num_points, 3)")
    if not means3D.is_cuda:
        raise RuntimeError("gs_icp_slam_b200 rasterizer: means3D must be a CUDA tensor (no CPU fallback)")
    dev = means3D.device
    P, H, W = means3D.size(0), int(image_height), int(image_width)
    with _on_device(dev):
        # The kernels write every element of the four outputs when P > 0 and all tiles are rendered here, so no
        # zero-fill launches are needed (the reference fills them: rasterize_points.cu:65-68).
        alloc = torch.empty if (P != 0 and _tile_shard[0] == 1) else torch.zeros
        out_depth = alloc((1, H, W), dtype=torch.float32, device=dev)
        out_color = alloc((NUM_CHANNELS, H, W), dtype=torch.float32, device=dev)
        radii = alloc((P,), dtype=torch.int32, device=dev)
        is_used = alloc((P,), dtype=torch.bool, device=dev)
        bufs = _buffers(dev)
        rendered = 0
        if P != 0:
            M = sh.size(1) if sh.numel() != 0 else 0
            keep, ptrs = zip(*[_arg(x, dev) for x in (background, means3D, sh, colors, opacity, scales, rotations,
                                                        cov3D_precomp, viewmatrix, projmatrix, campos)])
            args = _fill_args(_args_struct(), P, int(degree), M, H, W, float(tan_fovx), float(tan_fovy), float(scale_modifier),
                              prefiltered, debug, ptrs)
            stream = torch.cuda.current_stream(dev).cuda_stream
            rendered = check(
                lib.gsicp_raster_forward(C.byref(args), out_color.data_ptr(), out_depth.data_ptr(), radii.data_ptr(),
                                         is_used.data_ptr(), bufs.cb("geom"), bufs.cb("binning"), bufs.cb("img"), None,
                                         stream), "gsicp_raster_forward")
            del keep
        t = bufs.t
        empty = None
        if len(t) != 3:
            empty = torch.empty(0, dtype=torch.uint8, device=dev)
        return (rendered, out_depth, out_color, radii, is_used, t.get("geom", empty), t.get("binning", empty),
                t.get("img", empty))


def rasterize_gaussians_backward(background, means3D, radii, colors, scales, rotations, scale_modifier, cov3D_precomp,
                                 viewmatrix, projmatrix, tan_fovx, tan_fovy, dL_dout_depth, dL_dout_color, sh, degree,
                                 campos, geomBuffer, R, binningBuffer, imageBuffer, debug):
    """_C.rasterize_gaussians_backward (rasterize_points.cu:123-206).

    Returns (dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales, dL_drotations)."""
    dev = means3D.device
    P = means3D.size(0)
    H, W = dL_dout_color.size(1), dL_dout_color.size(2)
    M = sh.size(1) if sh.numel() != 0 else 0
    with _on_device(dev):
        # One UNINITIALISED slab for the eight gradient tensors: the per-Gaussian backward kernel writes every element
        # (zeros for Gaussians outside the view), so no fill launch precedes it.  The kernels are launched from raw offsets
        # into it; the tensor views are made afterwards, while the GPU is busy.
        sizes = (3 * P, 3 * P, NUM_CHANNELS * P, P, 6 * P, 3 * M * P, 3 * P, 4 * P)
        offs, off = [], 0
        for n in sizes:
            offs.append(off)
            off += (n + 3) // 4 * 4  # keep every view 16-byte aligned
        slab = (torch.empty if P != 0 else torch.zeros)(max(off, 1), dtype=torch.float32, device=dev)
        if P != 0:
            base = slab.data_ptr()
            p3d, p2d, pcol, popa, pcov, psh, psc, prot = (base + 4 * o for o in offs)
            keep, ptrs = zip(*[_arg(x, dev) for x in (background, means3D, sh, colors, None, scales, rotations, cov3D_precomp,
                                                        viewmatrix, projmatrix, campos, dL_dout_color, dL_dout_depth)])
            args = _fill_args(_args_struct(), P, int(degree), M, H, W, float(tan_fovx), float(tan_fovy), float(scale_modifier),
                              False, debug, ptrs[:11])
            stream = torch.cuda.current_stream(dev).cuda_stream
            radii_c = radii if radii.is_contiguous() else radii.contiguous()
            check(
                lib.gsicp_raster_backward(C.byref(args), int(R), radii_c.data_ptr(), geomBuffer.data_ptr(),
                                          binningBuffer.data_ptr(), imageBuffer.data_ptr(), ptrs[11], ptrs[12], p2d, pcol, popa,
                                          p3d, pcov, psh if M != 0 else None, psc, prot, None, stream),
                "gsicp_raster_backward")
            del keep
        shapes = ((P, 3), (P, 3), (P, NUM_CHANNELS), (P, 1), (P, 6), (P, M, 3), (P, 3), (P, 4))
        dL_dmeans3D, dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dcov3D, dL_dsh, dL_dscales, dL_drotations = (
            slab[o:o + n].view(shp) for o, n, shp in zip(offs, sizes, shapes))
        return dL_dmeans2D, dL_dcolors, dL_dopacity, dL_dmeans3D, dL_dcov3D, dL_dsh, dL_dscales, dL_drotations


def mark_visible(means3D, viewmatrix, projmatrix):
    """_C.mark_visible (rasterize_points.cu:208-227)."""
    dev = means3D.device
    P = means3D.size(0)
    present = torch.zeros((P,), dtype=torch.bool, device=dev)
    if P != 0:
        with torch.cuda.device(dev):
            m3, view, proj = (_f32c(x, dev) for x in (means3D, viewmatrix, projmatrix))
            check(lib.gsicp_mark_visible(P, m3.data_ptr(), view.data_ptr(), proj.data_ptr(), present.data_ptr(),
                                         torch.cuda.current_stream(dev).cuda_stream), "gsicp_mark_visible")
    return present


def export_binning(num_rendered, height, width, binningBuffer, imageBuffer):
    """Test hook: (point_list uint32[R] as int64 tensor, ranges int64[tiles,2]) from the saved state."""
    dev = imageBuffer.device
    tiles = ((width + 15) // 16) * ((height + 15) // 16)
    a = RasterArgs()
    a.width, a.height = width, height
    pl = torch.zeros(max(num_rendered, 1), dtype=torch.int32, device=dev)
    rg = torch.zeros(tiles * 2, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.gsicp_raster_export_binning(C.byref(a), int(num_rendered), binningBuffer.data_ptr(),
                                              imageBuffer.data_ptr(), pl.data_ptr(), rg.data_ptr(),
                                              torch.cuda.current_stream(dev).cuda_stream))
    return pl[:num_rendered].to(torch.int64), rg.view(tiles, 2).to(torch.int64)
