"""Host side of the GICP tracker: numpy in / numpy out over the C ABI (include/gsicp_b200.h).

`FastGICP` mirrors the pybind11 class the reference exports as `pygicp.FastGICP`
(submodules/fast_gicp/src/python/main.cpp:166-262): same method names, argument meaning, dtypes of the
returned arrays (float32 1-D copies, float32 4x4 pose) and error behaviour (stderr message + early return
where the reference does that).  All compute runs in libgsicp_b200.so on the GPU; there is no CPU path.
"""
import ctypes as C
import sys

import numpy as np

from . import _lib
from ._lib import check, lib


def _f32_1d(a):
    return np.ascontiguousarray(np.asarray(a), dtype=np.float32).reshape(-1)


class FastGICP:
    """pygicp.FastGICP drop-in.  Picklable like the reference (state is not carried across, main.cpp:183-201)."""

    def __init__(self):
        self._h = lib.gsicp_gicp_create()
        if not self._h:
            raise _lib.GsicpError("gsicp_gicp_create failed: " + _lib.last_error())
        self._stream_ptr = 0  # the handle's stream (0 = legacy default stream)

    def _device_input(self, t):
        """float32 contiguous view of a CUDA tensor, ordered for the handle's stream: the library enqueues an asynchronous
        copy on ITS stream, so that stream first waits for the work torch has queued on the tensor's producer stream, and the
        caching allocator is told the block is in use there (a conversion temporary dies when this call returns)."""
        import torch

        x = t.detach()
        if x.dtype is not torch.float32 or not x.is_contiguous():
            x = x.float().contiguous()
        cur = torch.cuda.current_stream(x.device)
        if cur.cuda_stream != self._stream_ptr:
            ext = torch.cuda.ExternalStream(self._stream_ptr, device=x.device) if self._stream_ptr else torch.cuda.default_stream(x.device)
            if ext.cuda_stream != cur.cuda_stream:
                ext.wait_stream(cur)
                x.record_stream(ext)
        return x

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                lib.gsicp_gicp_destroy(h)
            except Exception:
                pass

    # pickling: the reference's __setstate__ builds a fresh object (mp.spawn pickles the tracker)
    def __getstate__(self):
        return ()

    def __setstate__(self, state):
        self.__init__()

    # ---- parameters ----
    def set_num_threads(self, n):  # OpenMP knob of the CPU implementation: no-op on the GPU
        return None

    def set_correspondence_randomness(self, k):
        check(lib.gsicp_gicp_set_correspondence_randomness(self._h, int(k)))

    def set_max_correspondence_distance(self, d):
        check(lib.gsicp_gicp_set_max_correspondence_distance(self._h, float(d)))

    def set_max_knn_distance(self, d):
        check(lib.gsicp_gicp_set_max_knn_distance(self._h, float(d)))

    def set_max_iterations(self, n):
        check(lib.gsicp_gicp_set_max_iterations(self._h, int(n)))

    # ---- clouds ----
    @staticmethod
    def _cloud(points):
        if hasattr(points, "is_cuda") and points.is_cuda:  # zero-copy path for CUDA tensors (SURVEY §8f N1)
            return points, None
        a = np.asarray(points)
        if a.ndim != 2 or a.shape[1] != 3:
            raise TypeError("points must have shape (N, 3)")  # pybind would raise a TypeError as well
        if a.dtype == np.float32:
            return np.ascontiguousarray(a), 1
        return np.ascontiguousarray(a, dtype=np.float64), 0

    def set_input_source(self, points):
        a, f32 = self._cloud(points)
        if f32 is None:
            t = self._device_input(a)
            check(lib.gsicp_gicp_set_input_source_device(self._h, t.data_ptr(), t.shape[0]))
        else:
            check(lib.gsicp_gicp_set_input_source(self._h, a.ctypes.data, a.shape[0], f32))

    def set_input_target(self, points):
        a, f32 = self._cloud(points)
        if f32 is None:
            t = self._device_input(a)
            check(lib.gsicp_gicp_set_input_target_device(self._h, t.data_ptr(), t.shape[0]))
        else:
            check(lib.gsicp_gicp_set_input_target(self._h, a.ctypes.data, a.shape[0], f32))

    def set_source_filter(self, num_trackable, input_filter):
        if hasattr(input_filter, "is_cuda") and input_filter.is_cuda:  # zero-copy path (SURVEY §8f N1)
            import torch

            t = input_filter.detach().to(torch.int32).contiguous().view(-1)
            check(lib.gsicp_gicp_set_source_filter_device(self._h, int(num_trackable), t.data_ptr(), t.shape[0]))
            return
        f = np.ascontiguousarray(np.asarray(input_filter).reshape(-1), dtype=np.int32)
        check(lib.gsicp_gicp_set_source_filter(self._h, int(num_trackable), f.ctypes.data, f.shape[0]))

    def set_target_filter(self, num_trackable, input_filter):
        if hasattr(input_filter, "is_cuda") and input_filter.is_cuda:
            import torch

            t = input_filter.detach().to(torch.int32).contiguous().view(-1)
            check(lib.gsicp_gicp_set_target_filter_device(self._h, int(num_trackable), t.data_ptr(), t.shape[0]))
            return
        f = np.ascontiguousarray(np.asarray(input_filter).reshape(-1), dtype=np.int32)
        check(lib.gsicp_gicp_set_target_filter(self._h, int(num_trackable), f.ctypes.data, f.shape[0]))

    # ---- covariances ----
    def calculate_source_covariance(self):
        check(lib.gsicp_gicp_calculate_source_covariance(self._h))

    def calculate_target_covariance(self):
        check(lib.gsicp_gicp_calculate_target_covariance(self._h))

    def calculate_target_covariance_with_filter(self):
        check(lib.gsicp_gicp_calculate_target_covariance_with_filter(self._h))

    def calculate_target_covariance_withz(self):  # main.cpp:228
        check(lib.gsicp_gicp_calculate_target_covariance_withz(self._h))

    def set_source_z_values(self, z_values):  # main.cpp:246-249
        z = _f32_1d(z_values)
        check(lib.gsicp_gicp_set_source_z_values(self._h, z.ctypes.data, len(z)))

    def set_target_z_values(self, z_values):  # main.cpp:250-253
        z = _f32_1d(z_values)
        check(lib.gsicp_gicp_set_target_z_values(self._h, z.ctypes.data, len(z)))

    def swap_source_and_target(self):  # main.cpp:169
        check(lib.gsicp_gicp_swap_source_and_target(self._h))

    def _fromqs(self, fn, rotationsq, scales):
        if hasattr(rotationsq, "is_cuda") and rotationsq.is_cuda:  # zero-copy path for CUDA tensors
            r = self._device_input(rotationsq).view(-1)
            s = self._device_input(scales).view(-1)
            if r.numel() // 4 != s.numel() // 3:
                print("qs size not matched", file=sys.stderr)
                return
            dev_fn = getattr(lib, fn.__name__ + "_device")
            check(dev_fn(self._h, r.data_ptr(), s.data_ptr(), s.numel() // 3))
            return
        r, s = _f32_1d(rotationsq), _f32_1d(scales)
        if len(r) // 4 != len(s) // 3:
            print("qs size not matched", file=sys.stderr)  # main.cpp:235,241
            return
        check(fn(self._h, r.ctypes.data, s.ctypes.data, len(s) // 3))

    def set_source_covariances_fromqs(self, rotationsq, scales):
        self._fromqs(lib.gsicp_gicp_set_source_covariances_fromqs, rotationsq, scales)

    def set_target_covariances_fromqs(self, rotationsq, scales):
        self._fromqs(lib.gsicp_gicp_set_target_covariances_fromqs, rotationsq, scales)

    # ---- registration ----
    def align(self, initial_guess=None):
        g = np.eye(4, dtype=np.float32) if initial_guess is None else np.ascontiguousarray(initial_guess, dtype=np.float32)
        if g.shape != (4, 4):
            raise TypeError("initial_guess must be 4x4")
        out = np.empty((4, 4), dtype=np.float32)
        self.last_iterations = check(lib.gsicp_gicp_align(self._h, g.ctypes.data, out.ctypes.data), "align")
        self._final = out.copy()
        return out

    def get_final_transformation(self):  # LsqRegistration binding, main.cpp:171
        return getattr(self, "_final", np.eye(4, dtype=np.float32)).copy()

    def has_converged(self):
        return bool(check(lib.gsicp_gicp_has_converged(self._h)))

    def get_fitness_score(self, max_range):  # main.cpp:172
        out = C.c_double(0.0)
        check(lib.gsicp_gicp_get_fitness_score(self._h, float(max_range), C.byref(out)))
        return out.value

    def get_final_hessian(self):
        H = np.empty((6, 6), dtype=np.float64)
        check(lib.gsicp_gicp_get_final_hessian(self._h, H.ctypes.data))
        return H

    # ---- getters: 1-D float32 copies (main.cpp:206-233) ----
    def _vec(self, size_fn, get_fn, dtype=np.float32):
        n = check(size_fn(self._h))
        out = np.empty(n, dtype=dtype)
        if n:
            check(get_fn(self._h, out.ctypes.data))
        return out

    def get_source_rotationsq(self):
        return self._vec(lib.gsicp_gicp_source_rotationsq_size, lib.gsicp_gicp_get_source_rotationsq)

    def get_target_rotationsq(self):
        return self._vec(lib.gsicp_gicp_target_rotationsq_size, lib.gsicp_gicp_get_target_rotationsq)

    def get_source_scales(self):
        return self._vec(lib.gsicp_gicp_source_scales_size, lib.gsicp_gicp_get_source_scales)

    def get_target_scales(self):
        return self._vec(lib.gsicp_gicp_target_scales_size, lib.gsicp_gicp_get_target_scales)

    def get_source_correspondence(self):
        n = check(lib.gsicp_gicp_source_size(self._h))
        corr = np.empty(n, dtype=np.int32)
        sqd = np.empty(n, dtype=np.float32)
        check(lib.gsicp_gicp_get_source_correspondence(self._h, corr.ctypes.data, sqd.ctypes.data))
        return corr, sqd

    # ---- extras used by tests / bench (not part of the reference class) ----
    def source_size(self):
        return check(lib.gsicp_gicp_source_size(self._h))

    def target_size(self):
        return check(lib.gsicp_gicp_target_size(self._h))

    def get_source_covariances(self):
        n = self.source_size()
        out = np.empty((n, 3, 3), dtype=np.float64)
        check(lib.gsicp_gicp_get_source_covariances(self._h, out.ctypes.data))
        return out

    def get_target_covariances(self):
        n = self.target_size()
        out = np.empty((n, 3, 3), dtype=np.float64)
        check(lib.gsicp_gicp_get_target_covariances(self._h, out.ctypes.data))
        return out

    def linearize(self, pose):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        H, b, e = np.empty((6, 6)), np.empty(6), C.c_double(0)
        check(lib.gsicp_gicp_linearize(self._h, p.ctypes.data, H.ctypes.data, b.ctypes.data, C.byref(e)), "linearize")
        return H, b, e.value

    def compute_error(self, pose):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        e = C.c_double(0)
        check(lib.gsicp_gicp_compute_error(self._h, p.ctypes.data, C.byref(e)), "compute_error")
        return e.value

    def set_stream(self, cuda_stream):
        check(lib.gsicp_gicp_set_stream(self._h, int(cuda_stream)))
        self._stream_ptr = int(cuda_stream)

    def set_comm(self, comm):
        """Multi-GPU: shard the source points (k-NN covariances and LM loop) over the library's exchange group and exchange
        the normal equations inside the kernels (gs_icp_slam_b200.sharding.ShardGroup); None = single GPU."""
        check(lib.gsicp_gicp_set_comm(self._h, comm))

    def set_host_lm(self, on):
        """Test / A-B hook: drive the LM loop from the host instead of the device-resident kernel (same results)."""
        check(lib.gsicp_gicp_set_host_lm(self._h, int(bool(on))))
