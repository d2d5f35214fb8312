"""The device-side exchange protocols of csrc/comm.cuh on ONE GPU: two "ranks" of an exchange group live in one process
(gsicp_comm_connect_local: plain device pointers instead of CUDA IPC handles), each driven by its own host thread and
stream.  Point-sharded GICP — k-NN covariances, the persistent LM kernel (in-kernel exchange at every reduction point)
and the host-driven kernels (exchange in the last block) — must reproduce the unsharded result; so must the sum-merged
getters.  The real multi-process / NVLink path is tests/test_multigpu_gpu.py (needs >= 2 GPUs).

Two ranks sharing ONE CUDA context is an emulation with a hazard the real layout (one process and one context per GPU)
does not have: anything that synchronises the whole context while a peer's kernel spins on a flag deadlocks — lazy module
loading of a kernel's first launch does, and so does cudaFree/cudaHostAlloc.  So the ranks run in a child process that loads
the library's kernels up front (gsicp_test_preload_kernels), and every handle does one unsharded pass first (all scratch
sized, nothing left to allocate, every PyTorch kernel on the call path loaded)."""
import ctypes as C
import os
import subprocess
import sys
import threading

import numpy as np
import pytest
import torch

from gs_icp_slam_b200 import synthetic as S

pytestmark = pytest.mark.gpu


def _group(world, heap=64 << 20):
    from gs_icp_slam_b200._lib import check, lib

    comms = []
    for _ in range(world):
        c, h = C.c_void_p(), C.create_string_buffer(64)
        check(lib.gsicp_comm_alloc(heap, C.byref(c), h), "gsicp_comm_alloc")
        comms.append(c)
    arr = (C.c_void_p * world)(*[c.value for c in comms])
    for r, c in enumerate(comms):
        check(lib.gsicp_comm_connect_local(c, world, r, arr), "gsicp_comm_connect_local")
    return comms


def _run_ranks(world, fn):
    out, err = [None] * world, [None] * world

    def work(r):
        try:
            torch.cuda.set_device(0)
            out[r] = fn(r)
        except Exception as ex:  # surface in the main thread
            err[r] = ex

    th = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join(timeout=100)
    for e in err:
        if e is not None:
            raise e
    assert all(o is not None for o in out), "a rank did not finish"
    return out


def _two_ranks_match_single(host_lm, n_trackable=None):
    import gs_icp_slam_b200  # noqa: F401  (registers the drop-in module names)
    import pygicp
    from gs_icp_slam_b200._lib import lib

    if n_trackable is None:
        tgt, src, T = S.gicp_pair(30000, 20000, 60, 61)
        trk = np.arange(0, len(src), 3)  # a trackable subset: covariance slots differ from point indices
        corr_dist = 0.05
    else:
        tgt, src, T = S.gicp_pair(150000, 150000, 62, 63, 0.001, scale=2.0)
        trk = np.arange(n_trackable)
        corr_dist = 0.1
    filt_t = np.arange(1, len(tgt) + 1, dtype=np.int32)
    filt_s = S.trackable_filter(len(src), trk)

    def make():
        r = pygicp.FastGICP()
        r.set_max_correspondence_distance(corr_dist)
        r.set_max_knn_distance(99999)
        r.set_host_lm(host_lm)
        return r

    def align(r, comm, stream):
        if stream is not None:
            r.set_stream(stream.cuda_stream)
        if comm is not None:
            r.set_comm(comm)
        r.set_input_target(tgt)
        r.set_target_filter(len(tgt), filt_t)
        r.calculate_target_covariance_with_filter()
        res = []
        for guess in (np.eye(4), np.array(T) + 2e-3):
            r.set_input_source(src)
            r.set_source_filter(len(trk), filt_s)
            pose = r.align(guess.astype(np.float32))
            res.append((pose, r.last_iterations, r.get_source_correspondence(), r.get_source_rotationsq(), r.get_source_scales(),
                        r.get_final_hessian()))
        if comm is not None:
            r.set_comm(None)
        return res

    cuda = torch.device("cuda", 0)
    single = align(make(), None, None)
    comms = _group(2)
    try:
        streams = [torch.cuda.Stream(device=cuda) for _ in range(2)]
        regs = [make() for _ in range(2)]
        for r in range(2):  # unsharded pass on the rank's own stream: every buffer exists before a peer can spin
            warm = align(regs[r], None, streams[r])
            assert np.array_equal(warm[1][0], single[1][0])
        torch.cuda.synchronize()
        ranks = _run_ranks(2, lambda r: align(regs[r], comms[r], streams[r]))
    finally:
        torch.cuda.synchronize()
        for c in comms:
            lib.gsicp_comm_destroy(c)
    for res in ranks:
        for a, b in zip(res, single):
            assert a[1] == b[1], (a[1], b[1])
            assert np.abs(a[0].astype(np.float64) - b[0]).max() <= 1e-6
            assert np.array_equal(a[2][0], b[2][0]) and np.array_equal(a[2][1], b[2][1])
            assert np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4])
            assert np.abs(a[5] - b[5]).max() <= 1e-9 * np.abs(b[5]).max()
    # both ranks hold bit-identical poses (the redundant LM decisions stayed in lock step)
    assert np.array_equal(ranks[0][0][0], ranks[1][0][0]) and np.array_equal(ranks[0][1][0], ranks[1][1][0])



def test_two_ranks_on_one_gpu_match_single(cuda):
    """Both LM drivers (persistent kernel with in-kernel exchange; host-driven kernels with the exchange in the last block) in
    ONE child process (a hang there cannot take the pytest process and its CUDA context with it).  The third case has
    131 073 trackable source points: rank 0's shard (65 537) lies above kLmPersistentMax and rank 1's (65 536) does not,
    and both ranks must still run the same LM driver."""
    env = dict(os.environ)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env["PYTHONPATH"] = root + os.pathsep + env.get("PYTHONPATH", "")
    p = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=root, capture_output=True, text=True, timeout=150)
    ok = all(f"EXCHANGE-OK {case}" in p.stdout for case in ("False", "True", "131073"))
    assert p.returncode == 0 and ok, p.stdout[-2000:] + p.stderr[-4000:]


if __name__ == "__main__":
    import time

    t0 = time.time()
    from gs_icp_slam_b200._lib import check, lib as _l

    torch.cuda.init()
    torch.zeros(1, device="cuda")
    check(_l.gsicp_test_preload_kernels(), "gsicp_test_preload_kernels")
    print("child: CUDA ready after %.1f s (CUDA_MODULE_LOADING=%s)" % (time.time() - t0, os.environ.get("CUDA_MODULE_LOADING", "default")), flush=True)
    for host_lm in (False, True):
        _two_ranks_match_single(host_lm)
        print("EXCHANGE-OK", host_lm, "at %.1f s" % (time.time() - t0), flush=True)
    _two_ranks_match_single(False, n_trackable=131073)
    print("EXCHANGE-OK 131073 at %.1f s" % (time.time() - t0), flush=True)
