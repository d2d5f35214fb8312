"""Multi-GPU host logic (SURVEY.md §8e): one process per GPU, torch.distributed (NCCL on the GPUs, gloo in the CPU tests).

* rasterizer: screen tiles are interleaved over the ranks (tile % world == rank).  Every rank preprocesses all Gaussians
  but emits / sorts / renders only its own tiles and feeds the image gradients of its own pixels; the per-Gaussian render
  moments of the ranks add up inside gsicp_raster_backward, so every rank ends with the complete parameter gradients.
* GICP: source points are split into contiguous ranges (k-NN covariances and the LM loop); the 28 doubles of the normal
  equations (21 H + 6 b + error) are exchanged at every reduction point.
`ShardGroup` wires both to the library's in-kernel exchange over peer memory (csrc/comm.cuh), which needs CUDA IPC
between the ranks.  The module-level helpers partition pixels (tile_owner_mask, sharded_l1) and source points
(source_range), and sum the gradients of parameters that live outside the library (allreduce_grads).
"""
import torch

TILE = 16


def tile_owner_mask(height, width, world, rank, device="cpu"):
    """float32 [1,H,W]: 1 where the pixel's 16x16 tile belongs to `rank` (tile_id % world == rank)."""
    ty, tx = (height + TILE - 1) // TILE, (width + TILE - 1) // TILE
    tid = torch.arange(ty, device=device)[:, None] * tx + torch.arange(tx, device=device)[None, :]
    own = (tid % world == rank).repeat_interleave(TILE, 0).repeat_interleave(TILE, 1)[:height, :width]
    return own.float()[None]


def source_range(n, world, rank):
    """[begin, end) of the source points rank `rank` linearises — must match shard_range() in csrc/gicp.cu."""
    per = (n + world - 1) // world
    return min(n, per * rank), min(n, per * (rank + 1))


def sharded_l1(pred, target, mask, n_total):
    """sum |pred - target| over the rank's pixels divided by the global element count: the rank's share of a mean L1."""
    return ((pred - target).abs() * mask).sum() / float(n_total)


def allreduce_grads(params, group=None):
    """Sum the .grad of every tensor in `params` over the ranks with ONE collective (flat buffer)."""
    import torch.distributed as dist

    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, group=group)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n


class ShardGroup:
    """One rank's membership of a sharded run: wires the rasterizer (tile shards + render-moment exchange) and FastGICP
    objects (source-point shards for the k-NN covariances and the LM loop + normal-equation exchange) to the exchange layer.

    The exchange group is the library's own (csrc/comm.cuh): every rank allocates a symmetric device segment, the 64-byte
    CUDA IPC handles travel once through torch.distributed.all_gather_object, and from then on the kernels exchange through
    the peers' segments over NVLink with device-side flags: no host-launched collective, no Python in the loop.  The
    constructor is collective; it raises on every rank when the group cannot be set up on all of them."""

    def __init__(self, device, world, rank, group=None, heap_bytes=256 << 20):
        self.device, self.world, self.rank, self.group = device, world, rank, group
        self._gicp = []
        self._raster = False
        self._comm = None
        self._connect(heap_bytes)

    def _connect(self, heap_bytes):
        import ctypes as C

        import torch.distributed as dist

        from ._lib import last_error, lib

        comm = C.c_void_p()
        handle = C.create_string_buffer(64)

        with torch.cuda.device(self.device):
            # a rank whose allocation fails still takes part in the two collectives below, so nobody is left waiting
            alloc_rc = lib.gsicp_comm_alloc(int(heap_bytes), C.byref(comm), handle)
            why = last_error() if alloc_rc != 0 else ""
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle.raw) if alloc_rc == 0 else None, group=self.group)
            ok = all(isinstance(h, (bytes, bytearray)) and len(h) == 64 for h in handles)
            rc = lib.gsicp_comm_connect(comm, self.world, self.rank, b"".join(handles)) if ok else -1
            if ok and rc != 0:
                why = last_error()
            # every rank must agree before anybody relies on the peers' segments
            flag = torch.tensor([1 if rc == 0 else 0], device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
            if int(flag.item()) != 1:
                if alloc_rc == 0:
                    lib.gsicp_comm_destroy(comm)
                raise RuntimeError("exchange group could not be set up on every rank: " + (why or "a peer failed"))
        self._comm = comm

    def attach_rasterizer(self):
        from . import rasterizer

        rasterizer.set_tile_shard(self.world, self.rank)
        rasterizer.set_comm(self._comm)
        self._raster = True

    def attach_gicp(self, reg):
        reg.set_comm(self._comm)
        self._gicp.append(reg)

    def close(self):
        if self._raster:
            from . import rasterizer

            rasterizer.set_tile_shard(1, 0)
            rasterizer.set_comm(None)
            self._raster = False
        for reg in self._gicp:
            try:
                reg.set_comm(None)
            except Exception:
                pass
        self._gicp = []
        if self._comm is not None:
            from ._lib import lib

            torch.cuda.synchronize(self.device)
            if torch.distributed.is_initialized():
                torch.distributed.barrier(group=self.group)  # nobody unmaps while a peer's kernel may still touch the segment
            lib.gsicp_comm_destroy(self._comm)
            self._comm = None
