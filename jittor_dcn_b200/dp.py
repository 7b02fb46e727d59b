"""Data-parallel plumbing for the DeformConv2d path (SURVEY.md 8e).

The path shards only along the batch: rank r of g takes samples [r*B/g, (r+1)*B/g), weights
are replicated, and a training step ends with ONE all-reduce of a flat float32 bucket holding
every parameter gradient (DCN weight/bias, offset-conv weight/bias, the host model's other
parameters).  On CUDA the all-reduce is `dcn_allreduce_sum_f32` of the C ABI (NCCL over
NVLink, dlopen'ed); `torch.distributed` is used for rendez-vous only.  With a gloo process
group (CPU tests of this host logic) the same bucket goes through `dist.all_reduce`.
"""
import ctypes

import torch
import torch.distributed as dist

from . import _lib
from .functional import _run


def shard_range(global_batch, rank, world):
    """[begin, end) of the samples rank `rank` owns; the shards tile the batch exactly."""
    if world <= 0 or not 0 <= rank < world:
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, rem = divmod(global_batch, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


class GradBucket:
    """One contiguous float32 buffer aliasing-free copy of all gradients, in parameter order."""

    def __init__(self, params):
        self.params = [p for p in params if p.requires_grad]
        self.sizes = [p.numel() for p in self.params]
        self.numel = sum(self.sizes)
        dev = self.params[0].device if self.params else torch.device("cpu")
        # padded to a multiple of 4 floats: the peer-memory all-reduce walks the bucket in 16-byte pieces
        self._store = torch.zeros((self.numel + 3) // 4 * 4, dtype=torch.float32, device=dev)
        self.flat = self._store[:self.numel]

    def pack(self):
        off = 0
        for p, n in zip(self.params, self.sizes):
            if p.grad is None:
                self.flat[off:off + n].zero_()
            else:
                self.flat[off:off + n].copy_(p.grad.reshape(-1))
            off += n
        return self.flat

    def unpack(self):
        off = 0
        for p, n in zip(self.params, self.sizes):
            g = self.flat[off:off + n].view_as(p)
            if p.grad is None:
                p.grad = g.clone()
            else:
                p.grad.copy_(g)
            off += n


class DcnComm:
    """NCCL communicator behind the C ABI (dcn_comm_*); one per process = one per GPU."""

    def __init__(self, rank, world, device):
        lib = _lib.load()
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = ctypes.create_string_buffer(128)
            _lib.check(lib.dcn_comm_unique_id(buf), "dcn_comm_unique_id")
            uid = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
        uid = uid.to(device)
        dist.broadcast(uid, 0)          # rendez-vous over the existing process group
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(device):
            _lib.check(lib.dcn_comm_init(rank, world, bytes(uid.cpu().numpy().tobytes()),
                                         ctypes.byref(self.handle)), "dcn_comm_init")
        self.world, self.device, self.lib = world, device, lib

    def allreduce_mean_(self, flat):
        """flat <- mean over ranks (equal shards; see allreduce_gradients for uneven ones)."""
        return self.allreduce_sum_(flat, 1.0 / self.world)

    def allreduce_sum_(self, flat, scale=1.0):
        """flat <- scale * sum over ranks, in place, on the current stream (capturable in a CUDA graph)."""
        _run("dcn_allreduce_sum_f32", self.device, None, (self.handle, flat, flat.numel(), float(scale)))
        return flat

    def close(self):
        if self.handle:
            self.lib.dcn_comm_destroy(self.handle)
            self.handle = ctypes.c_void_p()


class DcnP2P:
    """The same exchange as ONE kernel over NVLink peer memory (dcn_p2p_* of the C ABI, csrc/dcn_p2p.cu): every
    rank publishes its bucket in a CUDA-IPC buffer and sums all copies itself.  No NCCL call on the hot path, and —
    unlike a captured NCCL collective — nothing in it that a CUDA graph of the training step cannot replay.
    `torch.distributed` only carries the 64-byte IPC handles once, at construction."""

    def __init__(self, rank, world, device, max_floats):
        lib = _lib.load()
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(device):
            _lib.check(lib.dcn_p2p_create(rank, world, int(max_floats), ctypes.byref(self.handle)), "dcn_p2p_create")
            n = int(lib.dcn_p2p_handle_bytes())
            buf = ctypes.create_string_buffer(n)
            _lib.check(lib.dcn_p2p_local_handle(self.handle, buf), "dcn_p2p_local_handle")
            mine = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone()
            on_dev = dist.get_backend() == "nccl"
            mine = mine.to(device) if on_dev else mine
            every = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            blob = b"".join(bytes(t.cpu().numpy().tobytes()) for t in every)
            _lib.check(lib.dcn_p2p_connect(self.handle, blob), "dcn_p2p_connect")
        dist.barrier()
        self.world, self.device, self.lib = world, device, lib

    def allreduce_mean_(self, flat):
        return self.allreduce_sum_(flat, 1.0 / self.world)

    def allreduce_sum_(self, flat, scale=1.0):
        _run("dcn_p2p_allreduce_sum_f32", self.device, None, (self.handle, flat, flat.numel(), float(scale)))
        return flat

    def close(self):
        if self.handle:
            self.lib.dcn_p2p_destroy(self.handle)
            self.handle = ctypes.c_void_p()


def shard_weight(global_batch, rank, world):
    """Weight of rank `rank`'s gradients in the global-batch gradient: B_local / B_global.  Every rank's loss is
    the MEAN over its own shard, so the global-batch mean is sum_r (B_r / B) * grad_r; only for equal shards is
    that the plain average 1 / world."""
    b, e = shard_range(global_batch, rank, world)
    return (e - b) / float(global_batch)


def allreduce_gradients(bucket, comm=None, group=None, weight=None):
    """Combine the gradients of `bucket.params` over all ranks with ONE collective.

    weight = None: plain average (equal shards).  weight = shard_weight(B, rank, world): each rank's
    per-shard-mean gradients are scaled by B_local / B_global before the sum, which reproduces the single-process
    gradient of the global-batch mean loss for ANY split (uneven shards, B % world != 0).
    BatchNorm batch statistics stay per rank, as in the reference (no SyncBN, train.py:146-159)."""
    flat = bucket.pack()
    if weight is not None:
        flat.mul_(float(weight))
    if comm is not None:
        comm.allreduce_sum_(flat, 1.0 if weight is not None else 1.0 / comm.world)
    else:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        if weight is None:
            flat.mul_(1.0 / dist.get_world_size(group))
    bucket.unpack()
    return flat
