"""Multi-GPU plumbing for the renderer: one process per GPU (``torchrun``), the batch of views
sharded across ranks, NCCL all-reduce ONLY for gradients of tensors shared by every view.

The reference has nothing here ("multiple GPUs" in its README means ``--gpu N``,
``examples_pytorch/example1.py:46-47``).  The path shards trivially: every view is independent in
the forward pass and in the per-view backward pass, so there is no data-path collective.  The one
real exchange is multi-view optimisation of ONE mesh / texture (``examples_pytorch/example2.py``):
the parameter is expanded to the local views, its gradient is summed over them on the device and
then summed over ranks (12*nv bytes for vertices, 12*T for textures).

Works with any ``torch.distributed`` backend: ``nccl`` on the B200 box, ``gloo`` in the CPU tests.
"""
import torch
import torch.distributed as dist


def world():
    """(rank, world_size) of the default process group, (0, 1) when not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(num_views, rank=None, world_size=None):
    """Contiguous, balanced [begin, end) slice of ``num_views`` owned by ``rank``.
    The first ``num_views % world_size`` ranks get one extra view."""
    if rank is None or world_size is None:
        rank, world_size = world()
    base, extra = divmod(num_views, world_size)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def shard_views(tensor, rank=None, world_size=None):
    """Slice dim 0 (views) of ``tensor`` for this rank.  Per-view faces [B, nf, 3] are sharded like the vertices."""
    b, e = shard_range(tensor.shape[0], rank, world_size)
    return tensor[b:e]


class _ShareAcrossViews(torch.autograd.Function):
    """[1, ...] parameter -> [views, ...] expanded view; backward sums the gradient over the local
    views and all-reduces it over ranks so every rank holds the full multi-view gradient."""

    @staticmethod
    def forward(ctx, param, views, group):
        ctx.group = group
        return param.expand(views, *param.shape[1:])

    @staticmethod
    def backward(ctx, grad):
        g = grad.sum(0, keepdim=True).contiguous()
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(ctx.group) > 1:
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=ctx.group)
        return g, None, None


def share_across_views(param, local_views, group=None):
    """Use one mesh / texture ``param`` of shape [1, ...] for ``local_views`` views on this rank.
    After ``backward()`` ``param.grad`` is identical on every rank: the sum over ALL views of the job."""
    assert param.shape[0] == 1, "shared parameter must have a leading dimension of 1"
    return _ShareAcrossViews.apply(param, local_views, group)


class _Exchange:
    """Symmetric-memory exchange buffers for the fused camera-backward + all-reduce kernel
    (csrc/nr_camera.cu: k_camera_backward_shared_exchange): every rank maps every rank's buffer over NVLink."""

    _cache = {}

    def __init__(self, nv, group, device):
        import ctypes
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        L = _lib.lib()
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        nbytes = L.nr_camera_exchange_bytes(nv, self.world)
        if nbytes <= 0:
            raise RuntimeError("mesh too large for the exchange buffer")
        self.nv = nv
        self.buffer = symm.empty((nbytes + 3) // 4, dtype=torch.int32, device=device)
        self.buffer.zero_()
        self.handle = symm.rendezvous(self.buffer, group if group is not None else dist.group.WORLD)
        self.pointers = (ctypes.c_void_p * self.world)(*[int(p) for p in self.handle.buffer_ptrs])
        self.epoch = torch.zeros(4, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group)                 # every rank's buffer is zeroed before anybody's first exchange

    @classmethod
    def get(cls, nv, group, device):
        """The exchange of (group, mesh size, device), or None when peer memory cannot be set up (then NCCL)."""
        key = (id(group) if group is not None else 0, nv, str(device))
        if key not in cls._cache:
            try:
                cls._cache[key] = cls(nv, group, device)
            except Exception as e:          # no symmetric memory on this system / backend: the NCCL path stays
                import warnings
                warnings.warn("fused all-reduce over peer memory unavailable (%s: %s); using %s all_reduce"
                              % (type(e).__name__, e, dist.get_backend(group)))
                cls._cache[key] = None
        return cls._cache[key]


# The fused exchange is a collective every rank must enter the same number of times.  Measured on one 8-GPU
# B200 box (config 3, profiles/r2_scaling_cfg3.jsonl): 0.171 / 0.181 / 0.204 ms per step on 2 / 4 / 8 GPUs against
# 0.216 ms with ncclAllReduce inside the captured step on 8, and the sum is bit-identical on every rank: it is the
# default up to FUSED_MAX_WORLD ranks (the kernel's peer table).  NR_FUSED_ALLREDUCE=0 keeps the NCCL all-reduce.
_FUSED_ENV = __import__("os").environ.get("NR_FUSED_ALLREDUCE")
FUSED_ALLREDUCE = _FUSED_ENV != "0"
FUSED_MAX_WORLD = 16


def fused_allowed(world_size):
    return FUSED_ALLREDUCE and world_size <= FUSED_MAX_WORLD


class _ShareAcrossRanks(torch.autograd.Function):
    """Identity; the backward sums the gradient over the ranks (in place, on the stream of the backward, so a
    captured step replays the collective too)."""

    @staticmethod
    def forward(ctx, param, group):
        ctx.group = group
        return param.view_as(param)

    @staticmethod
    def backward(ctx, grad):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(ctx.group) > 1:
            grad = grad.contiguous()
            dist.all_reduce(grad, op=dist.ReduceOp.SUM, group=ctx.group)
        return grad, None


def share_across_ranks(param, group=None):
    """Mark ``param`` (e.g. ONE mesh [1,nv,3] handed to ``Renderer.render*`` with per-view ``viewpoints`` [B,3]:
    the fused camera transform projects it into the local views and sums its gradient over them) as shared by
    every rank: after ``backward()`` ``param.grad`` is the sum over ALL views of the job, identical on every
    rank.  The all-reduce moves 12*nv bytes (vertices) or 12*T (textures) per step.

    A [1,nv,3] CUDA mesh that goes into the fused camera transform (``Renderer.transform_vertices``) does not
    even see a separate all-reduce: its camera-backward kernel exchanges the gradient slices with the peer GPUs
    over NVLink itself (``_Exchange``), in rank order, so the result is bit-identical on every rank."""
    out = _ShareAcrossRanks.apply(param, group)
    if (param.is_cuda and param.ndim == 3 and param.shape[0] == 1 and param.shape[2] == 3
            and dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
            and fused_allowed(dist.get_world_size(group)) and dist.get_backend(group) == "nccl"):
        # camera.transform_vertices takes `param` itself as its autograd input when it fuses the exchange, so
        # this node only reduces what OTHER consumers of `out` send back
        out._nr_shared = (param, group)
    return out


def allreduce_shared_grads(params, group=None):
    """Sum ``p.grad`` over ranks for parameters that every rank holds a replica of (when they were
    not routed through :func:`share_across_views`)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    for p in params:
        if p.grad is not None:
            dist.all_reduce(p.grad, op=dist.ReduceOp.SUM, group=group)


def gather_images(local_images, group=None):
    """All-gather per-rank image batches (equal local batch on every rank) into the global batch
    in rank order.  Not on the training path; for inspection / evaluation."""
    rank, ws = world()
    if ws == 1:
        return local_images
    out = [torch.empty_like(local_images) for _ in range(ws)]
    dist.all_gather(out, local_images.contiguous(), group=group)
    return torch.cat(out, 0)
