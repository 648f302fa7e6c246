"""Frame sharding across the GPUs of one box.  One process per GPU; the scene is replicated; the frame is split by image rows or
by sample-index range; ONE reduction of the film accumulators per frame.  The reference has no distributed path (SURVEY.md
section 8e); the only shared output of the hot path is the per-pixel Sensor accumulator (sensor.rs:76-77), so a sum of
accumulators is the whole exchange.

The exchange itself lives INSIDE libtcpt (include/tcpt.h "multi-GPU"): `tcpt_comm_init` makes an NCCL communicator owned by the
context, `tcpt_render_sharded` renders this rank's shard, runs one `ncclReduce` onto rank 0 and hands back one complete frame
there.  torch.distributed is only the plumbing that carries the 128-byte NCCL unique id from rank 0 to the other ranks
(`init_comm`); a host without PyTorch passes the id over any transport it likes.

  mode "tile": rank r renders rows y with y % world == r and ALL samples -> every pixel is summed in the reference's
               sample order on one GPU, other ranks contribute exact zeros: the reduced film is bitwise equal to 1 GPU.
  mode "spp" : rank r renders samples [r*spp/world, (r+1)*spp/world) of every pixel -> best balance; per-pixel float sums are
               re-associated across ranks (tolerance-level equality).

Adaptive frames (`RendererImage.render_adaptive_sharded`, tcpt_render_adaptive_sharded) take tile shards only, one grouped reduce per frame.
"""
from __future__ import annotations

from dataclasses import dataclass


@dataclass
class Shard:
    row_offset: int = 0
    row_stride: int = 0
    spp_begin: int = 0
    spp_end: int = 0

    def as_kwargs(self):
        return dict(row_offset=self.row_offset, row_stride=self.row_stride, spp_begin=self.spp_begin, spp_end=self.spp_end)


def shard_plan(rank: int, world: int, mode: str, spp: int, spp_begin: int = 0, spp_end: int | None = None) -> Shard:
    """The slice of the frame rank `rank` of `world` renders (the rule of tcpt_shard_params, restated for host-side planning and for
    the CPU tests).  [spp_begin, spp_end) restricts the whole job to a sample window."""
    spp_end = spp if spp_end is None else spp_end
    if not (0 <= rank < world) or not (0 <= spp_begin <= spp_end <= spp):
        raise ValueError("bad shard request")
    if mode == "tile":
        return Shard(row_offset=rank, row_stride=world, spp_begin=spp_begin, spp_end=spp_end)
    if mode == "spp":
        n = spp_end - spp_begin
        b = spp_begin + (n * rank) // world
        e = spp_begin + (n * (rank + 1)) // world
        return Shard(row_offset=0, row_stride=0, spp_begin=b, spp_end=e)
    raise ValueError(f"unknown shard mode {mode!r}")


def init_comm(ctx, rank: int | None = None, world: int | None = None) -> None:
    """Give `ctx` (a capi.Context on this rank's GPU) its NCCL communicator.  Collective: every rank calls it.  The unique id is made on
    rank 0 (tcpt_comm_get_unique_id) and carried by torch.distributed's broadcast; everything after that is libtcpt's own NCCL."""
    import torch.distributed as dist
    from . import capi
    if rank is None:
        rank = dist.get_rank() if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size() if dist.is_initialized() else 1
    if world == 1:
        return
    box = [capi.Context.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    ctx.comm_init(world, rank, box[0])


def reduce_film(acc, dst: int = 0, all_ranks: bool = False):
    """Sum film accumulators held in torch tensors over ranks (host-logic tests on gloo / CPU tensors; the GPU path reduces inside
    libtcpt, see render_sharded)."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        return acc
    if all_ranks:
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    else:
        dist.reduce(acc, dst=dst, op=dist.ReduceOp.SUM)
    return acc


def render_sharded(image, sampler, mode: str = "tile", device_acc=None, stream=None, spp_window=None, max_slots: int = 0):
    """Render this rank's shard of `image` (a RendererImage) and reduce to rank 0 through libtcpt's communicator (init_comm first).
    With `device_acc` (a zeroed torch CUDA tensor [H, W, 3] f32) the film stays on the device (tcpt_render_sharded_device) and the
    tensor is returned; without it, rank 0's `image.pixels` / `image.accumulators` receive the complete frame (tcpt_render_sharded)."""
    import ctypes as C

    from . import capi
    if device_acc is None:
        return image.render_sharded(sampler, mode=mode, spp_window=spp_window, max_slots=max_slots)
    import torch
    r = image.renderer
    ctx = r.args.scene.ctx
    kw = {"spp_begin": spp_window[0], "spp_end": spp_window[1]} if spp_window else {}
    p = r.params(sampler, max_slots=max_slots, **kw)
    s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
    ctx.check(ctx.lib.tcpt_render_sharded_device(ctx.handle, C.byref(p), capi.SHARD_MODES[mode], C.c_void_p(device_acc.data_ptr()), C.c_void_p(s)))
    image.stats = ctx.stats()
    return device_acc
