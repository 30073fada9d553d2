"""Multi-GPU plumbing for the hot path (SURVEY.md §8e): one process per GPU, rays sharded, the neural
point cloud / occupancy grid / weights / reference images replicated, one NCCL all-reduce of the
gradients per training step.  Rendering needs no collective at all (frames / ray blocks are
independent units).

The reference has no multi-GPU path (its querier owns one pycuda context, SURVEY.md §2.3); this is new.

Semantics preserved on every replica:
  * the loss of the reference is a MEAN over the ray-masked rays of the whole batch
    (models/base_rendering_model.py:1114-1118), so a rank's gradients are scaled by
    n_local_valid / n_global_valid before the SUM all-reduce (device-side, no host sync);
  * dense Adam (every point row is updated every step, zero gradients still decay the moments):
    point-attribute gradients are all-reduced DENSE, so each replica applies the identical update.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def shard_patches(n_rays: int, rays_per_patch: int, rank: int, world: int) -> Tuple[int, int]:
    """contiguous [begin, end) ray range of `rank`; whole patches only (the blur module and
    drop_patch_rays work on whole 8x8 patches).  Earlier ranks get the remainder patches."""
    assert n_rays % rays_per_patch == 0, "ray count must be a whole number of patches"
    n_patch = n_rays // rays_per_patch
    base, rem = divmod(n_patch, world)
    p0 = rank * base + min(rank, rem)
    p1 = p0 + base + (1 if rank < rem else 0)
    return p0 * rays_per_patch, p1 * rays_per_patch


def shard_patch_rows(patch_num: int, patch_size: int, rank: int, world: int) -> Tuple[int, int]:
    """[begin, end) ray range of `rank` for a training frame whose rays are the raster of a (patch_num*patch_size)^2 pixel grid
    (data/scannet_ft_dataset.py:917-945): whole ROWS of patches, i.e. multiples of patch_size * S consecutive rays, so that
    every 8x8 patch stays on one rank (a contiguous 64-ray range of the raster is one pixel row of 8 different patches)."""
    S = patch_num * patch_size
    r0, r1 = shard_patches(patch_num * patch_size * S, patch_size * S, rank, world)
    return r0, r1


def shard_frame(frame: Dict[str, torch.Tensor], rank: int, world: int, rays_per_patch: int = 64) -> Dict[str, torch.Tensor]:
    """slice the per-ray entries of a frame dict (SURVEY.md Appendix A.1); everything else is replicated.
    Frames that carry the dilated-patch layout (`dilation_PatchNum`, `dilation_PatchSize`) are cut along whole patch rows
    (`shard_patch_rows`); other frames (full-frame rendering) in contiguous multiples of `rays_per_patch` rays."""
    R = frame["raydir"].shape[1]
    PN, PS = frame.get("dilation_PatchNum"), frame.get("dilation_PatchSize")
    if PN is not None and PS is not None and (int(PN) * int(PS)) ** 2 == R:
        b, e = shard_patch_rows(int(PN), int(PS), rank, world)
    else:
        b, e = shard_patches(R, rays_per_patch, rank, world)
    out = dict(frame)
    for k in ("raydir", "gt_image"):
        if k in frame and frame[k] is not None and frame[k].dim() >= 2 and frame[k].shape[1] == R:
            out[k] = frame[k][:, b:e].contiguous()
    pix = frame.get("pixel_idx")
    if pix is not None and torch.is_tensor(pix):
        if pix.dim() == 3 and pix.shape[1] == R:                       # (1,R,2)
            out["pixel_idx"] = pix[:, b:e].contiguous()
        elif pix.dim() == 4 and pix.shape[1] * pix.shape[2] == R:      # (1,S_h,S_w,2) as the dataset / FrameProducer hand it over
            out["pixel_idx"] = pix.reshape(pix.shape[0], R, 2)[:, b:e].contiguous()
    return out


def _flatten(tensors: Sequence[torch.Tensor]) -> torch.Tensor:
    return torch.cat([t.reshape(-1) for t in tensors]) if len(tensors) else torch.empty(0)


def _unflatten_into(flat: torch.Tensor, tensors: Sequence[torch.Tensor]) -> None:
    off, views = 0, []
    for t in tensors:
        n = t.numel()
        views.append(flat[off:off + n].view_as(t))
        off += n
    if views:
        torch._foreach_copy_(list(tensors), views)             # one multi-tensor launch instead of one copy per parameter


def global_mean_scale(n_local_valid: torch.Tensor, group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """(scale, n_global) with scale = n_local / n_global as DEVICE tensors (one scalar all-reduce, no host sync).  Multiplying the
    local loss (a mean over the local ray-masked rays) by `scale` BEFORE backward makes the SUM of the ranks' gradients the
    gradient of the global-mean loss -- without a scaling pass over the 39*N-float point-gradient tables afterwards."""
    n_local = n_local_valid.detach().to(torch.float32).reshape(1)
    n_global = n_local.clone()
    dist.all_reduce(n_global, op=dist.ReduceOp.SUM, group=group)
    return n_local / torch.clamp(n_global, min=1.0), n_global


def allreduce_gradients(params: Iterable[torch.nn.Parameter], n_local_valid: Optional[torch.Tensor] = None, group=None,
                        bucket_bytes: int = 64 << 20, prescaled: bool = False, defer_large: bool = False):
    """SUM all-reduce every gradient: small tensors coalesced into buckets, tensors >= bucket_bytes reduced in place.  Parameters
    whose grad is None on this rank (e.g. it saw no valid ray) take part with zeros so the collective sequence is identical on all
    ranks.  prescaled=False: the gradients are first scaled by n_local/n_global (global-mean normalisation); prescaled=True: the
    caller already scaled its loss with global_mean_scale().  defer_large=True: the in-place reductions of the large tensors are
    launched LAST and returned un-waited as [(work, tensor)] -- the caller overlaps them with whatever does not read those
    gradients (train_step: the MLP optimiser step and the query / pyramid / packing of the next forward).
    Returns n_global (or None when prescaled) and, with defer_large, the pending list."""
    params = [p for p in params if p.requires_grad]
    n_global = None
    if not prescaled:
        scale, n_global = global_mean_scale(n_local_valid, group)
    for p in params:
        if p.grad is None:
            p.grad = torch.zeros_like(p)
        if not prescaled:
            p.grad.mul_(scale.to(p.grad.dtype))
    small = [p.grad for p in params if p.grad.numel() * p.grad.element_size() < bucket_bytes]
    large = [p.grad for p in params if p.grad.numel() * p.grad.element_size() >= bucket_bytes]
    handles = []
    # small gradients first (MLP + conv weights: 449,381 floats = 1.8 MB): their consumer, the MLP optimiser step, is next in line
    bucket, size = [], 0
    def flush():
        nonlocal bucket, size
        if bucket:
            flat = _flatten(bucket)
            handles.append((dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=True), flat, bucket))
            bucket, size = [], 0
    for g in small:
        nb = g.numel() * g.element_size()
        if size + nb > bucket_bytes:
            flush()
        bucket.append(g)
        size += nb
    flush()
    pending = [(dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group, async_op=True), g) for g in large]
    for h, flat, tensors in handles:
        h.wait()
        _unflatten_into(flat, tensors)
    if defer_large:
        return n_global, pending
    for h, _ in pending:
        h.wait()
    return n_global


class PeerBucket:
    """SUM all-reduce of a small set of fp32 gradients through NVLink peer memory (csrc/peer.cu) instead of an NCCL collective: the
    gradients are copied into a symmetric buffer (one multi-tensor launch), a device-side barrier makes every rank's copy visible,
    ONE own kernel per rank reads all copies over NVLink and sums them in rank order (bit-identical on every rank), a second barrier
    releases the buffers.  Plumbing (symmetric allocation, rendezvous, barrier) is torch.distributed._symmetric_memory."""

    def __init__(self, numel: int, device, group=None):
        import torch.distributed._symmetric_memory as symm_mem
        self.n = (int(numel) + 3) // 4 * 4
        self.buf = symm_mem.empty(self.n, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.hdl = symm_mem.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.world = int(self.hdl.world_size)
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        self.multicast = int(getattr(self.hdl, "multicast_ptr", 0) or 0)
        self.out = torch.empty(self.n, dtype=torch.float32, device=device)
        if self.world > 16 or len(self.ptrs) != self.world:
            raise RuntimeError("PeerBucket: unsupported world size")

    def allreduce_(self, grads: Sequence[torch.Tensor], use_multimem: bool = False) -> None:
        """in place: every tensor of `grads` becomes the sum over the ranks"""
        import ctypes as C
        from . import ops
        from ._lib import check, lib, ptr, stream
        views_in, views_out, off = [], [], 0
        for g in grads:
            n = g.numel()
            views_in.append(self.buf[off:off + n].view_as(g))
            views_out.append(self.out[off:off + n].view_as(g))
            off += n
        assert off <= self.n
        torch._foreach_copy_(views_in, list(grads))
        self.hdl.barrier(channel=0)                      # every rank's copy is complete
        with ops._launch(name="peer_sum"):
            if use_multimem and self.multicast:
                check(lib().hnr_multimem_sum_f32(C.c_void_p(self.multicast), self.n, ptr(self.out), stream()), "multimem_sum")
            else:
                arr = (C.c_void_p * self.world)(*self.ptrs)
                check(lib().hnr_peer_sum_f32(arr, self.world, self.n, ptr(self.out), stream()), "peer_sum")
        self.hdl.barrier(channel=1)                      # every rank has read every copy: the buffers may be overwritten
        torch._foreach_copy_(list(grads), views_out)


_PEER_BUCKETS = {}
_PEER_DISABLED = [False]


def peer_bucket(numel: int, device, group=None) -> Optional[PeerBucket]:
    """the PeerBucket for this (group, size), created collectively on first use; None when peer memory cannot be set up on this
    system (no NVLink peer access / non-CUDA backend): the caller then uses an NCCL collective on small_bucket_group()"""
    import os
    if _PEER_DISABLED[0] or os.environ.get("HNR_SMALL_BUCKET", "peer") == "nccl" or torch.device(device).type != "cuda":
        return None
    key = (id(group), int(numel), torch.device(device).index)
    if key not in _PEER_BUCKETS:
        try:
            _PEER_BUCKETS[key] = PeerBucket(numel, device, group)
        except Exception as e:                              # noqa: BLE001 -- any failure here means "not available on this box"
            import warnings
            warnings.warn(f"hybridneuralrendering_b200: NVLink peer-memory all-reduce unavailable ({e!r}); the small gradient bucket uses NCCL")
            _PEER_DISABLED[0] = True
            return None
    return _PEER_BUCKETS[key]


_SMALL_GROUPS = {}


def small_bucket_group(group=None):
    """a SECOND communicator over the same ranks for the small (MLP + conv) gradient bucket.  Collectives of one communicator
    execute in issue order on one stream: on the main group the 1.8 MB bucket would queue behind the 312 MB..1.25 GB point-table
    all-reduce that train_step starts first, and the network's optimiser step (and with it the next forward) would wait for the
    big transfer.  Created collectively on first use (every rank reaches train_step's first call together)."""
    key = id(group)
    if key not in _SMALL_GROUPS:
        ranks = dist.get_process_group_ranks(group) if group is not None else None
        _SMALL_GROUPS[key] = dist.new_group(ranks=ranks)
    return _SMALL_GROUPS[key]


def flush_pending(net) -> None:
    """apply a deferred point-table update now (call before evaluating, checkpointing or pruning / growing points)"""
    cb = getattr(net, "before_point_read", None)
    if cb is not None:
        net.before_point_read = None
        cb()


def train_step(net, frame_shard: Dict[str, torch.Tensor], optimizers: Sequence[torch.optim.Optimizer], group=None,
               zero_one_weight: float = 1e-4, next_frame_shard: Optional[Dict[str, torch.Tensor]] = None, large_bytes: int = 4 << 20,
               timeline: Optional[list] = None):
    """One data-parallel training step on this rank's rays: forward (fused hot path), loss, backward, gradient all-reduce with
    global-mean normalisation, optimiser steps.  Returns (loss, n_global_valid), both device tensors.

    Every rank must hold WHOLE dilated-patch rasters (its own (PN*PS)^2-ray batch, the unit the reference's patch drop and blur
    module work on); the global batch is the union of the ranks' rasters.
    Overlap (world > 1): the loss is pre-scaled by n_local/n_global (no scaling pass over the tables); the in-place all-reduce of
    the point tables (39*N floats) is started as soon as backward has produced them, BEFORE the parked gradient tails (weight
    gradients, image-branch tail: ops.defer_weight_gradients) are issued; the small MLP bucket is reduced on its own communicator
    (small_bucket_group) and its optimiser stepped at once; the all-reduce of the point tables is left in flight
    and the optimiser(s) that own those tables step at the LAST possible moment -- inside the next forward, after its query and
    pyramid but before the first kernel that reads the tables (`net.before_point_read`), or at flush_pending(net).  That deferred
    step consumes the previous step's gradients, so the gradients are zeroed after the forward and flush_pending(net), not before.
    `next_frame_shard`: the shard of the NEXT step, if known -- its voxel query is enqueued before this step's backward pass so
    that the next forward does not stall at the query's read-back (NeuralPointsRayMarching.prefetch_query)."""
    from . import ops
    from .renderer import training_loss
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    opt = getattr(net, "opt", None)

    def mark(name):
        """profiling aid (scripts/dp_timeline.py): a CUDA event on the main stream at this point of the step"""
        if timeline is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            timeline.append((name, ev))
    mark("start")
    if world > 1 and opt is not None and getattr(opt, "is_train", False) and getattr(opt, "drop_ratio", 0) > 0 and getattr(opt, "use_nearest", 0) > 0:
        toks = str(opt.dilation_setup).split("_")
        if frame_shard["raydir"].shape[1] != (int(toks[0]) * int(toks[1])) ** 2:
            raise NotImplementedError("data-parallel training with the patch drop needs whole (PN*PS)^2-ray rasters per rank: the reference's "
                                      "drop positions (point_aggregators.py:1222-1237) index the raster of ONE batch; give every rank its "
                                      "own raster instead of slicing one with shard_frame")
    out = net(**frame_shard)                        # a deferred point update of the previous step is applied inside (before_point_read)
    flush_pending(net)                               # ... or here, if the forward had nothing to read (no kept ray)
    # zeroed only now: the deferred point-table step above reads the previous step's all-reduced gradients, and an optimiser skips a
    # parameter whose grad is None.  The forward produces no gradients, so zeroing after it changes nothing for the other parameters
    for o in optimizers:
        o.zero_grad(set_to_none=True)
    mark("forward_end")
    n_local = (out["ray_mask"] > 0).sum()
    scale = n_global = None
    if world > 1:
        scale, n_global = global_mean_scale(n_local, group)
    if next_frame_shard is not None and getattr(net, "near_far", None) is not None:
        net.prefetch_query(**next_frame_shard)
    # the weight-gradient launches are parked during backward and issued below, AFTER the all-reduce of the point tables has been
    # started: ~1.4 ms of kernels that nothing else waits for cover the collective (ops.defer_weight_gradients)
    with ops.defer_weight_gradients() as deferred:
        if out["coarse_raycolor"].shape[1] > 0:
            loss = training_loss(out, frame_shard["gt_image"], zero_one_weight)
            with ops.tag("backward"):
                (loss * scale[0] if scale is not None else loss).backward()
        else:
            loss = torch.zeros((), device=out["ray_mask"].device)
    mark("backward_end")
    if world == 1:
        with ops.tag("backward"):
            deferred.run()
        mark("tails_end")
        for o in optimizers:
            o.step()
        mark("end")
        return loss.detach(), n_local
    params = [p for o in optimizers for g in o.param_groups for p in g["params"]]
    is_large = lambda p: p.numel() * p.element_size() >= large_bytes
    large_params = [p for p in params if is_large(p)]
    _, pending = allreduce_gradients(large_params, None, group, bucket_bytes=large_bytes, prescaled=True, defer_large=True)
    with ops.tag("backward"):
        deferred.run()
    mark("tails_end")
    small_params = [p for p in params if not is_large(p) and p.requires_grad]
    for p in small_params:
        if p.grad is None:
            p.grad = torch.zeros_like(p)
    pb = peer_bucket(sum(p.numel() for p in small_params), small_params[0].device, group) if small_params else None
    if pb is not None:
        # the network's gradients (1.8 MB): own one-shot all-reduce over NVLink peer memory (csrc/peer.cu)
        import os
        pb.allreduce_([p.grad for p in small_params], use_multimem=os.environ.get("HNR_SMALL_BUCKET") == "multimem")
    else:
        allreduce_gradients(small_params, None, small_bucket_group(group), bucket_bytes=64 << 20, prescaled=True)
    mark("small_bucket_done")
    late = [o for o in optimizers if any(is_large(p) for g in o.param_groups for p in g["params"])]
    for o in optimizers:
        if o not in late:
            o.step()
    mark("end")

    def apply_late():
        mark("late_begin")                           # (inside the NEXT forward: after its packing / pyramid / query)
        for h, _ in pending:
            h.wait()
        mark("late_allreduce_done")
        for o in late:
            o.step()
        mark("late_end")
    if late and hasattr(net, "before_point_read"):
        net.before_point_read = apply_late
    else:
        apply_late()
    return loss.detach(), n_global
