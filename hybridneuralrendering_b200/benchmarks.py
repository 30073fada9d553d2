"""Benchmark bodies shared by bench.py and scripts/: the training step of BASELINE.json configs[2]
(ScanNet scene0241_01-shaped hybrid training step: 640x480 frames, 4096-ray batch = 8x8 dilated patches of 8x8,
V=8 reference-view feature maps, 2M neural points, SR=24, K=8) on synthetic data."""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch

from . import ops

TRAIN_WORKLOAD = "ScanNet scene0241_01-shaped hybrid training step: 640x480 frames, 4096-ray batch, 8 reference-view feature maps, 2M points"


FRAME_SET = 8          # distinct frames a training benchmark cycles through (see train_step_benchmark)

LARGE_WORKLOAD = "large-scale scene: 8M neural points, 1296x968 frames, 4096-ray rasters sharded across the GPUs with NCCL gradient allreduce over NVLink"


def build_train_case(dev, points: int = 2_000_000, views: int = 8, seed: int = 0, size=(6.0, 5.0, 3.0), H: int = 480, W: int = 640,
                     max_o: int = 1_000_000, n_frames: int = 1):
    """net + frame of a training step: room-shaped point cloud (replicated: the same on every rank), 4096-ray dilated-patch
    rasters (8x8 patches of 8x8; the seed moves the camera and the patches).  n_frames > 1: returns a LIST of frames with seeds
    seed, seed + 1, ... -- a training loop sees a different frame every step."""
    from . import NeuralPoints, NeuralPointsRayMarching, PointAggregator, make_opt
    from . import synthetic as syn
    opt = make_opt("scannet", use_nearest=views, SR=24, is_train=True, drop_ratio=0.5, dilation_setup="8_8_1_8",
                   max_o=max_o)           # >= occupied voxels of the room (SURVEY.md §8d: generator must respect max_o)
    xyz = syn.room_scene(points, 0, size=size)
    att = syn.point_attributes(np.random.default_rng(0), len(xyz))
    c = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    pts = NeuralPoints(32, len(xyz), opt, dev)
    pts.set_points(c(xyz), c(att["emb"])[None], points_color=c(att["color"])[None], points_dir=c(att["dir"])[None],
                   points_conf=c(att["conf"])[None], parameter=True)
    torch.manual_seed(0)
    agg = PointAggregator(opt).to(dev)
    net = NeuralPointsRayMarching(aggregator=agg, neural_points=pts, opt=opt).to(dev)
    net.near_far = (0.1, 8.0)
    frames = []
    for i in range(n_frames):
        fr = syn.room_frame(H=H, W=W, V=views, patch_num=8, patch_size=8, seed=seed + i, size=size)
        frames.append({k: (c(v) if isinstance(v, np.ndarray) and v.dtype.kind == "f" else v) for k, v in fr.items()})
    return net, (frames[0] if n_frames == 1 else frames)


def make_optimizers(net):
    """the reference's two Adam groups (mvs_points_volumetric_model.py:94-104: network lr 5e-4, point parameters lr 2e-3), each stepped
    by ONE multi-tensor launch (optim.FusedAdam)"""
    from .optim import FusedAdam
    opt_net = FusedAdam([p for n, p in net.named_parameters() if p.requires_grad and not n.startswith("neural_points.")], lr=5e-4)
    opt_pts = FusedAdam([p for n, p in net.named_parameters() if p.requires_grad and n.startswith("neural_points.")], lr=2e-3)
    return [opt_net, opt_pts]


def _device_max(ms: float, dev, world: int) -> float:
    import torch.distributed as dist
    if world <= 1:
        return ms
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def train_step_benchmark(dev, steps: int = 5, warmup: int = 3, world: int = 1, points: int = 2_000_000, views: int = 8,
                         rank: int = 0, stage_split: bool = True, prefetch: bool = True, size=(6.0, 5.0, 3.0), H: int = 480, W: int = 640,
                         max_o: int = 1_000_000, e2e: bool = True, workload: str = TRAIN_WORKLOAD, capture=None) -> Dict:
    """One training step = forward + loss + backward (+ NCCL gradient all-reduce when world > 1) + both Adam steps, through
    parallel.train_step, on this rank's own 4096-ray raster; the next step's voxel query is software-pipelined one step ahead
    (`prefetch`).  `steps` steps are timed as ONE region between barriers (CUDA events, L2 flushed between steps), max over ranks.
    `capture(net, loss, n_valid)`, if given, is called once after the timed steps, before any later step changes the model, with
    what the last timed step returned and the model it updated.
    Returns a dict; 'value' = rays of ALL ranks / that time."""
    import torch.distributed as dist
    from . import parallel
    # FRAME_SET distinct frames (camera pose, patch positions, reference views), the same set on every rank; rank r trains on frame
    # (r + step) % FRAME_SET: every step all ranks hold different rasters (as a data-parallel loader would hand them out), and over a run
    # every rank -- and the 1-GPU run -- sees the same mix of light and heavy frames (75 k .. 83 k valid samples per 4096 rays)
    net, frames = build_train_case(dev, points, views, seed=0, size=size, H=H, W=W, max_o=max_o, n_frames=FRAME_SET)
    frame = frames[rank % FRAME_SET]
    agg = net.aggregator
    R = frame["raydir"].shape[1]
    opts = make_optimizers(net)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    it = [0]

    def next_pair():
        """(frame of this step, frame of the next step)"""
        i = it[0]
        it[0] += 1
        return frames[(rank + i) % FRAME_SET], frames[(rank + i + 1) % FRAME_SET]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # at least one pass over the whole frame set: every frame has its own valid-sample count, i.e. its own activation sizes, and the
    # caching allocator serves a new size with a cudaMalloc (a device synchronisation) the first time it sees it.
    # The barrier comes BEFORE the last warm-up step: the timed region then starts behind issued work, as every step of a training
    # run does, and not on an idle device that waits for the host to issue its first launches (a fixed gap that a window of few
    # steps would count as step time)
    for _ in range(max(warmup, FRAME_SET + 1) - 1):
        cur, nx = next_pair()
        parallel.train_step(net, cur, opts, next_frame_shard=nx if prefetch else None)
    parallel.flush_pending(net)
    barrier()
    cur, nx = next_pair()
    parallel.train_step(net, cur, opts, next_frame_shard=nx if prefetch else None)
    parallel.flush_pending(net)
    ops.LAUNCHES = 0
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    import time as _time
    s.record()
    t_host = _time.perf_counter()
    for _ in range(steps):
        flush.zero_()
        cur, nx = next_pair()
        loss, n_valid = parallel.train_step(net, cur, opts, next_frame_shard=nx if prefetch else None)
    parallel.flush_pending(net)
    e.record()
    host_ms = (_time.perf_counter() - t_host) / steps * 1e3           # time the HOST needs to issue a step (no synchronisation in the loop)
    barrier()
    launches = ops.LAUNCHES
    ms_local = s.elapsed_time(e) / steps
    ms_step = _device_max(ms_local, dev, world)
    if capture is not None:
        capture(net, loss, n_valid)
    res = {"metric": "train rays/s (fwd+bwd)", "value": world * R / (ms_step * 1e-3), "unit": "rays/s", "ms_per_step": ms_step,
           "rays_per_step_per_gpu": R, "points": points, "views": views, "loss": float(loss), "launches_per_step": launches // steps,
           "host_issue_ms_per_step": host_ms, "frame_set": FRAME_SET,
           "step": "forward + loss + backward" + (" + NCCL gradient all-reduce" if world > 1 else "") + " + Adam (network + point tables)",
           "config": workload}
    nxt = frame if prefetch else None
    # ---- end to end: the frame dict arrives in pinned host memory every step, the loss goes back to the host every step
    if e2e:
        hosts = [{k: v.cpu().pin_memory() for k, v in f.items() if torch.is_tensor(v)} for f in frames]
        rest = {k: v for k, v in frame.items() if not torch.is_tensor(v)}
        host = hosts[0]
        # the timed steps of this loop train on the SAME frames, in the same order, as the timed steps of the resident loop above (the
        # frames differ by +-5 % in valid samples; two warm-up steps precede the timed ones here)
        cnt = [max(warmup, FRAME_SET + 1) - 2]

        # double-buffered loader, as a training loop would run it: the host->device copy of a frame is issued on a copy stream one step
        # BEFORE the step that first touches it (its query is prefetched during the previous step), so the 29.6 MB transfer overlaps
        # with compute; every step still copies one whole frame dict inside the timed region
        copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream()

        def up():
            h = hosts[(rank + cnt[0]) % FRAME_SET]
            cnt[0] += 1
            with torch.cuda.stream(copy_stream):
                d = {k: v.to(dev, non_blocking=True) for k, v in h.items()}
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            for t in d.values():
                t.record_stream(main)
            return dict(rest, **d), ev

        def use(fe):
            main.wait_event(fe[1])
            return fe[0]
        loss_host = torch.zeros(steps + 2).pin_memory()
        cur = use(up())
        nxt_fe = up()
        def warm_step():
            nonlocal cur, nxt_fe
            n2 = use(nxt_fe)
            nxt_fe = up()                               # two steps ahead of its first use on the main stream
            parallel.train_step(net, cur, opts, next_frame_shard=n2 if prefetch else None)
            cur = n2
        warm_step()
        parallel.flush_pending(net)
        barrier()
        warm_step()                                     # as above: the timed region starts behind the last warm-up step's work
        parallel.flush_pending(net)
        s.record()
        for i in range(steps):
            flush.zero_()
            n2 = use(nxt_fe)                            # the NEXT step's frame (its query is launched before this step's backward)
            nxt_fe = up()
            loss, _ = parallel.train_step(net, cur, opts, next_frame_shard=n2 if prefetch else None)
            loss_host[i:i + 1].copy_(loss.reshape(1), non_blocking=True)
            cur = n2
        parallel.flush_pending(net)
        e.record()
        barrier()
        ms_e2e = _device_max(s.elapsed_time(e) / steps, dev, world)
        res["e2e"] = {"value": world * R / (ms_e2e * 1e-3), "unit": "rays/s", "ms_per_step": ms_e2e,
                      "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host.values())), "d2h_bytes_per_step": 4 + 8,
                      "what": "frame dict (rays, ground truth, camera, 8 reference views) copied from pinned host memory every step on a copy stream "
                              "(double-buffered loader: issued one step before its first use); loss and the query's two counts read back every step"}
    # ---- where the time goes: per-launch CUDA events of one more step (world == 1 only: the timers serialise nothing but add events)
    stages = {}
    if stage_split:
        barrier()
        ops.TIMERS = []
        ops.SIDE_LANE = False                 # per-kernel times: nothing runs beside the kernel being timed
        with ops.tag("step"):
            parallel.train_step(net, frame, opts, next_frame_shard=nxt)
        parallel.flush_pending(net)
        ops.SIDE_LANE = True
        torch.cuda.synchronize()
        for tg, a, b in ops.TIMERS:
            tg = tg.split("[")[0]
            stages[tg] = stages.get(tg, 0.0) + a.elapsed_time(b)
        ops.TIMERS = None
    # forward + backward alone (no optimiser), for continuity with round 1's "ms_fwd_bwd"
    from .renderer import training_loss
    params = [p for p in net.parameters() if p.requires_grad]

    def fwd_bwd():
        for p in params:
            p.grad = None
        out = net(**frame)
        l = training_loss(out, frame["gt_image"])
        if prefetch:
            net.prefetch_query(**frame)
        # as parallel.train_step issues it: the gradient tails (weight gradients, image-branch tail) parked during backward and run on
        # two streams afterwards
        with ops.defer_weight_gradients() as deferred:
            l.backward()
        deferred.run()
    for _ in range(2):
        fwd_bwd()
    barrier()
    s.record()
    for _ in range(steps):
        flush.zero_()
        fwd_bwd()
    e.record()
    barrier()
    res["ms_fwd_bwd"] = s.elapsed_time(e) / steps
    ex = net.last_extras
    res.update({"kept_rays": int(ex.n_rays), "valid_samples": int(ex.n_valid), "valid_neighbours": agg.last_valid_neighbours(),
                "stage_ms": {k: round(v, 3) for k, v in sorted(stages.items())}})
    if world > 1:
        # per-rank view (every rank trains on its own raster: the slowest rank sets the step time) and the same step WITHOUT the
        # gradient exchange, so that the exposed cost of the collective can be read off
        for _ in range(2):
            fwd_bwd()
        barrier()
        mine = {"rank": rank, "ms_step_local": round(ms_local, 3), "host_issue_ms_per_step": round(host_ms, 3), "ms_fwd_bwd_no_collective": round(res["ms_fwd_bwd"], 3), "valid_samples": int(ex.n_valid)}
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        res["ranks"] = allr
    return res


BLUR_WORKLOAD = "full model with blur handling: 32x32 patch rays (4x4 dilated patches of 8x8) + pre-defined degradation-kernel convolution, fwd+bwd"


def blur_train_step_benchmark(dev, steps: int = 5, warmup: int = 3, points: int = 2_000_000, views: int = 8, learnable: bool = False) -> Dict:
    """BASELINE.json configs[3]: as the training step, but 1,024 rays on a 4x4 grid of 8x8 patches, the output filled back to
    the patch raster and passed through the blur module (36 pre-defined 9x9 kernels + identity, per-patch best match,
    models/base_rendering_model.py:677-786) before the loss; forward + backward through blur and render."""
    from . import NeuralPoints, NeuralPointsRayMarching, PointAggregator, make_opt
    from . import synthetic as syn
    from .blur import blur_select, learnable_blur, predefined_blur_kernels
    from .neural_points_volumetric_model import fill_invalid
    opt = make_opt("scannet", use_nearest=views, SR=24, is_train=True, drop_ratio=0.5, dilation_setup="4_8_1_8", max_o=1_000_000,
                   learnable_blur_kernel=int(learnable), boundary_mode=1)
    xyz = syn.room_scene(points, 0)
    att = syn.point_attributes(np.random.default_rng(0), len(xyz))
    fr = syn.room_frame(H=480, W=640, V=views, patch_num=4, patch_size=8, seed=0)
    c = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    pts = NeuralPoints(32, len(xyz), opt, dev)
    pts.set_points(c(xyz), c(att["emb"])[None], points_color=c(att["color"])[None], points_dir=c(att["dir"])[None],
                   points_conf=c(att["conf"])[None], parameter=True)
    torch.manual_seed(0)
    net = NeuralPointsRayMarching(aggregator=PointAggregator(opt).to(dev), neural_points=pts, opt=opt).to(dev)
    net.near_far = (0.1, 8.0)
    frame = {k: (c(v) if isinstance(v, np.ndarray) and v.dtype.kind == "f" else v) for k, v in fr.items()}
    kernels = c(predefined_blur_kernels(3))[None]
    R = fr["raydir"].shape[1]
    params = [p for p in net.parameters() if p.requires_grad]

    def fwd_bwd():
        for p in params:
            p.grad = None
        out = net(**frame)
        full = fill_invalid(out, frame["bg_color"], net.last_extras.ray_ids)
        if learnable:
            blurred, _ = learnable_blur(full["coarse_raycolor"], frame["gt_image"], out["blur_predictor"], 4, 8, 9, 4, 0, 1)
        else:
            blurred, _ = blur_select(full["coarse_raycolor"], frame["gt_image"], kernels, 4, 8)
        loss = torch.nn.functional.mse_loss(blurred, frame["gt_image"])
        loss.backward()
        return loss

    for _ in range(warmup):
        fwd_bwd()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    torch.cuda.synchronize()
    for s, e in ev:
        s.record()
        loss = fwd_bwd()
        e.record()
    torch.cuda.synchronize()
    ms = sum(s.elapsed_time(e) for s, e in ev) / steps
    return {"metric": "train rays/s (fwd+bwd, with blur module)", "value": R / (ms * 1e-3), "unit": "rays/s", "ms_fwd_bwd": ms, "rays": R,
            "valid_samples": int(net.last_extras.n_valid), "loss": float(loss.detach()),
            "config": BLUR_WORKLOAD.replace("pre-defined degradation-kernel convolution", "learnable per-patch blur kernel") if learnable else BLUR_WORKLOAD}
