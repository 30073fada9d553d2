"""world_size-2 gloo test (CPU) of the multi-GPU host logic: ray sharding by whole patches and the
gradient all-reduce with global-mean normalisation must reproduce the single-process full-batch gradients."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from hybridneuralrendering_b200 import parallel


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _toy(seed=0):
    g = torch.Generator().manual_seed(seed)
    big = torch.nn.Parameter(torch.randn(5000, 39, generator=g))          # "point table" (reduced in place)
    w1 = torch.nn.Parameter(torch.randn(39, 16, generator=g) * 0.1)       # small "MLP" tensors (coalesced bucket)
    w2 = torch.nn.Parameter(torch.randn(16, 3, generator=g) * 0.1)
    unused = torch.nn.Parameter(torch.zeros(7))                           # never receives a gradient
    return [big, w1, w2, unused]


def _loss(params, idx, gt, valid):
    big, w1, w2, _ = params
    pred = torch.tanh(big[idx] @ w1) @ w2                                  # (R,3)
    m = valid.bool()
    return torch.nn.functional.mse_loss(pred[m], gt[m])                    # MEAN over the valid rays, like the reference loss


def _data(R=256, seed=1):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, 5000, (R,), generator=g)
    gt = torch.rand(R, 3, generator=g)
    valid = torch.rand(R, generator=g) > 0.3
    valid[:64] = False                                                     # rank 0's first patch has no valid ray
    return idx, gt, valid


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    params = _toy()
    idx, gt, valid = _data()
    b, e = parallel.shard_patches(idx.shape[0], 64, rank, world)
    n_local = valid[b:e].sum()
    if int(n_local) > 0:
        _loss(params, idx[b:e], gt[b:e], valid[b:e]).backward()
    n_global = parallel.allreduce_gradients(params, n_local, bucket_bytes=1 << 16)
    torch.save({"grads": [p.grad.clone() for p in params], "n_global": n_global, "range": (b, e)}, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


def _worker_prescaled(rank, world, port, out_dir):
    """the overlapped form train_step uses: loss pre-scaled by n_local/n_global, small bucket first, large tensors left in flight"""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    params = _toy()
    idx, gt, valid = _data()
    b, e = parallel.shard_patches(idx.shape[0], 64, rank, world)
    n_local = valid[b:e].sum()
    scale, n_global = parallel.global_mean_scale(n_local)
    if int(n_local) > 0:
        (_loss(params, idx[b:e], gt[b:e], valid[b:e]) * scale[0]).backward()
    _, pending = parallel.allreduce_gradients(params, None, bucket_bytes=1 << 16, prescaled=True, defer_large=True)
    assert len(pending) == 1 and pending[0][1] is params[0].grad          # the "point table" is the one large tensor
    small_done = [p.grad.clone() for p in params[1:]]                      # usable before the large reduction is waited for
    for h, _ in pending:
        h.wait()
    torch.save({"grads": [params[0].grad.clone()] + small_done, "n_global": n_global, "range": (b, e)}, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


def test_prescaled_overlapped_allreduce_matches_full_batch_gradients(tmp_path):
    world = 2
    mp.spawn(_worker_prescaled, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    params = _toy()
    idx, gt, valid = _data()
    _loss(params, idx, gt, valid).backward()
    outs = [torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in range(world)]
    assert float(outs[0]["n_global"]) == float(valid.sum())
    for r in range(world):
        for p, g in zip(params, outs[r]["grads"]):
            ref = p.grad if p.grad is not None else torch.zeros_like(p)
            np.testing.assert_allclose(g.numpy(), ref.numpy(), rtol=1e-5, atol=1e-8)


class _NoDefer:
    """stand-in for ops.defer_weight_gradients (whose runner needs CUDA streams): nothing is parked, so there is nothing to run"""

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def run(self):
        pass


class _ToyNet(torch.nn.Module):
    """the parts of NeuralPointsRayMarching that train_step relies on: a point table over the deferred-step threshold (32768 x 39
    fp32 = 5.1 MB > 4 MB), a small "MLP", and the `before_point_read` hook, run before the table is read"""

    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(0)
        self.table = torch.nn.Parameter(torch.randn(_TABLE_ROWS, 39, generator=g))
        self.w1 = torch.nn.Parameter(torch.randn(39, 16, generator=g) * 0.1)
        self.w2 = torch.nn.Parameter(torch.randn(16, 3, generator=g) * 0.1)
        self.before_point_read = None

    def forward(self, idx, valid, **_):
        if self.before_point_read is not None:
            cb, self.before_point_read = self.before_point_read, None
            cb()
        m = valid.bool()
        color = torch.tanh(self.table[idx[m]] @ self.w1) @ self.w2
        return {"coarse_raycolor": color[None], "ray_mask": valid.to(torch.int8)[None]}


_TABLE_ROWS = 32768
_STEPS = 3


def _toy_optimizers(net):
    """the two Adam groups of benchmarks.make_optimizers (network lr 5e-4, point table lr 2e-3), as torch.optim.Adam"""
    return [torch.optim.Adam([net.w1, net.w2], lr=5e-4), torch.optim.Adam([net.table], lr=2e-3)]


def _toy_raster(step, rank, R=256):
    """rank `rank`'s own raster of training step `step`"""
    g = torch.Generator().manual_seed(1000 + 10 * step + rank)
    idx = torch.randint(0, _TABLE_ROWS, (R,), generator=g)
    gt = torch.rand(1, R, 3, generator=g)
    valid = torch.rand(R, generator=g) > 0.3
    return {"idx": idx, "valid": valid, "gt_image": gt}


def _worker_train_steps(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), HNR_SMALL_BUCKET="nccl")
    from hybridneuralrendering_b200 import ops
    ops.defer_weight_gradients = _NoDefer
    dist.init_process_group("gloo", rank=rank, world_size=world)
    net = _ToyNet()
    opts = _toy_optimizers(net)
    losses, n_globals = [], []
    for k in range(_STEPS):
        loss, n_global = parallel.train_step(net, _toy_raster(k, rank), opts)
        losses.append(float(loss))
        n_globals.append(float(n_global))
    parallel.flush_pending(net)
    torch.save({"params": {n: p.detach().clone() for n, p in net.named_parameters()},
                "steps": {n: int(opts[i].state[p]["step"]) for i, n, p in ((1, "table", net.table), (0, "w1", net.w1), (0, "w2", net.w2))},
                "losses": losses, "n_global": n_globals}, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


def test_train_step_trains_point_tables_across_steps(tmp_path):
    """three data-parallel train_steps on two ranks, then flush_pending, against one process that steps Adam on the n_valid-weighted
    mean of both rasters' gradients every step.  The point table's optimiser step is deferred into the next forward; it must see the
    gradients of the step before (it was skipped when they had already been zeroed: step count 1, the table moved only at the flush)."""
    world = 2
    mp.spawn(_worker_train_steps, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    outs = [torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in range(world)]
    net = _ToyNet()
    opts = _toy_optimizers(net)
    start = net.table.detach().clone()
    for k in range(_STEPS):
        for o in opts:
            o.zero_grad(set_to_none=True)
        rasters = [_toy_raster(k, r) for r in range(world)]
        n = [r["valid"].sum().to(torch.float32) for r in rasters]
        n_global = n[0] + n[1]
        for r, fr in enumerate(rasters):
            # the same float32 scale train_step applies to each rank's loss (global_mean_scale)
            out = net(**fr)
            loss = torch.nn.functional.mse_loss(out["coarse_raycolor"], fr["gt_image"][:, fr["valid"]])
            (loss * (n[r] / n_global)).backward()
        for o in opts:
            o.step()
        for r in range(world):
            assert outs[r]["n_global"][k] == float(n_global)
    for r in range(world):
        assert outs[r]["steps"] == {"table": _STEPS, "w1": _STEPS, "w2": _STEPS}
        for name, p in net.named_parameters():
            # both sides run the same float32 torch arithmetic; rtol 1e-6 leaves room for the all-reduce summing the two ranks'
            # gradients in another order than the reference's accumulation (atol: 1e-6 of the smaller learning rate, for entries near 0)
            np.testing.assert_allclose(outs[r]["params"][name].numpy(), p.detach().numpy(), rtol=1e-6, atol=5e-10, err_msg=name)
    for name in outs[0]["params"]:
        assert torch.equal(outs[0]["params"][name], outs[1]["params"][name]), name
    # every row a ray of any step read has moved (with the update skipped, only the rows of the last step moved, at the flush)
    touched = torch.cat([_toy_raster(k, r)["idx"][_toy_raster(k, r)["valid"]] for k in range(_STEPS) for r in range(world)]).unique()
    assert bool((outs[0]["params"]["table"][touched] != start[touched]).any(dim=1).all())


def test_shard_patches_partition():
    for R, world in ((3136, 8), (4096, 3), (64, 4)):
        spans = [parallel.shard_patches(R, 64, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == R
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert all((e - b) % 64 == 0 for b, e in spans)


def test_allreduce_matches_full_batch_gradients(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    params = _toy()
    idx, gt, valid = _data()
    _loss(params, idx, gt, valid).backward()
    outs = [torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in range(world)]
    assert float(outs[0]["n_global"]) == float(valid.sum())
    for r in range(world):
        for p, g in zip(params, outs[r]["grads"]):
            ref = p.grad if p.grad is not None else torch.zeros_like(p)
            np.testing.assert_allclose(g.numpy(), ref.numpy(), rtol=1e-5, atol=1e-8)
    for a, b in zip(outs[0]["grads"], outs[1]["grads"]):
        assert torch.equal(a, b)                                           # replicas hold identical gradients


def test_shard_frame_slices_only_ray_entries():
    R = 256
    frame = {"raydir": torch.zeros(1, R, 3), "gt_image": torch.zeros(1, R, 3), "pixel_idx": torch.zeros(1, R, 2),
             "campos": torch.zeros(1, 3), "images_nearest": torch.zeros(1, 2, 4, 4, 3)}
    s = parallel.shard_frame(frame, 1, 2)
    assert s["raydir"].shape == (1, 128, 3) and s["gt_image"].shape == (1, 128, 3) and s["images_nearest"].shape == (1, 2, 4, 4, 3)


def test_shard_frame_keeps_patches_whole():
    """training frames (dilated patch layout): every rank gets whole rows of patches of the raster, for any world size"""
    PN, PS = 8, 8
    S = PN * PS
    R = S * S
    patch_of_ray = ((torch.arange(S)[:, None] // PS) * PN + torch.arange(S)[None, :] // PS).reshape(-1)      # raster -> patch id
    frame = {"raydir": torch.arange(R, dtype=torch.float32)[None, :, None].expand(1, R, 3), "gt_image": torch.zeros(1, R, 3),
             "pixel_idx": torch.zeros(1, S, S, 2), "dilation_PatchNum": np.array([PN]), "dilation_PatchSize": np.array([PS])}
    for world in (1, 2, 3, 4, 8):
        seen = []
        owners = {}
        for rank in range(world):
            sh = parallel.shard_frame(frame, rank, world)
            ids = sh["raydir"][0, :, 0].long()
            assert sh["pixel_idx"].shape == (1, len(ids), 2) and sh["gt_image"].shape == (1, len(ids), 3)
            assert len(ids) % (PS * S) == 0 and torch.equal(ids, torch.arange(int(ids[0]), int(ids[0]) + len(ids)))
            for pch in patch_of_ray[ids].unique().tolist():
                assert owners.setdefault(pch, rank) == rank, "a patch is split between ranks"
            assert (torch.bincount(patch_of_ray[ids], minlength=PN * PN)[patch_of_ray[ids].unique()] == PS * PS).all()
            seen.append(ids)
        assert torch.equal(torch.cat(seen), torch.arange(R))
