"""Consecutive training steps.  The single-step tests check one step's gradients on a freshly built model; the state a training run
carries from step to step is checked here: the weight images cached on the modules and keyed on the parameters' versions, the voxel
query prefetched one step ahead, the weight-gradient tails that train_step parks during backward, and, with two ranks, the point-table
optimiser step deferred into the next forward.  Each is compared with a reference that has none of that state.  Also FusedAdam at its
edges against fp64 torch.optim.Adam.

Every jittered depth-candidate draw is taken up front from a seeded generator and handed to the queries in call order, so that the
product (which draws step k+1's candidates during step k) and the references see the same sample positions.  The patch drop does not
draw: its positions follow from the options alone."""
import datetime
import math
import os
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_gpu_e2e import _build, _frame_cuda, check_gradients_vs_oracle
from hybridneuralrendering_b200 import make_opt, ops, parallel
from hybridneuralrendering_b200 import synthetic as syn
from hybridneuralrendering_b200.benchmarks import make_optimizers
from hybridneuralrendering_b200.optim import FusedAdam
from hybridneuralrendering_b200.renderer import training_loss
from oracle import render_oracle as ro

pytestmark = pytest.mark.gpu

NEAR, FAR = 0.1, 8.0
R = 256                       # rays of a 4_4_1_8 raster: 4 x 4 patches of 4 x 4
DP_STEPS = 3


def _opt():
    return make_opt("scannet", use_nearest=2, SR=24, is_train=True, drop_ratio=0.5, dilation_setup="4_4_1_8")


def _scene():
    xyz = syn.room_scene(30000, 6)
    return xyz, syn.point_attributes(np.random.default_rng(6), len(xyz)), ro.random_params(8)


def _frames(seeds):
    return [_frame_cuda(syn.room_frame(H=48, W=64, V=2, patch_num=4, patch_size=4, seed=s)) for s in seeds]


def _net(opt, xyz, att, P, values=None):
    """the test scene's model; seeded, so that parameters the aggregator parameters P do not cover start alike in every process.
    `values`: {name: tensor} copied over the trainable parameters (a fresh model at those values)"""
    torch.manual_seed(0)
    net = _build(opt, xyz, att, P)
    net.near_far = (NEAR, FAR)
    if values is not None:
        with torch.no_grad():
            for n, p in _trainable(net):
                p.copy_(values[n])
    return net


def _trainable(net):
    return [(n, p) for n, p in net.named_parameters() if p.requires_grad]


def _lr(name):
    """the learning rates of benchmarks.make_optimizers"""
    return 2e-3 if name.startswith("neural_points.") else 5e-4


def _draw_ts(net, seed):
    torch.manual_seed(seed)
    return net.neural_points.querier.candidate_ts(R, NEAR, FAR, "cuda")


def _feed_ts(net, ts_list):
    """from now on the query of `net` takes its depth candidates from ts_list, in call order; returns the call counter"""
    it, calls = iter(ts_list), [0]

    def candidate_ts(n_rays, near, far, device):
        calls[0] += 1
        ts = next(it)
        assert ts.shape[1] == n_rays and (near, far) == (NEAR, FAR)
        return ts
    net.neural_points.querier.candidate_ts = candidate_ts
    return calls


class _Adam64:
    """torch.optim.Adam (betas 0.9 / 0.999, eps 1e-8, no weight decay) on fp64 master copies; a parameter without a gradient is
    skipped and keeps its own step count, as in torch"""

    def __init__(self, named):
        self.p = {n: p.detach().double().clone() for n, p in named}
        self.m = {n: torch.zeros_like(p) for n, p in self.p.items()}
        self.v = {n: torch.zeros_like(p) for n, p in self.p.items()}
        self.t = {n: 0 for n in self.p}

    def step(self, grads):
        b1, b2, eps = 0.9, 0.999, 1e-8
        for n, g in grads.items():
            if g is None:
                continue
            g = g.double()
            self.t[n] += 1
            t = self.t[n]
            self.m[n].mul_(b1).add_(g, alpha=1 - b1)
            self.v[n].mul_(b2).addcmul_(g, g, value=1 - b2)
            denom = self.v[n].sqrt() / math.sqrt(1 - b2 ** t) + eps
            self.p[n].sub_(_lr(n) / (1 - b1 ** t) * self.m[n] / denom)


def _compare_params(named, ref, what, report):
    """every element within 1e-3 lr + 1e-6 |p| of the reference.  Adam's first steps move an element by about lr sign(g) whatever |g|:
    a gradient at the noise floor of the fp32 atomics may take the other sign and move its element by 2 lr the other way, so at most
    max(2, 1e-5 numel) elements per tensor may exceed the bound.  A tensor with more such elements still passes when none deviates by
    more than 0.1 lr: a hidden unit whose pre-activation lies within the atomics' rounding noise of 0 may take the other LeakyReLU slope
    on one side (the summation order of the forward differs from run to run), which shifts whole weight rows by a small fraction of lr.
    A lost or misapplied optimiser step moves elements by about lr.  Appends (what, name, worst |d| / lr, elements over the bound)."""
    bad = []
    for n, p in named:
        r = ref[n].to(p.device, torch.float64)
        d = (p.detach().double() - r).abs()
        over = int((d > 1e-3 * _lr(n) + 1e-6 * r.abs()).sum())
        report.append((what, n, float(d.max()) / _lr(n), over))
        if over > max(2, int(1e-5 * d.numel())) and float(d.max()) > 0.1 * _lr(n):
            bad.append((n, over, d.numel(), float(d.max()) / _lr(n)))
    assert not bad, (what, bad)


def _print_report(title, report):
    worst = max(report, key=lambda e: e[2])
    print(f"\n{title}: worst |d| = {worst[2]:.3g} lr ({worst[0]}, {worst[1]}); elements over the bound: "
          + (", ".join(f"{w} {n} {c}" for w, n, _, c in report if c) or "none"))


def test_training_trajectory_matches_cache_free_reference():
    """four parallel.train_steps (prefetched query, parked gradient tails, FusedAdam through raw pointers, weight images cached on the
    modules) against, every step, a model built fresh from the reference's current parameters: plain forward, training_loss,
    backward, then Adam in fp64 on master copies"""
    opt = _opt()
    xyz, att, P = _scene()
    frames = _frames((3, 4, 5))
    steps = 4
    seq = [frames[k % len(frames)] for k in range(steps + 1)]
    net = _net(opt, xyz, att, P)
    ts = [_draw_ts(net, 100 + k) for k in range(steps + 1)]          # candidates of step k; the last one for step 3's prefetch
    calls = _feed_ts(net, ts)
    opts = make_optimizers(net)
    named = _trainable(net)
    ref = _Adam64(named)
    start = {n: p.detach().clone() for n, p in named}
    report = []
    for k in range(steps):
        loss, n_valid = parallel.train_step(net, seq[k], opts, next_frame_shard=seq[k + 1])
        rnet = _net(opt, xyz, att, P, values=ref.p)
        _feed_ts(rnet, [ts[k]])
        out = rnet(**seq[k])
        rloss = training_loss(out, seq[k]["gt_image"])
        rloss.backward()
        ref.step({n: p.grad for n, p in _trainable(rnet)})
        assert int(n_valid) == int((out["ray_mask"] > 0).sum())
        # same kernels on (nearly) the same parameters: the loss differs by atomics ordering and the fp32 / fp64 Adam only
        np.testing.assert_allclose(float(loss), float(rloss), rtol=1e-5, atol=0)
        _compare_params(named, ref.p, f"step {k}", report)
        if k == 0:
            # the product's first step: Adam moves an element by lr g / (|g| + eps), >= 2/3 lr where |g| >= 2 eps, so every row
            # with such a gradient element moved by at least 0.5 lr
            for n, p in named:
                if not n.startswith("neural_points."):
                    continue
                rows = p.grad[0].abs().amax(-1) >= 2e-8
                moved = (p.detach() - start[n])[0].abs().amax(-1)
                assert int(rows.sum()) > 50, n
                assert bool((moved[rows] >= 0.5 * _lr(n)).all()), (n, float(moved[rows].min()))
    assert calls[0] == steps + 1                                        # every query took its candidates from the list, in order
    _print_report("trajectory vs cache-free fp64-Adam reference", report)


def test_gradients_at_updated_parameters_match_oracle():
    """step 2's gradients on the model that train_step and FusedAdam just updated (warm weight caches, prefetched query) against the
    fp64 oracle evaluated at the updated parameters, with the kink-masked loss and tolerances of test_train_step_gradients_match_oracle"""
    opt = _opt()
    xyz, att, P = _scene()
    f0, f1 = _frames((3, 4))
    fr1 = syn.room_frame(H=48, W=64, V=2, patch_num=4, patch_size=4, seed=4)
    net = _net(opt, xyz, att, P)
    ts = [_draw_ts(net, 200), _draw_ts(net, 201)]
    calls = _feed_ts(net, ts)
    opts = make_optimizers(net)
    emb0 = net.neural_points.points_embeding.detach().clone()
    parallel.train_step(net, f0, opts, next_frame_shard=f1)
    for p in net.parameters():
        p.grad = None
    out = net(**f1)
    assert calls[0] == 2                                                # the forward used the prefetched query
    npts = net.neural_points
    assert not torch.equal(npts.points_embeding.detach(), emb0)
    pts = dict(xyz=xyz, **{k: getattr(npts, name).detach()[0].cpu().numpy() for k, name in
                           (("emb", "points_embeding"), ("color", "points_color"), ("dir", "points_dir"), ("conf", "points_conf"))})
    sd = net.aggregator.state_dict()
    P1 = {k: sd[k].detach().float().cpu() if k in sd else P[k] for k in P}
    assert any(not torch.equal(P1[k], P[k].float()) for k in P)
    check_gradients_vs_oracle(net, out, fr1, ts[1], P1, pts, opt)


# ---------------------------------------------------------------- two ranks on one GPU
def _dp_frame_seed(step, rank):
    return 20 + 2 * step + rank


def _dp_ts_seed(step, rank):
    return 300 + 2 * step + rank


def _rank_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), HNR_SMALL_BUCKET="nccl")
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
    try:
        opt = _opt()
        xyz, att, P = _scene()
        frames = _frames([_dp_frame_seed(k, rank) for k in range(DP_STEPS)])
        net = _net(opt, xyz, att, P)
        calls = _feed_ts(net, [_draw_ts(net, _dp_ts_seed(k, rank)) for k in range(DP_STEPS)])
        opts = make_optimizers(net)
        n_global = []
        for k in range(DP_STEPS):
            # large_bytes: the 30k-point embedding table (3.8 MB) is below the default 4 MB at which the point-table step is deferred
            _, ng = parallel.train_step(net, frames[k], opts, next_frame_shard=frames[k + 1] if k + 1 < DP_STEPS else None,
                                        large_bytes=1 << 20)
            n_global.append(float(ng))
        assert net.before_point_read is not None                        # the last step's point-table update is still pending
        parallel.flush_pending(net)
        assert calls[0] == DP_STEPS
        torch.save({"params": {n: p.detach().cpu() for n, p in _trainable(net)}, "n_global": n_global,
                    "steps": sorted({o.state[p]["step"] for o in opts for p in o.state})}, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _reference_worker(_, out_dir):
    """the single-process reference of test_two_ranks_match_single_process_steps, in a fresh process like the ranks: per step, the
    backward of training_loss x n_r / (n_0 + n_1) of both rasters accumulated, then both FusedAdam groups stepped"""
    torch.cuda.set_device(0)
    world = 2
    opt = _opt()
    xyz, att, P = _scene()
    net = _net(opt, xyz, att, P)
    frames = [_frames([_dp_frame_seed(k, r) for k in range(DP_STEPS)]) for r in range(world)]
    ts = [[_draw_ts(net, _dp_ts_seed(k, r)) for k in range(DP_STEPS)] for r in range(world)]
    opts = make_optimizers(net)
    named = _trainable(net)
    start = {n: p.detach().cpu().clone() for n, p in named}
    n_global = []
    for k in range(DP_STEPS):
        for o in opts:
            o.zero_grad(set_to_none=True)
        # the valid-ray count of a raster depends on the query alone (the points' positions are not trained)
        n = [(net.neural_points.query({"raydir": frames[r][k]["raydir"], "campos": frames[r][k]["campos"],
                                       "camrotc2w": frames[r][k]["camrotc2w"]}, NEAR, FAR, ts=ts[r][k])[4] > 0).sum().to(torch.float32)
             for r in range(world)]
        for r in range(world):
            _feed_ts(net, [ts[r][k]])
            out = net(**frames[r][k])
            assert int((out["ray_mask"] > 0).sum()) == int(n[r])
            (training_loss(out, frames[r][k]["gt_image"]) * (n[r] / (n[0] + n[1]))).backward()
        for o in opts:
            o.step()
        n_global.append(float(n[0] + n[1]))
    torch.save({"params": {n: p.detach().cpu() for n, p in named}, "start": start, "n_global": n_global}, os.path.join(out_dir, "ref.pt"))


def _run_spawned(fn, args, nprocs):
    ctx = mp.spawn(fn, args=args, nprocs=nprocs, join=False)
    try:
        deadline = time.monotonic() + 300
        while not ctx.join(timeout=5):
            assert time.monotonic() < deadline, "the processes did not finish within 300 s"
    finally:
        for p in ctx.processes:
            if p.is_alive():
                p.kill()
            p.join()


def test_two_ranks_match_single_process_steps(tmp_path):
    """parallel.train_step on 2 gloo ranks sharing this GPU (each rank its own raster; HNR_SMALL_BUCKET=nccl: no symmetric memory),
    3 steps and flush_pending, against one process that accumulates, per step, the backward of training_loss x n_r / (n_0 + n_1)
    of both rasters and then steps both FusedAdam groups.  The point-table step is deferred into the next forward on the ranks.
    The reference runs in a fresh process too, so both sides start from the same process state whatever ran before in this one (the
    noise floor of the fp32 atomics, which decides the Adam sign of the near-zero point-table gradients, otherwise follows it)."""
    world = 2
    _run_spawned(_rank_worker, (world, _free_port(), str(tmp_path)), world)
    outs = [torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in range(world)]
    _run_spawned(_reference_worker, (str(tmp_path),), 1)
    ref = torch.load(os.path.join(tmp_path, "ref.pt"))
    for r in range(world):
        assert outs[r]["n_global"] == ref["n_global"]
    assert outs[0]["steps"] == outs[1]["steps"] == [DP_STEPS]
    for n_ in outs[0]["params"]:
        assert torch.equal(outs[0]["params"][n_], outs[1]["params"][n_]), n_
    assert set(outs[0]["params"]) == set(ref["params"])
    report = []
    _compare_params(list(outs[0]["params"].items()), ref["params"], "after flush", report)
    for n_, p in outs[0]["params"].items():
        if n_.startswith("neural_points."):
            assert int((p != ref["start"][n_])[0].any(-1).sum()) > 100, n_       # the point tables moved
    _print_report("two gloo ranks vs single process", report)


# ---------------------------------------------------------------- FusedAdam edges
def test_fused_adam_edges_match_fp64_adam():
    """FusedAdam against torch.optim.Adam on fp64 copies: weight decay, more than 64 tensors in a group (several launches), a
    parameter without a gradient on some steps (its step count diverges: a launch of its own), a non-contiguous gradient, a parameter
    4 bytes off a 16-byte boundary (the scalar path), sizes around the float4 tail and the 1024-element block; then the status guard"""
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(0)
    sizes = [1, 3, 4, 5, 1023, 1024, 1025, 4097] + [1 + i % 7 for i in range(60)]
    a = [torch.nn.Parameter(torch.randn(s, generator=g).to(dev)) for s in sizes]
    sometimes = torch.nn.Parameter(torch.randn(33, generator=g).to(dev))              # no gradient on steps 1 and 3
    strided = torch.nn.Parameter(torch.randn(8, 16, generator=g).to(dev))             # gets a transposed (non-contiguous) gradient
    buf = torch.zeros(1031, device=dev)
    buf[1:1026] = torch.randn(1025, generator=g).to(dev)
    offset = torch.nn.Parameter(buf[1:1026])                                           # data pointer 4 bytes past buf's
    assert offset.data_ptr() % 16 == 4
    groups = [(a + [sometimes], dict(lr=1e-2, weight_decay=0.01)), ([strided, offset], dict(lr=3e-3, weight_decay=0.0))]
    fused = FusedAdam([dict(params=ps, **hp) for ps, hp in groups])
    ref_params = [[p.detach().cpu().double().clone().requires_grad_(True) for p in ps] for ps, _ in groups]
    ref = torch.optim.Adam([dict(params=rp, **hp) for rp, (_, hp) in zip(ref_params, groups)], foreach=False)
    pairs = [(p, rp, hp["lr"]) for (ps, hp), rps in zip(groups, ref_params) for p, rp in zip(ps, rps)]
    steps = 5
    for k in range(steps):
        for p, rp, _ in pairs:
            if p is sometimes and k in (1, 3):
                p.grad = rp.grad = None
                continue
            if p is strided:
                gr = torch.randn(16, 8, generator=g).to(dev).t()
                assert not gr.is_contiguous()
            else:
                gr = torch.randn(p.shape, generator=g).to(dev)
            p.grad = gr
            rp.grad = gr.detach().cpu().double()
        fused.step()
        ref.step()
        for i, (p, rp, lr) in enumerate(pairs):
            # fp32 against fp64: a few ulps of the update per step and the rounding of p
            np.testing.assert_allclose(p.detach().cpu().double().numpy(), rp.detach().numpy(), rtol=1e-6, atol=1e-5 * lr, err_msg=f"p {i} step {k}")
            st, rst = fused.state[p], ref.state[rp]
            assert st["step"] == int(rst["step"]), i
            np.testing.assert_allclose(st["exp_avg"].cpu().double().numpy(), rst["exp_avg"].numpy(), rtol=1e-5, atol=1e-6, err_msg=f"m {i}")
            # the kernel takes the betas as fp32: 1 - fp32(0.999) is 1.3e-5 (relative) off 0.001, so v is too.  The bias correction is
            # computed from the same fp32 beta and cancels that factor in the update, which the comparison of p above holds to 1e-6
            np.testing.assert_allclose(st["exp_avg_sq"].cpu().double().numpy(), rst["exp_avg_sq"].numpy(), rtol=2e-5, atol=1e-9, err_msg=f"v {i}")
    assert fused.state[sometimes]["step"] == steps - 2 and fused.state[a[0]]["step"] == steps
    assert torch.equal(buf[0], torch.zeros((), device=dev)) and torch.equal(buf[1026:], torch.zeros(5, device=dev))    # nothing outside p written

    # the range guard: with the status word set, the step is skipped on the device and p, m, v keep every bit
    for p, _, _ in pairs:
        p.grad = torch.randn(p.shape, generator=g).to(dev)
    before = [(p.detach().clone(), fused.state[p]["exp_avg"].clone(), fused.state[p]["exp_avg_sq"].clone()) for p, _, _ in pairs]
    word = ops.status_word(dev)
    try:
        word.fill_(1)
        fused.step()
        torch.cuda.synchronize()
    finally:
        word.zero_()
    for (p, _, _), (p0, m0, v0) in zip(pairs, before):
        assert torch.equal(p.detach(), p0) and torch.equal(fused.state[p]["exp_avg"], m0) and torch.equal(fused.state[p]["exp_avg_sq"], v0)
