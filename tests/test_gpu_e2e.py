"""GPU end-to-end parity: NeuralPointsRayMarching (query + aggregation + compositing, fused path)
against the CPU oracle pipeline on small seeded scenes: forward, and one training step's gradients."""
import numpy as np
import pytest
import torch

from helpers import T, assert_close, cuda, grad_atol
from hybridneuralrendering_b200 import make_opt
from hybridneuralrendering_b200 import synthetic as syn
from oracle import pipeline_oracle as po
from oracle import render_oracle as ro

pytestmark = pytest.mark.gpu
RTOL = 1e-4


def _build(opt, xyz, att, P):
    from hybridneuralrendering_b200 import NeuralPoints, NeuralPointsRayMarching, PointAggregator
    dev = torch.device("cuda")
    pts = NeuralPoints(32, len(xyz), opt, dev)
    pts.set_points(cuda(xyz), cuda(att["emb"])[None], points_color=cuda(att["color"])[None], points_dir=cuda(att["dir"])[None],
                   points_conf=cuda(att["conf"])[None], parameter=True)
    agg = PointAggregator(opt).cuda()
    agg.load_state_dict(P, strict=False)
    return NeuralPointsRayMarching(aggregator=agg, neural_points=pts, opt=opt).cuda()


def _frame_cuda(fr):
    return {k: (cuda(v) if isinstance(v, np.ndarray) and v.dtype.kind == "f" else v) for k, v in fr.items()}


def _product_projections(net, fr, loc_w):
    """P1 of the product (project_views_kernel: neural_points_volumetric_model.py:248-255, :296-310) on the given sample positions
    (V,S,2), (V,S,3) -- with the world->camera matrices the aggregator itself prepares"""
    from hybridneuralrendering_b200 import ops
    V = int(net.opt.use_nearest)
    _, w2c = net.aggregator.prepare_views(cuda(fr["images_nearest"]), cuda(fr["c2w_nearest"])[0, :V])
    lw = cuda(np.ascontiguousarray(loc_w)).reshape(-1, 3)
    return ops.project_views(lw, w2c, cuda(fr["intrinsic_nearest"][0]).reshape(3, 3), cuda(fr["campos"]).reshape(-1)[:3],
                             cuda(fr["campos_nearest"][0, :V]).reshape(-1, 3))


def _check_projections(xy, delta, ref):
    """product projections vs the oracle's own: sub-pixel (1e-3 px, relative 1e-5 for far-off-screen points), unit-vector
    differences to 1e-6.  The oracle then truncates the PRODUCT's floats, so the discontinuous nearest-pixel lookup cannot differ."""
    own = ref["xy_own"].reshape(xy.shape).double()
    assert float(((xy.cpu().double() - own).abs() / (1.0 + 1e-2 * own.abs())).max()) < 1e-3
    assert float((delta.cpu().double() - ref["delta_view"].reshape(delta.shape).double()).abs().max()) < 1e-6


def test_render_forward_matches_oracle():
    opt = make_opt("scannet", use_nearest=3, SR=24)
    xyz = syn.room_scene(40000, 5)
    att = syn.point_attributes(np.random.default_rng(5), len(xyz))
    fr = syn.room_frame(H=48, W=64, V=3, patch_num=4, patch_size=4, seed=2)
    P = ro.random_params(7)
    net = _build(opt, xyz, att, P)
    ts = net.neural_points.querier.candidate_ts(fr["raydir"].shape[1], 0.1, 8.0, "cuda")
    with torch.no_grad():
        out = net(**_frame_cuda(fr))
    pts = dict(xyz=xyz, **att)
    q = po.query(pts, fr, opt, ts.cpu().numpy().reshape(-1))
    np.testing.assert_array_equal(out["ray_mask"].cpu().numpy(), q["ray_mask"])
    xy, delta = _product_projections(net, fr, q["sample_loc_w"])
    ref = po.render(P, ro.AggCfg(use_nearest=3), pts, fr, opt, None, q=q, xy_override=xy.cpu())
    _check_projections(xy, delta, ref)
    assert out["coarse_raycolor"].shape == ref["ray_color"].shape and ref["ray_color"].shape[1] > 100
    # every ray, no allowance: rtol 1e-4 (north_star) with the absolute floors of DESIGN.md §4
    assert_close(out["coarse_raycolor"], ref["ray_color"], RTOL, 1e-5)
    assert_close(out["coarse_point_opacity"], ref["opacity"], RTOL, 1e-6)
    assert_close(out["coarse_is_background"], ref["bg_T"], RTOL, 1e-6)
    assert_close(out["conf_coefficient"], ref["conf_coefficient"], 0, 0)
    assert_close(out["weight"], ref["weight"], 1e-5, 1e-7)


def test_train_step_gradients_match_oracle():
    from hybridneuralrendering_b200.neural_points_volumetric_model import fill_invalid
    opt = make_opt("scannet", use_nearest=2, SR=24, is_train=True, drop_ratio=0.5, dilation_setup="4_4_1_8")
    xyz = syn.room_scene(30000, 6)
    att = syn.point_attributes(np.random.default_rng(6), len(xyz))
    fr = syn.room_frame(H=48, W=64, V=2, patch_num=4, patch_size=4, seed=3)
    P = ro.random_params(8)
    net = _build(opt, xyz, att, P)
    torch.manual_seed(3)
    R = fr["raydir"].shape[1]
    st = torch.cuda.get_rng_state()
    ts = net.neural_points.querier.candidate_ts(R, 0.1, 8.0, "cuda")       # the jittered draw the forward will repeat
    torch.cuda.set_rng_state(st)
    out = net(**_frame_cuda(fr))
    mask = check_gradients_vs_oracle(net, out, fr, ts, P, dict(xyz=xyz, **att), opt)
    full = fill_invalid(out, cuda(fr["bg_color"]), net.last_extras.ray_ids)
    assert full["coarse_raycolor"].shape == (1, R, 3)
    assert_close(full["coarse_raycolor"][:, ~mask], torch.ones_like(full["coarse_raycolor"][:, ~mask]), 0, 0)


def check_gradients_vs_oracle(net, out, fr, ts, P, pts, opt):
    """backward of the kink-masked training loss from the forward `out` of `net` (frame `fr`, candidate parameters `ts`), compared with
    the fp64 oracle at aggregator parameters P and point attributes `pts`: the loss and every gradient.  Returns the ray mask."""
    R = fr["raydir"].shape[1]
    mask = out["ray_mask"][0] > 0
    q = po.query(pts, fr, opt, ts.cpu().numpy().reshape(R, -1))
    np.testing.assert_array_equal(out["ray_mask"].cpu().numpy(), q["ray_mask"])
    xy, delta = _product_projections(net, fr, q["sample_loc_w"])
    cfg = ro.AggCfg(use_nearest=2, is_train=True, drop_ratio=0.5, dilation_setup="4_4_1_8")
    # fp64 oracle on the product's projections; rays with a hidden unit within 1e-5 of a LeakyReLU kink are masked out of the colour
    # loss on BOTH sides (LeakyReLU' jumps there: the slope an fp32 implementation takes depends on its summation order)
    ref = po.render(P, cfg, pts, fr, opt, None, dtype=torch.float64, params_grad=True, q=q, xy_override=xy.cpu(), kink_eps=1e-5)
    _check_projections(xy, delta, ref)
    assert int(mask.sum()) == ref["ray_color"].shape[1]
    keep = ref["kink_free"].to(torch.float64)[None, :, None]
    assert float(keep.mean()) > 0.5
    gt = T(fr["gt_image"])[:, mask.cpu()]
    v = out["conf_coefficient"].clamp(1e-3, 1 - 1e-3)
    keep_g = keep.float().cuda()
    loss = torch.nn.functional.mse_loss(out["coarse_raycolor"] * keep_g, gt.cuda() * keep_g) + 1e-4 * torch.mean(torch.log(v) + torch.log(1 - v))
    loss.backward()
    rv = ref["conf_coefficient"].clamp(1e-3, 1 - 1e-3)
    rloss = torch.nn.functional.mse_loss(ref["ray_color"] * keep, gt.double() * keep) + 1e-4 * torch.mean(torch.log(rv) + torch.log(1 - rv))
    rloss.backward()
    assert_close(loss, rloss, 1e-4, 1e-7)
    npts = net.neural_points
    for name, leaf in (("points_embeding", "emb"), ("points_conf", "conf"), ("points_color", "color"), ("points_dir", "dir")):
        g, r = getattr(npts, name).grad[0], ref["leaf"][leaf].grad
        assert int((r.abs().sum(-1) > 0).sum()) > 50
        assert_close(g, r, RTOL, grad_atol(r), name)                    # every row: rtol 1e-4 + 1e-4 x max magnitude
    n = 0
    for k, p in net.aggregator.named_parameters():
        r = ref["params"][k].grad if k in ref["params"] else None
        if r is None or float(r.abs().max()) == 0:
            continue
        assert_close(p.grad, r, RTOL, grad_atol(r), k)
        n += 1
    assert n >= 40
    return mask


def test_fused_training_forward_equals_layered_training_forward():
    """A/B of the two graph-recording paths of the per-neighbour stage: fused tensor-core kernel with saved activations
    (NbrMlpFusedFn) vs layer-by-layer kernels -- same outputs and same gradients within rtol 1e-4."""
    opt = make_opt("scannet", use_nearest=2, SR=24, is_train=True, drop_ratio=0.5, dilation_setup="4_4_1_8")
    xyz = syn.room_scene(30000, 9)
    att = syn.point_attributes(np.random.default_rng(9), len(xyz))
    fr = syn.room_frame(H=48, W=64, V=2, patch_num=4, patch_size=4, seed=5)
    P = ro.random_params(10)
    res = []
    for fused in (True, False):
        net = _build(opt, xyz, att, P)
        net.aggregator.fused_train_forward = fused
        torch.manual_seed(3)
        out = net(**_frame_cuda(fr))
        gt = cuda(fr["gt_image"])[:, out["ray_mask"][0] > 0]
        loss = torch.nn.functional.mse_loss(out["coarse_raycolor"], gt)
        loss.backward()
        res.append((out["coarse_raycolor"].detach(), {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}))
    (ca, ga), (cb, gb) = res
    assert_close(ca, cb, RTOL, 1e-6)
    assert set(ga) == set(gb) and len(ga) > 40
    for k in ga:
        # LeakyReLU' jumps at 0: a hidden unit whose pre-activation is within rounding noise of 0 may take the other slope in
        # one of the two (differently rounded) forwards and shift the gradients that flow through that single unit; everything
        # else must agree to rtol 1e-4
        a, b = ga[k].double(), gb[k].double()
        bad = (a - b).abs() > RTOL * b.abs() + grad_atol(gb[k])
        assert int(bad.sum()) <= max(2, int(1e-4 * bad.numel())), (k, int(bad.sum()), bad.numel())
        assert float((a - b).abs().max()) <= 0.02 * float(b.abs().max()) + 1e-12, k


def test_full_frame_render_is_deterministic_and_finite_at_config2_size():
    """size-independent properties at BASELINE configs[1] size (800x800, 1M points): two renders of the same frame are
    bit-identical (no atomics / no run-to-run ordering on the inference path), every pixel is finite and inside the colour
    range, rays that hit nothing carry the background colour, and a shifted ray chunking gives the same image."""
    from hybridneuralrendering_b200.renderer import render_rays
    opt = make_opt("lego", use_nearest=4, is_train=False)
    xyz = syn.lego_scene(1_000_000, 0)
    att = syn.point_attributes(np.random.default_rng(0), len(xyz))
    fr = syn.lego_frame(H=800, W=800, V=4, seed=0)
    net = _build(opt, xyz, att, ro.random_params(0))
    net.near_far = (2.0, 6.0)
    frame = {k: cuda(np.ascontiguousarray(fr[k])) for k in ("campos", "camrotc2w", "raydir", "near", "far", "intrinsic", "bg_color",
                                                             "images_nearest", "c2w_nearest", "campos_nearest", "intrinsic_nearest")}
    a = render_rays(net, frame).clone()
    b = render_rays(net, frame).clone()
    assert torch.equal(a, b)
    assert bool(torch.isfinite(a).all()) and float(a.min()) >= -0.0011 and float(a.max()) <= 1.0011
    hit = (a - 1.0).abs().amax(-1) > 0
    assert 0.1 < float(hit.float().mean()) < 0.9                     # the object covers part of the frame, the rest is background
    c = render_rays(net, frame, chunk_rays=200_000)                  # different chunking -> same pixels
    assert_close(c, a, RTOL, 1e-6)
