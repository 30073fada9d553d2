"""GPU parity: compositing, blur, dense layers (called through the C ABI via the host wrappers)."""
import numpy as np
import pytest
import torch

from helpers import T, assert_close, blur_predictor, cuda, grad_atol, load_golden
from oracle import render_oracle as ro

pytestmark = pytest.mark.gpu

RTOL = 1e-4   # north_star: renders / gradients within rtol 1e-4 in fp32
# opacity = 1 - exp(-sigma*dist) is evaluated in fp32 by the reference too: its absolute error is one
# ulp of 1.0 (6e-8) whatever the magnitude of the result, so tiny opacities carry an absolute tolerance
OPACITY_ATOL = 2e-7


def test_ray_march_golden_fwd_bwd():
    from hybridneuralrendering_b200.diff_ray_marching import alpha_blend, radiance_render, ray_march
    G = load_golden("misc")
    f = cuda(G["rm_feats"]).clone().requires_grad_(True)
    o = ray_march(cuda(G["rm_dist"]), cuda(G["rm_valid"]), f, radiance_render, alpha_blend, cuda(G["rm_bg"]))
    assert_close(o[0], G["rm_ray_color"], RTOL, 1e-6)
    assert_close(o[2], G["rm_opacity"], RTOL, OPACITY_ATOL)
    assert_close(o[3], G["rm_accT"], RTOL, 1e-12)
    assert_close(o[4], G["rm_bw"], RTOL, OPACITY_ATOL)
    assert_close(o[5], G["rm_bgT"], RTOL, 1e-12)
    (o[0] * cuda(G["rm_G"])).sum().backward()
    assert_close(f.grad, G["rm_grad_feats"], RTOL, grad_atol(G["rm_grad_feats"], 1e-6))


@pytest.mark.parametrize("R,SR", [(1, 1), (7, 24), (33, 80), (5, 130)])
def test_ray_march_random_vs_oracle_all_outputs(R, SR):
    from hybridneuralrendering_b200.diff_ray_marching import alpha_blend, radiance_render, ray_march
    rng = np.random.default_rng(R * 1000 + SR)
    feats = T(rng.random((1, R, SR, 4)).astype(np.float32) * np.array([30, 1, 1, 1], np.float32))
    valid = T(rng.random((1, R, SR)) > 0.25)
    dist = T((rng.random((1, R, SR)) * 0.03).astype(np.float32))
    bg = T(np.array([[0.2, 0.9, 1.0]], np.float32))
    gC, gO, gT, gW, gB = [T(rng.standard_normal(s).astype(np.float32)) for s in ((1, R, 3), (1, R, SR), (1, R, SR), (1, R, SR, 1), (1, R, 1))]
    fo = feats.double().clone().requires_grad_(True)
    oo = ro.ray_march(dist.double(), valid, fo, bg.double())
    (oo[0] * gC).sum().backward(retain_graph=True)
    g1 = fo.grad.clone(); fo.grad = None
    ((oo[0] * gC).sum() + (oo[2] * gO).sum() + (oo[3] * gT).sum() + (oo[4] * gW).sum() + (oo[5] * gB).sum()).backward()
    g2 = fo.grad.clone()
    fg = feats.cuda().clone().requires_grad_(True)
    og = ray_march(dist.cuda(), valid.cuda(), fg, radiance_render, alpha_blend, bg.cuda())
    for i in (0, 2, 3, 4, 5):
        assert_close(og[i], oo[i], RTOL, OPACITY_ATOL if i in (2, 4) else 1e-9, f"output {i}")
    (og[0] * gC.cuda()).sum().backward(retain_graph=True)
    assert_close(fg.grad, g1, RTOL, grad_atol(g1, 1e-5))
    fg.grad = None
    ((og[0] * gC.cuda()).sum() + (og[2] * gO.cuda()).sum() + (og[3] * gT.cuda()).sum() + (og[4] * gW.cuda()).sum() + (og[5] * gB.cuda()).sum()).backward()
    assert_close(fg.grad, g2, RTOL, grad_atol(g2, 1e-5))


def test_ray_dist_prologue_fused():
    from hybridneuralrendering_b200.diff_ray_marching import ray_march_from_depth
    rng = np.random.default_rng(5)
    R, SR, vz = 41, 24, 0.008
    loc = T(rng.random((1, R, SR, 3)).astype(np.float32))
    z = np.sort(rng.random((1, R, SR)).astype(np.float32) * 0.3, axis=-1)
    z[0, :, 5] = z[0, :, 4]            # zero-length segment -> replaced by vsize
    z[0, :, 9] = z[0, :, 8] - 0.01      # non-monotone depth -> cummax
    z[0, 3, 12:] = 0.0                  # unfilled slots
    loc[..., 2] = T(z)
    valid = T(rng.random((1, R, SR)) > 0.2)
    feats = T(rng.random((1, R, SR, 4)).astype(np.float32) * np.array([40, 1, 1, 1], np.float32))
    d_ref = ro.ray_dist_from_depth(loc[..., 2], valid, vz, True)
    o_ref = ro.ray_march(d_ref, valid, feats, torch.ones(1, 3))
    color, opacity, accT, bw, bgT, dist = ray_march_from_depth(loc.cuda(), valid.cuda(), feats.cuda(), vz, 1, torch.ones(1, 3).cuda())
    np.testing.assert_array_equal(dist.cpu().numpy(), d_ref.numpy())      # exact: same float ops
    assert_close(color, o_ref[0], RTOL, 1e-6)
    assert_close(bgT, o_ref[5], RTOL, 1e-12)


def test_blur_golden_fwd_bwd():
    from hybridneuralrendering_b200.blur import blur_select
    G = load_golden("blur")
    PN, PS, Nk = [int(v) for v in G["meta"]]
    pred = cuda(G["pred"]).clone().requires_grad_(True)
    out, sel = blur_select(pred, cuda(G["gt"]), cuda(G["kernels"]), PN, PS)
    _, sel_ref = ro.blur_select(T(G["pred"]), T(G["gt"]), T(G["kernels"]), PN, PS)
    np.testing.assert_array_equal(sel.cpu().numpy(), sel_ref.numpy().astype(np.int32))      # argmin index: exact
    assert_close(out, G["out"], RTOL, 1e-6)
    (out * cuda(G["G"])).sum().backward()
    assert_close(pred.grad, G["grad_pred"], RTOL, 1e-6)


def test_blur_module_method_dropin_shipped_shape():
    """7x7 patches of 8x8 with the 36 shipped kernels, through blur_update_output(model)."""
    import types
    from hybridneuralrendering_b200.blur import blur_update_output, predefined_blur_kernels
    rng = np.random.default_rng(1)
    PN, PS = 7, 8
    K = predefined_blur_kernels(3)
    assert K.shape == (36, 9, 9)
    pred, gt = T(rng.random((1, (PN * PS) ** 2, 3), dtype=np.float32)), T(rng.random((1, (PN * PS) ** 2, 3), dtype=np.float32))
    ref, sel = ro.blur_select(pred, gt, T(K)[None], PN, PS)
    m = types.SimpleNamespace(output={"coarse_raycolor": pred.cuda()}, gt_image=gt.cuda(), blur_kernels=T(K)[None], dilation_PatchNum=PN, dilation_PatchSize=PS)
    blur_update_output(m)
    assert_close(m.output["coarse_raycolor"], ref, RTOL, 1e-6)


def test_learnable_blur_golden_fwd_bwd():
    """N3 (SURVEY 8f): learnable_blur_update_output through the drop-in method body vs outputs and gradients of the unmodified
    reference (tests/golden/blur_learn.npz), every norm / mode / boundary branch of the fixture."""
    import types
    from hybridneuralrendering_b200.blur import learnable_blur_update_output
    G = load_golden("blur_learn")
    PN, PS, KS = [int(v) for v in G["meta"]]
    for ci, (mode, norm, bmode) in enumerate(G["cases"].tolist()):
        blk = blur_predictor(ro.blur_predictor_params(100 + ci, PS, KS, mode))
        pred = cuda(G["pred"]).clone().requires_grad_(True)
        opt = types.SimpleNamespace(learnable_blur_kernel_size=KS, learnable_blur_kernel_mode=mode, learnable_blur_kernel_norm=norm,
                                    learnable_blur_kernel_conv=0, boundary_mode=bmode)
        m = types.SimpleNamespace(output={"coarse_raycolor": pred}, gt_image=cuda(G["gt"]), dilation_PatchNum=PN, dilation_PatchSize=PS, opt=opt)
        learnable_blur_update_output(m, blk)
        out = m.output["coarse_raycolor"]
        assert_close(out, G[f"c{ci}_out"], RTOL, 1e-6, f"case {ci} out")
        (out * cuda(G["G"])).sum().backward()
        assert_close(pred.grad, G[f"c{ci}_grad_pred"], RTOL, grad_atol(G[f"c{ci}_grad_pred"]), f"case {ci} d pred")
        for li in range(4):
            lin = blk[2 * li]
            assert_close(lin.weight.grad, G[f"c{ci}_gW{li}"], RTOL, grad_atol(G[f"c{ci}_gW{li}"]), f"case {ci} dW{li}")
            assert_close(lin.bias.grad, G[f"c{ci}_gb{li}"], RTOL, grad_atol(G[f"c{ci}_gb{li}"]), f"case {ci} db{li}")


def test_learnable_blur_shipped_shape_vs_oracle():
    """7x7 patches of 8x8, 9x9 predicted kernels, mode 4 / boundary 1 (the *_learnable.sh configuration) vs the oracle, plus the
    identity property: a combine weight of 0 (last predictor bias -> -inf) leaves the rendered colours unchanged."""
    from hybridneuralrendering_b200.blur import learnable_blur
    rng = np.random.default_rng(5)
    PN, PS, KS = 7, 8, 9
    P = ro.blur_predictor_params(7, PS, KS, 4)
    pred, gt = T(rng.random((1, (PN * PS) ** 2, 3), dtype=np.float32)), T(rng.random((1, (PN * PS) ** 2, 3), dtype=np.float32))
    ref, raw_ref = ro.learnable_blur(pred, gt, P, PN, PS, KS, 4, 0, 1)
    out, raw = learnable_blur(pred.cuda(), gt.cuda(), blur_predictor(P), PN, PS, KS, 4, 0, 1)
    assert_close(raw, raw_ref, RTOL, 1e-6)
    assert_close(out, ref, RTOL, 1e-6)
    P[-1][1][-1] = -1e4                          # sigmoid -> 0: kernel = identity
    out, raw = learnable_blur(pred.cuda(), gt.cuda(), blur_predictor(P), PN, PS, KS, 4, 0, 1)
    assert float(raw[:, -1].abs().max()) == 0.0
    assert_close(out, pred, 1e-6, 1e-7)


@pytest.mark.parametrize("M,N,ks,act", [(1, 1, (5,), 0), (130, 256, (284,), 1), (257, 256, (256, 7), 1), (300, 64, (45, 128, 3), 1),
                                         (77, 1, (64,), 2), (64, 3, (45, 83), 3), (1000, 45, (45,), 0), (0, 8, (4,), 1),
                                         # heads at training sizes: small-N weight-gradient kernel with its grid-stride row loop
                                         (40003, 1, (64,), 2), (30011, 3, (45, 83), 3), (5000, 4, (100, 20, 8), 1)])
def test_linear_fwd_bwd_vs_torch(M, N, ks, act):
    from hybridneuralrendering_b200 import ops
    rng = np.random.default_rng(M + N)
    K = sum(ks)
    srcs = [T(rng.standard_normal((M, k)).astype(np.float32)) for k in ks]
    W, b = T((rng.standard_normal((N, K)) * 0.1).astype(np.float32)), T(rng.standard_normal(N).astype(np.float32))
    res = T(rng.standard_normal((M, N)).astype(np.float32)) if act == 0 else None
    G = T(rng.standard_normal((M, N)).astype(np.float32))

    def ref():
        xs = [s.double().clone().requires_grad_(True) for s in srcs]
        Wd, bd = W.double().clone().requires_grad_(True), b.double().clone().requires_grad_(True)
        y = torch.nn.functional.linear(torch.cat(xs, 1), Wd, bd)
        y = [y, torch.nn.functional.leaky_relu(y, 0.01), torch.sigmoid(y), torch.sigmoid(y) * 1.002 - 0.001][act]
        if res is not None:
            y = y + res.double()
        (y * G.double()).sum().backward()
        return y, [x.grad for x in xs], Wd.grad, bd.grad

    y_ref, gx_ref, gW_ref, gb_ref = ref()
    xs = [s.cuda().clone().requires_grad_(True) for s in srcs]
    Wc, bc = W.cuda().clone().requires_grad_(True), b.cuda().clone().requires_grad_(True)
    y = ops.linear(xs, Wc, bc, act, res=res.cuda() if res is not None else None)
    assert_close(y, y_ref, 1e-5, 1e-5)
    if M > 0:
        (y * G.cuda()).sum().backward()
        for a, r in zip(xs, gx_ref):
            assert_close(a.grad, r, 1e-4, grad_atol(r, 1e-5))
        assert_close(Wc.grad, gW_ref, 1e-4, grad_atol(gW_ref, 1e-5))
        assert_close(bc.grad, gb_ref, 1e-4, grad_atol(gb_ref, 1e-5))


def test_linear_strided_sources_and_shared_block():
    """column-slice sources (row stride > width) and a source shared by V row blocks (mods)"""
    from hybridneuralrendering_b200 import ops
    rng = np.random.default_rng(0)
    V, Nv = 3, 50
    g = T(rng.standard_normal((Nv, 128)).astype(np.float32))
    a = T(rng.standard_normal((V * Nv, 45)).astype(np.float32))
    W, b = T((rng.standard_normal((64, 45 + 128)) * 0.1).astype(np.float32)), T(rng.standard_normal(64).astype(np.float32))
    gd, ad, Wd = g.double().requires_grad_(True), a.double().requires_grad_(True), W.double().requires_grad_(True)
    y_ref = torch.nn.functional.leaky_relu(torch.nn.functional.linear(torch.cat([ad, gd.repeat(V, 1)], 1), Wd, b.double()), 0.01)
    y_ref.square().sum().backward()
    gc, ac, Wc = g.cuda().requires_grad_(True), a.cuda().requires_grad_(True), W.cuda().requires_grad_(True)
    y = ops.linear([ac, gc], Wc, b.cuda(), 1, mods=(0, Nv), M=V * Nv)
    assert_close(y, y_ref, 1e-5, 1e-5)
    y.square().sum().backward()
    assert_close(gc.grad, gd.grad, 1e-4, grad_atol(gd.grad, 1e-5))
    assert_close(ac.grad, ad.grad, 1e-4, grad_atol(ad.grad, 1e-5))
    assert_close(Wc.grad, Wd.grad, 1e-4, grad_atol(Wd.grad, 1e-5))
    # slices
    gi, gv = gc[:, :45], gc[:, 45:]
    W2 = T((rng.standard_normal((3, 128)) * 0.1).astype(np.float32)).cuda()
    y2 = ops.linear([gi, gv], W2, None, 0)
    assert_close(y2, g.double() @ W2.cpu().double().t(), 1e-5, 1e-5)


def test_linear_backward_needed_columns_and_narrow_slice():
    """data gradient restricted to the leading columns the caller consumes (layer 0 of the per-neighbour MLP: 224 of 284) and the
    narrow-slice kernel (block3's 7 extra inputs) vs fp64"""
    from hybridneuralrendering_b200 import ops
    rng = np.random.default_rng(3)
    M, N = 3000, 256
    for K, k_need in ((284, 224), (263, None)):
        X = T(rng.standard_normal((M, K)).astype(np.float32))
        W = T((rng.standard_normal((N, K)) * 0.1).astype(np.float32))
        Y = torch.nn.functional.leaky_relu(X.double() @ W.double().t(), 0.01)
        dY = T(rng.standard_normal((M, N)).astype(np.float32))
        ref = (dY.double() * torch.where(Y > 0, 1.0, 0.01)) @ W.double()
        (dX,), dW, db = ops.linear_backward(W.cuda(), Y.float().cuda(), [X.cuda()], (), dY.cuda(), ops.ACT_LRELU, [True], k_need=k_need)
        kk = k_need or K
        assert_close(dX[:, :kk], ref[:, :kk], 1e-4, grad_atol(ref, 1e-5))
        assert_close(dW, (dY.double() * torch.where(Y > 0, 1.0, 0.01)).t() @ X.double(), 1e-4, 1e-3)


def test_fused_adam_matches_torch_adam_dense_semantics():
    """fused dense Adam (SURVEY §8f N2) vs torch.optim.Adam over several steps, including rows whose gradient is zero
    (dense semantics: they still move while their moments decay) and a non-multiple-of-4 tensor"""
    from hybridneuralrendering_b200.optim import FusedAdam
    torch.manual_seed(0)
    shapes = [(1, 5000, 32), (1, 5000, 1), (777,), (3, 3)]
    pa = [torch.nn.Parameter(torch.randn(s, device="cuda")) for s in shapes]
    pb = [torch.nn.Parameter(p.detach().clone()) for p in pa]
    oa = FusedAdam(pa, lr=2e-3, betas=(0.9, 0.999), eps=1e-8)
    ob = torch.optim.Adam(pb, lr=2e-3, betas=(0.9, 0.999), eps=1e-8)
    for it in range(5):
        for a, b in zip(pa, pb):
            g = torch.randn_like(a) * (10.0 ** (-it))
            if a.dim() == 3:
                g[:, ::3] = 0                                       # untouched rows
            a.grad, b.grad = g.clone(), g.clone()
        oa.step(); ob.step()
    for a, b in zip(pa, pb):
        assert_close(a, b, 1e-6, 1e-7)


@pytest.mark.parametrize("V,H,W", [(2, 48, 64), (3, 37, 51), (1, 121, 162)])
def test_own_pyramid_kernels_match_torch_conv(V, H, W):
    """csrc/pyramid.cu (six 3x3 convolutions + LeakyReLU, NHWC, exact fp32) vs torch conv2d in fp64: the three levels, and every weight /
    bias gradient for random level gradients (odd sizes included: stride-2 output size floor((H-1)/2)+1)"""
    from hybridneuralrendering_b200 import ops
    from hybridneuralrendering_b200.point_aggregators import _conv_block
    torch.manual_seed(V * H)
    blocks = [_conv_block(3, 6).cuda(), _conv_block(6, 12).cuda(), _conv_block(12, 24).cuda()]
    for blk in blocks:
        for m in (blk[0], blk[2]):
            torch.nn.init.normal_(m.weight, std=0.3)
            torch.nn.init.normal_(m.bias, std=0.1)
    params = []
    for blk in blocks:
        params += [blk[0].weight, blk[0].bias, blk[2].weight, blk[2].bias]
    img = torch.rand(V, H, W, 3, device="cuda")
    lv = ops.PyramidFn.apply(img, *params)
    gs = [torch.randn_like(t) for t in lv]
    gs[1][:, ::3] = 0                          # sparse level gradients, like the image gather's scatter
    torch.autograd.backward(lv, gs)
    got = [p.grad.clone() for p in params]
    # fp64 reference
    pd = [p.detach().double().requires_grad_(True) for p in params]
    x = img.double().permute(0, 3, 1, 2)
    outs = []
    for i in range(3):
        x = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(x, pd[4 * i], pd[4 * i + 1], stride=2, padding=1), 0.01)
        x = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(x, pd[4 * i + 2], pd[4 * i + 3], stride=1, padding=1), 0.01)
        outs.append(x)
    for a, b in zip(lv, outs):
        assert a.shape == b.permute(0, 2, 3, 1).shape
        assert_close(a, b.permute(0, 2, 3, 1), 1e-5, 2e-6 * float(b.abs().max()))
    # gradients: drop upstream gradient where a pre-activation is within 1e-6 of the LeakyReLU kink? not needed: fp32 vs fp64 on the
    # same side of 0 except for |x| < 1e-7 -- measure-zero for these random inputs
    torch.autograd.backward(outs, [g.double().permute(0, 3, 1, 2) for g in gs])
    for a, r in zip(got, pd):
        assert_close(a, r.grad, 1e-4, 1e-5 * float(r.grad.abs().max()))


def test_fused_training_loss_matches_torch():
    """csrc/loss.cu: masked MSE (+1e-6) x frame_weight + 1e-4 x zero-one regulariser (base_rendering_model.py:1114-1118, :1229-1240) in
    one launch vs the same expression in torch fp64 -- value and both gradients, incl. conf values outside the clamp"""
    from hybridneuralrendering_b200.renderer import training_loss
    g = torch.Generator().manual_seed(3)
    R, Rk, SR, K = 500, 333, 24, 8
    ids = torch.randperm(R, generator=g)[:Rk].sort()[0].int().cuda()
    color = torch.rand(1, Rk, 3, generator=g).cuda().requires_grad_(True)
    cc = (torch.rand(1, Rk, SR, K, generator=g) * 1.2 - 0.1).cuda().requires_grad_(True)        # some values beyond [1e-3, 1 - 1e-3]
    gt = torch.rand(1, R, 3, generator=g).cuda()
    out = {"coarse_raycolor": color, "conf_coefficient": cc, "ray_ids": ids, "ray_mask": None}
    loss = training_loss(out, gt, 1e-4, 0.7)
    (loss * 3.0).backward()
    c64, cc64 = color.detach().double().requires_grad_(True), cc.detach().double().requires_grad_(True)
    v = cc64.clamp(1e-3, 1 - 1e-3)
    ref = (torch.nn.functional.mse_loss(c64, gt.double()[:, ids.long()]) + 1e-6) * 0.7 + 1e-4 * torch.mean(torch.log(v) + torch.log(1 - v))
    (ref * 3.0).backward()
    assert_close(loss, ref, 1e-5, 1e-8)
    assert_close(color.grad, c64.grad, 1e-5, 1e-10)
    assert_close(cc.grad, cc64.grad, 1e-5, 1e-12)
    # the block partials are added in a fixed order: the same value in every run, whatever order the blocks finish in
    with torch.no_grad():
        again = [training_loss(out, gt, 1e-4, 0.7) for _ in range(50)]
    assert all(torch.equal(a, loss.detach()) for a in again)


@pytest.mark.parametrize("world,n", [(1, 64), (3, 4096), (8, 354624)])
def test_peer_sum_kernel_sums_in_rank_order(world, n):
    """csrc/peer.cu on one device: `world` local buffers stand in for the peers' copies of the symmetric buffer.  The sum must be the
    fp32 sum in rank order (what makes the result bit-identical on every rank of a data-parallel run); the multi-process path over
    real NVLink peers is checked by scripts/check_peer_allreduce.py against NCCL (bit-identical replicas, 2 and 8 GPUs)."""
    import ctypes as C
    from hybridneuralrendering_b200._lib import check, lib, ptr
    g = torch.Generator(device="cuda").manual_seed(world)
    bufs = [torch.randn(n, device="cuda", generator=g) * (10.0 ** (r % 3)) for r in range(world)]
    out = torch.empty(n, device="cuda")
    arr = (C.c_void_p * world)(*[b.data_ptr() for b in bufs])
    check(lib().hnr_peer_sum_f32(arr, world, n, ptr(out), None), "peer_sum")
    ref = torch.zeros(n, device="cuda")
    for b in bufs:
        ref = ref + b                      # same order, same fp32 additions
    assert torch.equal(out, ref)
    with pytest.raises(RuntimeError):
        check(lib().hnr_peer_sum_f32(arr, world, n - 1, ptr(out), None), "peer_sum")          # n % 4 != 0 is rejected


def test_strided_blend_and_image_gather_backward_match_the_dense_entry_points():
    """the 48-wide aligned training rows [aux 45 | dview 3]: hnr_blend_bwd_ld / hnr_image_gather_bwd_ld on strided rows give what the
    45-wide entry points give on packed rows (padding columns of d_aux zero-filled, columns >= 45 of the incoming gradient ignored)"""
    from hybridneuralrendering_b200 import ops
    from hybridneuralrendering_b200._lib import check, i64_array, lib, ptr, ptr_array
    rng = np.random.default_rng(11)
    V, Nv, S = 3, 517, 700
    aux = cuda(rng.standard_normal((V, Nv, 45)).astype(np.float32))
    aux48 = torch.zeros((V, Nv, 48), device="cuda"); aux48[..., :45] = aux; aux48[..., 45:] = 7.0
    sig = cuda(rng.random((V * Nv, 1)).astype(np.float32))
    okm = cuda((rng.random((V, Nv)) > 0.2).astype(np.float32))
    keep = cuda((rng.random(Nv) > 0.3).astype(np.uint8))
    dm = cuda(rng.standard_normal((Nv, 45)).astype(np.float32))
    d_aux, d_sig = torch.empty_like(aux), torch.empty_like(sig)
    check(lib().hnr_blend_bwd(ptr(aux), ptr(sig), ptr(okm), ptr(keep), ptr(dm), V, Nv, ptr(d_aux), ptr(d_sig), None), "blend_bwd")
    d_aux48, d_sig2 = torch.full_like(aux48, float("nan")), torch.empty_like(sig)
    check(lib().hnr_blend_bwd_ld(ptr(aux48), 48, ptr(sig), ptr(okm), ptr(keep), ptr(dm), V, Nv, ptr(d_aux48), 48, ptr(d_sig2), None), "blend_bwd_ld")
    assert torch.equal(d_aux48[..., :45], d_aux) and torch.equal(d_sig2, d_sig) and float(d_aux48[..., 45:].abs().max()) == 0.0
    # image-gather backward: gradient rows 45 vs 48 wide
    H, W = 24, 32
    shapes = [(V, H, W, 3), (V, 12, 16, 6), (V, 6, 8, 12), (V, 3, 4, 24)]
    hw = [x for s in shapes for x in s[1:3]]
    xy = cuda((rng.random((V, S, 2)) * np.array([W + 4, H + 4]) - 2).astype(np.float32))
    vlist = cuda(np.sort(rng.choice(S, Nv, replace=False)).astype(np.int32))
    g45 = cuda(rng.standard_normal((V, Nv, 45)).astype(np.float32))
    g48 = torch.full((V, Nv, 48), 3.0, device="cuda"); g48[..., :45] = g45
    res = []
    for g, ld in ((g45, 45), (g48, 48)):
        grads = [None] + [torch.zeros(s, device="cuda") for s in shapes[1:]]
        check(lib().hnr_image_gather_bwd_ld(ptr_array(grads), i64_array(hw), ptr(xy), ptr(vlist), ptr(g), ld, V, S, Nv, None), "image_gather_bwd_ld")
        res.append(grads[1:])
    for a, b in zip(*res):
        assert float((a - b).abs().max()) <= 1e-5 * float(a.abs().max() + 1e-30)          # atomics: arrival order only


@pytest.mark.parametrize("M,K,act", [(5000, 64, 2), (777, 128, 2), (130, 64, 1), (300, 45, 2)])
def test_one_pass_head_backward_matches_torch(M, K, act):
    """ops.linear_head_backward (one pass over y for a one-output layer; generic kernels for widths other than 64 / 128) vs autograd"""
    from hybridneuralrendering_b200 import ops
    rng = np.random.default_rng(M + K)
    y = cuda(rng.standard_normal((M, K)).astype(np.float32))
    W = cuda((rng.standard_normal((1, K)) * 0.3).astype(np.float32))
    b = cuda(np.array([0.1], np.float32))
    dH = cuda(rng.standard_normal((M, 1)).astype(np.float32))
    yd, Wd, bd = y.double().requires_grad_(True), W.double().requires_grad_(True), b.double().requires_grad_(True)
    pre = yd @ Wd.t() + bd
    hd = torch.sigmoid(pre) if act == 2 else torch.nn.functional.leaky_relu(pre, 0.01)
    hd.backward(dH.double())
    dY, dW, db = ops.linear_head_backward(W, hd.detach().float(), y, dH, act)
    assert dW.shape == W.shape and db.shape == b.shape
    assert_close(dY, yd.grad, RTOL, grad_atol(yd.grad))
    assert_close(dW, Wd.grad, RTOL, grad_atol(Wd.grad))
    assert_close(db, bd.grad, RTOL, grad_atol(bd.grad))
