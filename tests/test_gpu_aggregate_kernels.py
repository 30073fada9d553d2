"""The aggregation glue (csrc/aggregate.cu) and the image-branch kernels (csrc/aggregate.cu, csrc/pyramid.cu), each alone through the
C ABI against an fp64 reference on the GPU (tests/helpers.py ref_*, written from oracle/render_oracle.py and checked against it by
test_oracle_golden.test_kernel_references_match_oracle), at the benchmark's sizes and at the edges where these kernels can go wrong:
fully masked samples and slots that alias point 0, both sides of the grid-stride caps, points shared by thousands of rows, out-of-bounds
and zeroed pixels, both launch paths of the image gather, 48-wide padded rows, and the multi-row weight-gradient strips of the pyramid
backward.  Forward outputs: rtol 1e-5 with a stated atol, exact where the kernel copies or clamps.  Gradients: 1e-4 x the tensor's
max magnitude (helpers.grad_atol) plus a per-point / per-row bound where rows span orders of magnitude.  Each tolerance is stated at
its assert."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from hybridneuralrendering_b200 import mlp_tc, ops  # noqa: E402
from hybridneuralrendering_b200._lib import check, i64_array, lib, ptr, ptr_array, stream  # noqa: E402

from helpers import (PYRAMID_STRIDES, grad_atol, ref_alpha_ksum, ref_blend, ref_image_gather, ref_nbr_features,  # noqa: E402
                     ref_nbr_weights, ref_pyramid)

NUM_SMS = 148           # HNR_NUM_SMS (csrc/common.cuh): the launchers size their grids in multiples of it
D = torch.float64


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _close(got, ref, rtol, atol, what):
    """|got - ref| <= atol + rtol |ref| elementwise (atol may be a tensor broadcast against ref; a zero tolerance demands equality);
    prints the largest deviation as a fraction of the tolerance"""
    got, ref = got.detach().double(), ref.detach().double()
    frac = float(((got - ref).abs() / (atol + rtol * ref.abs()).clamp_min(1e-300)).max()) if ref.numel() else 0.0
    print(f"DEV {what}: {frac:.3g}")
    assert frac <= 1.0, (what, frac)


def _grad_close(got, ref, what, scale=None):
    """the standing gradient bar: |got - ref| <= 1e-4 x max |ref|; with `scale` (broadcast against ref) also the per-row / per-point
    bound |got - ref| <= 1e-4 x scale"""
    _close(got, ref, 0.0, grad_atol(ref), what)
    if scale is not None:
        _close(got, ref, 0.0, 1e-4 * scale.double() + 1e-30, what + " (per row)")


def _rotation(g):
    q, r = torch.linalg.qr(torch.randn(3, 3, device="cuda", generator=g, dtype=D))
    return (q * torch.sign(torch.diagonal(r))).float()


def _camera(g):
    """ops.make_cam block for a camera 3 units behind the unit box: c2w rotation about its optical (z) axis, so that every point of
    the box stays 2..4 units deep; random world->camera rotation Rw2c"""
    campos = torch.tensor([0.3, -0.2, -3.0], device="cuda")
    c, s = float(np.cos(0.5)), float(np.sin(0.5))
    camrot = torch.tensor([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]], device="cuda")
    return ops.make_cam(campos, camrot, _rotation(g)), campos


def _pers(p, cam):
    c = (p - cam[:3]) @ cam[3:12].reshape(3, 3)
    return torch.stack([c[:, 0] / c[:, 2], c[:, 1] / c[:, 2], c[:, 2]], -1)


def _unit(g, n):
    v = torch.randn(n, 3, device="cuda", generator=g)
    return v / v.norm(dim=-1, keepdim=True)


def _scatter_ref(n, idx, terms):
    """fp64 index_add of per-row terms (rows, C) into n points, and the sum of their magnitudes (the per-point scale)"""
    z = torch.zeros((n,) + terms.shape[1:], device="cuda", dtype=D)
    return z.index_add(0, idx, terms), z.index_add(0, idx, terms.abs())


# ---------------------------------------------------------------------------------------------------------- weights, confidence
def _nbr_weights(xyz, conf, pidx, mask, loc_w, outs=True):
    S, K = pidx.shape
    w = torch.full((S, K), float("nan"), device="cuda")
    cc = torch.full((S, K), float("nan"), device="cuda") if outs else None
    valid = torch.full((S,), 7, device="cuda", dtype=torch.uint8) if outs else None
    check(lib().hnr_nbr_weights(ptr(xyz), ptr(conf), ptr(pidx), ptr(mask), ptr(loc_w), S, K, ptr(w), ptr(cc), ptr(valid), stream()), "nbr_weights")
    return w, cc, valid


@pytest.mark.parametrize("by_mask", [False, True])
@pytest.mark.parametrize("K", [8, 5])
def test_nbr_weights_and_conf_gradient(K, by_mask):
    """hnr_nbr_weights: all-masked samples, one live slot, a neighbour at distance 0 (the 1e-6 clamp), masking by pidx < 0 or by an
    explicit mask over pidx >= 0, conf below / above / on the clamp bounds; then NbrWeightsFn's backward through hnr_conf_bwd (the clamp
    is straight-through: every slot's gradient reaches its point, masked slots reach point 0)"""
    g = _gen(10 * K + by_mask)
    N, S = 5000, 3000
    xyz = torch.rand(N, 3, device="cuda", generator=g) * 2 - 1
    pidx = torch.randint(1, N, (S, K), device="cuda", generator=g, dtype=torch.int32)
    pidx.view(-1)[3 * K:3 * K + 200] = torch.arange(200, device="cuda", dtype=torch.int32)        # the points with edge confidences
    dead = torch.rand(S, K, device="cuda", generator=g) < 0.3
    dead[0] = True                                    # every slot masked: weights 0, valid 0
    dead[1] = True
    dead[1, K // 2] = False                           # exactly one live slot: weight 1
    dead[2] = False
    loc_w = xyz[pidx[:, 0].long()] + 0.05 * torch.randn(S, 3, device="cuda", generator=g)
    loc_w[2] = xyz[pidx[2, 1].long()]                 # a neighbour at distance 0: 1 / max(|d|, 1e-6)
    mask = (~dead).to(torch.uint8) if by_mask else None
    if not by_mask:
        pidx[dead] = -1
    conf = torch.rand(N, device="cuda", generator=g) * 1.4 - 0.2
    conf[:200] = torch.tensor([np.float32(1e-4), 1.0, 5e-5, 1.5, -0.1], device="cuda").repeat(40)       # on both bounds, below, above
    w, cc, valid = _nbr_weights(xyz, conf, pidx, mask, loc_w)
    rw, rc, rv = ref_nbr_weights(xyz.double(), conf.double(), pidx, mask, loc_w.double())
    live = (mask != 0) if by_mask else (pidx >= 0)
    assert torch.equal(valid, rv.to(torch.uint8)) and int(valid[0]) == 0 and int(valid[1]) == 1        # exact
    assert torch.equal(cc.double(), rc)                                      # a clamp of the table value: exact
    assert float(w[~live].abs().max()) == 0.0                                # masked slots: exactly 0
    assert float(w[2, 1]) > 0.999
    # fp32: a norm, two reciprocals and a K-term sum per sample: a few ulp; atol 0 (the smallest weights, 1e-8 next to the clamped
    # distance, are held to the same relative bound)
    _close(w, rw, 1e-5, 0.0, "nbr_weights weight")
    w2, _, _ = _nbr_weights(xyz, None, pidx, mask, loc_w, outs=False)        # conf NULL, confc / valid NULL
    assert torch.equal(w2, w)
    _, cc1, _ = _nbr_weights(xyz, None, pidx, mask, loc_w)
    assert float((cc1 - 1).abs().max()) == 0.0                               # no confidence table: 1 exactly
    # backward: d conf = index_add over all S*K slots of the upstream gradient
    cg = conf.clone().requires_grad_(True)
    _, confc, _ = ops.NbrWeightsFn.apply(xyz, cg, pidx, mask, loc_w)
    up = torch.randn(S, K, device="cuda", generator=g)
    confc.backward(up)
    ref, mag = _scatter_ref(N, pidx.long().clamp_min(0).view(-1), up.double().view(-1))
    _grad_close(cg.grad, ref, "conf_up_bwd d_conf", mag)


@pytest.mark.parametrize("terms", ["regulariser", "cancelling"])
def test_conf_bwd_at_benchmark_size(terms):
    """hnr_conf_bwd at configs[2]'s 4096 rays x SR 24 x K 8 = 786k slots, >= 300k of them masked (all alias point 0), 16 hot points shared
    by ~2.4k slots each; both kernels (the d_wc term of the vlist samples, the upstream conf_coefficient gradient of every slot).
    Masked slots all carry the same gradient, as the zero-one regulariser gives them (they all read conf[0]); 'cancelling' adds +-2^20
    pairs on the first masked slots, which an fp32 running sum per thread would let swallow the small terms after them."""
    g = _gen(11 + (terms == "cancelling"))
    R, SR, K, N = 4096, 24, 8, 200_000
    S = R * SR
    pidx = torch.randint(17, N, (S, K), device="cuda", generator=g, dtype=torch.int32)      # point 0 only through masked slots
    hot = torch.rand(S, K, device="cuda", generator=g) < 0.05
    pidx[hot] = torch.randint(1, 17, (int(hot.sum()),), device="cuda", generator=g, dtype=torch.int32)
    dead = torch.rand(S, K, device="cuda", generator=g) < 0.4
    dead[torch.rand(S, device="cuda", generator=g) < 0.1] = True                               # fully masked samples
    pidx[dead] = -1
    d_confc = torch.randn(S, K, device="cuda", generator=g) * 1e-3
    d_confc[dead] = float(np.float32(1.2345678e-4))
    if terms == "cancelling":
        pidx.view(-1)[:512] = -1
        d_confc.view(-1)[:512] = torch.tensor([2.0 ** 20, -2.0 ** 20], device="cuda").repeat(256)
    n_masked = int((pidx < 0).sum())
    assert n_masked >= 300_000
    valid = (pidx >= 0).any(1)
    vlist = valid.nonzero()[:, 0].to(torch.int32)
    Nv = vlist.shape[0]
    weight = torch.rand(S, K, device="cuda", generator=g) * (pidx >= 0)
    d_wc = torch.randn(Nv, K, device="cuda", generator=g)
    d_conf = torch.zeros(N, device="cuda")
    check(lib().hnr_conf_bwd(ptr(d_wc), ptr(weight), ptr(vlist), ptr(pidx), ptr(d_confc), Nv, S, K, ptr(d_conf), stream()), "conf_bwd")
    vl = vlist.long()
    idx = torch.cat([pidx.long().clamp_min(0).view(-1), pidx[vl].long().clamp_min(0).view(-1)])
    t = torch.cat([d_confc.double().view(-1), (d_wc.double() * weight[vl].double()).view(-1)])
    ref, mag = _scatter_ref(N, idx, t)
    # every point: the standing bar and 1e-4 x the sum of its terms' magnitudes (hot points: thousands of fp32 atomics)
    _grad_close(d_conf, ref, f"conf_bwd d_conf ({terms})", mag)
    # point 0: hundreds of thousands of terms.  The kernel sums them in double per thread and per block and adds <= 296 block sums in
    # fp32: relative error ~1e-6.  Bound 1e-5 x |d_conf[0]|
    r0 = float(ref[0])
    _close(d_conf[:1], ref[:1], 1e-5, 0.0, f"conf_bwd d_conf[0] ({terms})")
    if terms == "regulariser":
        # an fp32 running sum of the same terms in slot order (what serialised same-address atomics compute) misses that bound
        seq = float(np.add.accumulate(d_confc[pidx < 0].cpu().numpy(), dtype=np.float32)[-1])
        print(f"DEV conf_bwd fp32 sequential sum of the {n_masked} point-0 terms: relative error {abs(seq - r0) / abs(r0):.3g}")
        assert abs(seq - r0) > 1e-5 * abs(r0)


# ---------------------------------------------------------------------------------------------------------- MLP input rows
def _nbr_case(g, N, S, K, Nv, dead_frac=0.3):
    """point tables near a unit box, samples whose first neighbour lies within ~0.05 (like the query's output), an unsorted vlist
    with gaps"""
    xyz = torch.rand(N, 3, device="cuda", generator=g) * 2 - 1
    pidx = torch.randint(0, N, (S, K), device="cuda", generator=g, dtype=torch.int32)
    dead = torch.rand(S, K, device="cuda", generator=g) < dead_frac
    loc_w = xyz[pidx[:, 0].long()] + 0.05 * torch.randn(S, 3, device="cuda", generator=g)
    vlist = torch.randperm(S, device="cuda", generator=g)[:Nv].to(torch.int32)
    return xyz, pidx, dead, loc_w, vlist


@pytest.mark.parametrize("pers", ["table", "from_cam"])
def test_nbr_features_match_fp64(pers):
    """hnr_nbr_features: X0 = [emb | PE(emb) | PE(d)] (284 columns) and E = [colour | dirR - viewR | <dirR, viewR>] (7) for every
    (vlist sample, slot), with the point's perspective coordinates from the table or computed from cam (xyz_pers NULL)"""
    g = _gen(21 + (pers == "table"))
    N, S, K, Nv = 20000, 6000, 8, 4500
    xyz, pidx, dead, loc_w, vlist = _nbr_case(g, N, S, K, Nv)
    pidx[dead] = -1
    cam, _ = _camera(g)
    xyz_pers, loc_pers = _pers(xyz, cam), _pers(loc_w, cam)
    emb = torch.randn(N, 32, device="cuda", generator=g) * 1.5
    color, dirs, rays = torch.rand(N, 3, device="cuda", generator=g), _unit(g, N), _unit(g, S)
    X0 = torch.full((Nv * K, 284), float("nan"), device="cuda")
    E = torch.full((Nv * K, 7), float("nan"), device="cuda")
    xp = xyz_pers if pers == "table" else None
    check(lib().hnr_nbr_features(ptr(xyz), ptr(xp), ptr(emb), ptr(color), ptr(dirs), ptr(pidx), ptr(vlist), ptr(loc_w), ptr(loc_pers), ptr(rays),
                                 ptr(cam), Nv, K, 32, ptr(X0), ptr(E), stream()), "nbr_features")
    rX0, rE = ref_nbr_features(xyz.double(), xp.double() if xp is not None else None, emb.double(), color.double(), dirs.double(), pidx, vlist,
                               loc_w.double(), loc_pers.double(), rays.double(), cam.double())
    assert torch.equal(X0[:, :32].double(), rX0[:, :32]) and torch.equal(E[:, :3].double(), rE[:, :3])        # copies: exact
    # PE(emb): sincosf of the exact fp32 argument e * 2^f: <= 2 ulp of a value in [-1, 1] (~1.2e-7); atol 1e-6
    _close(X0[:, 32:224], rX0[:, 32:224], 0.0, 1e-6, "nbr_features PE(emb)")
    # PE(d): the argument is 2^f d with d computed in fp32 from coordinates of magnitude <= 4 (rotations, a division, products that
    # cancel: <= ~1e-6 absolute), so it carries 2^f times that: atol 1e-6 (sincosf) + 1e-6 x 2^f for the columns of frequency f
    f = (torch.arange(60, device="cuda") // 2) % 5
    _close(X0[:, 224:], rX0[:, 224:], 0.0, 1e-6 * (1 + 2.0 ** f.double()), "nbr_features PE(d)")
    # rotations of unit vectors and their dot product in fp32: rtol 1e-5, atol 1e-6
    _close(E[:, 3:], rE[:, 3:], 1e-5, 1e-6, "nbr_features E")


@pytest.mark.parametrize("by_mask", [False, True])
@pytest.mark.parametrize("ldx", [284, 224])
def test_nbr_features_bwd_match_fp64(ldx, by_mask):
    """hnr_nbr_features_bwd (ldx 284) / _ld (224, the fused chain's width): d_emb, d_color, d_dir = the fp64 adjoint of the MLP input
    rows scattered by index_add, with one point shared by >= 10k live rows; masked rows (pidx < 0, or an explicit mask over pidx >= 0) carry
    NaN gradients, which must not reach any output; each output may be NULL on its own"""
    g = _gen(31 + ldx + by_mask)
    N, S, K, Nv = 30000, 6000, 8, 5000
    xyz, pidx, dead, loc_w, vlist = _nbr_case(g, N, S, K, Nv)
    slots = (vlist.long()[:, None] * K + torch.arange(K, device="cuda")).view(-1)
    pidx.view(-1)[slots[torch.randperm(slots.numel(), device="cuda", generator=g)[:15000]]] = 5           # a hot point
    mask = (~dead).to(torch.uint8) if by_mask else None
    if not by_mask:
        pidx[dead] = -1
    cam, _ = _camera(g)
    emb = torch.randn(N, 32, device="cuda", generator=g) * 1.5
    rays = _unit(g, S)
    rows = Nv * K
    dX0 = torch.randn(rows, ldx, device="cuda", generator=g)
    dE = torch.randn(rows, 7, device="cuda", generator=g)
    rdead = dead[vlist.long()].view(-1)
    dX0[rdead], dE[rdead] = float("nan"), float("nan")
    assert int((~rdead & (pidx[vlist.long()].view(-1) == 5)).sum()) >= 10000
    # fp64 adjoint per live row
    lr = (~rdead).nonzero()[:, 0]
    s = vlist.long().repeat_interleave(K)[lr]
    gi = pidx[vlist.long()].view(-1)[lr].long()
    e = emb[gi].double()
    dx, de = dX0[lr].double(), dE[lr].double()
    fr = 2.0 ** torch.arange(3, device="cuda", dtype=D)
    a = e[..., None] * fr
    dpe = dx[:, 32:224].view(-1, 32, 3, 2)
    t_emb = dx[:, :32] + (fr * (a.cos() * dpe[..., 0] - a.sin() * dpe[..., 1])).sum(-1)
    m_emb = dx[:, :32].abs() + (fr * ((a.cos() * dpe[..., 0]).abs() + (a.sin() * dpe[..., 1]).abs())).sum(-1)
    rt = cam[12:21].reshape(3, 3).double()
    gv = de[:, 3:6] + de[:, 6:7] * (rays[s].double() @ rt)
    refs = [_scatter_ref(N, gi, t_emb)[0], _scatter_ref(N, gi, de[:, :3])[0], _scatter_ref(N, gi, gv @ rt.t())[0]]
    mags = [_scatter_ref(N, gi, m_emb)[0], _scatter_ref(N, gi, de[:, :3])[1], _scatter_ref(N, gi, (de[:, 3:6].abs() + (de[:, 6:7] * (rays[s].double() @ rt)).abs()) @ rt.t().abs())[0]]
    names = ("d_emb", "d_color", "d_dir")
    for sel in ((1, 1, 1), (1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 1, 1)):
        outs = [torch.zeros(N, c, device="cuda") if on else None for on, c in zip(sel, (32, 3, 3))]
        if ldx == 284:
            check(lib().hnr_nbr_features_bwd(ptr(dX0), ptr(dE), ptr(emb), ptr(pidx), ptr(mask), ptr(vlist), ptr(rays), ptr(cam), Nv, K,
                                             ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), stream()), "nbr_features_bwd")
        else:
            check(lib().hnr_nbr_features_bwd_ld(ptr(dX0), ldx, ptr(dE), ptr(emb), ptr(pidx), ptr(mask), ptr(vlist), ptr(rays), ptr(cam), Nv, K,
                                                ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), stream()), "nbr_features_bwd_ld")
        for o, r, m, nm in zip(outs, refs, mags, names):
            if o is not None:
                assert bool(torch.isfinite(o).all()), nm                      # no masked row was read
                # the standing bar, and per point 1e-4 x the sum of its terms' magnitudes (>= 10k fp32 atomics on the hot point)
                _grad_close(o, r, f"nbr_features_bwd {nm}", m)


# ---------------------------------------------------------------------------------------------------------- density head + K-sum
@pytest.mark.parametrize("Nv,K", [(1, 8), (4735, 8), (4737, 8), (9471, 8), (9473, 8), (80000, 8), (1, 5), (9473, 5)])
def test_alpha_ksum_match_fp64(Nv, K):
    """hnr_alpha_ksum_fwd, hnr_alpha_ksum_bwd (<8> for K = 8, the generic <0> otherwise) and hnr_alpha_ksum_bwd_img (K = 8), on both
    sides of the grid-stride caps (one pass covers 4 * 148 * 8 = 4736 samples in the image variant, 8 * 148 * 8 = 9472 in the plain
    one) and at the benchmark's sample count; softplus inputs on both sides of its x > 20 branch"""
    assert (4 * NUM_SMS * 8, 8 * NUM_SMS * 8) == (4736, 9472)
    g = _gen(Nv * 10 + K)
    S = Nv + Nv // 2 + 3
    rows = Nv * K
    vlist = torch.randperm(S, device="cuda", generator=g)[:Nv].to(torch.int32)
    vl = vlist.long()
    H = torch.nn.functional.leaky_relu(torch.randn(rows, 256, device="cuda", generator=g), 0.01)
    weight = torch.rand(S, K, device="cuda", generator=g) * (torch.rand(S, K, device="cuda", generator=g) > 0.2)
    weight = weight / weight.sum(1, keepdim=True).clamp_min(1e-8)
    confc = torch.rand(S, K, device="cuda", generator=g) * (1 - 1e-4) + 1e-4
    w_alpha = torch.randn(256, device="cuda", generator=g) * 0.25
    b_alpha = torch.tensor([18.0], device="cuda")            # raw - 1 ~ 17 +- 3: both sides of the threshold 20
    cam, _ = _camera(g)
    rays = _unit(g, S)
    sigma = torch.full((Nv, 1), float("nan"), device="cuda")
    X5 = torch.full((Nv, 280), float("nan"), device="cuda")
    araw = torch.full((rows,), float("nan"), device="cuda")
    check(lib().hnr_alpha_ksum_fwd(ptr(H), ptr(weight), ptr(confc), ptr(vlist), ptr(w_alpha), ptr(b_alpha), ptr(rays), ptr(cam), Nv, K, 256,
                                   ptr(sigma), ptr(X5), ptr(araw), stream()), "alpha_ksum_fwd")
    view = rays[vl].double() @ cam[12:21].reshape(3, 3).double()
    wc = (weight[vl].double() * confc[vl].double()).requires_grad_(True)
    Hd, wad, bad = H.double().requires_grad_(True), w_alpha.double().requires_grad_(True), b_alpha.double().requires_grad_(True)
    rs, rX5, rraw = ref_alpha_ksum(Hd, wc, wad, bad, view)
    if rows > 100:
        assert bool((rraw - 1 > 20).any()) and bool((rraw - 1 < 20).any())
    # raw: a 256-term fp32 dot (|terms| sum ~40, result ~18): ~1e-6 relative
    _close(araw, rraw, 1e-5, 0.0, "alpha_ksum_fwd alpha_raw")
    _close(sigma[:, 0], rs, 1e-5, 1e-6, "alpha_ksum_fwd sigma")
    # 8-term weighted sums of O(1) values that may cancel: rtol 1e-5, atol 1e-6
    _close(X5[:, :256], rX5[:, :256], 1e-5, 1e-6, "alpha_ksum_fwd X5 K-sum")
    # view encoding: sincosf of 2^f x (a rotated unit vector, fp32: ~1e-7): atol 1e-6 x 2^f for the columns of frequency f
    f = (torch.arange(24, device="cuda") % 12) % 4
    _close(X5[:, 256:], rX5[:, 256:], 0.0, 1e-6 * 2.0 ** f.double(), "alpha_ksum_fwd X5 view encoding")
    # backward from the kernel's own alpha_raw, like the product
    d_sigma = torch.randn(Nv, 1, device="cuda", generator=g)
    dX5 = torch.randn(Nv, 280, device="cuda", generator=g)
    (rs * d_sigma[:, 0].double()).sum().add((rX5[:, :256] * dX5[:, :256].double()).sum()).backward()
    dH = torch.full_like(H, float("nan"))
    d_wc = torch.full((Nv, K), float("nan"), device="cuda")
    d_wa, d_ba = torch.zeros(256, device="cuda"), torch.zeros(1, device="cuda")
    check(lib().hnr_alpha_ksum_bwd(ptr(H), ptr(weight), ptr(confc), ptr(vlist), ptr(w_alpha), ptr(araw), ptr(d_sigma), ptr(dX5), Nv, K, 256,
                                   ptr(dH), ptr(d_wc), ptr(d_wa), ptr(d_ba), stream()), "alpha_ksum_bwd")
    # dH rows scale with wc (0 for masked slots): per row 1e-4 x the row's max magnitude
    _grad_close(dH, Hd.grad, f"alpha_ksum_bwd<{8 if K == 8 else 0}> dH", Hd.grad.abs().amax(1, keepdim=True))
    # d_wc = softplus(raw - 1) d_sigma + <H, dX5>: per element 1e-4 x the magnitude of its terms
    sp = torch.nn.functional.softplus(rraw.detach() - 1).view(Nv, K) * d_sigma.double()
    hd_mag = (H.double().abs().view(Nv, K, 256) * dX5[:, None, :256].double().abs()).sum(-1)
    _grad_close(d_wc, wc.grad, f"alpha_ksum_bwd<{8 if K == 8 else 0}> d_wc", sp.abs() + hd_mag)
    _grad_close(d_wa, wad.grad, f"alpha_ksum_bwd<{8 if K == 8 else 0}> d_walpha")
    _grad_close(d_ba, bad.grad, f"alpha_ksum_bwd<{8 if K == 8 else 0}> d_balpha")
    if K != 8:
        return
    # image variant: H_3 as a bf16 hi/lo split image; the fp64 reference runs on the joined image values, the result is the gated
    # gradient dZ_3 = dH * LeakyReLU'(H_3) as a split image
    h3 = mlp_tc.dense_to_image(H)
    Hj = mlp_tc.image_to_dense(h3, rows, 256)
    wcj = wc.detach().clone().requires_grad_(True)
    Hjd, waj, baj = Hj.double().requires_grad_(True), w_alpha.double().requires_grad_(True), b_alpha.double().requires_grad_(True)
    rs2, rX52, rraw2 = ref_alpha_ksum(Hjd, wcj, waj, baj, view)
    (rs2 * d_sigma[:, 0].double()).sum().add((rX52[:, :256] * dX5[:, :256].double()).sum()).backward()
    rdz = Hjd.grad * torch.where(Hj > 0, 1.0, 0.01).double()
    dz = mlp_tc.image_empty(rows, 256, "cuda")
    d_wc2 = torch.full((Nv, K), float("nan"), device="cuda")
    d_wa2, d_ba2 = torch.zeros(256, device="cuda"), torch.zeros(1, device="cuda")
    d_confc = torch.zeros(S, K, device="cuda")
    check(lib().hnr_alpha_ksum_bwd_img(ptr(h3), ptr(weight), ptr(confc), ptr(vlist), ptr(w_alpha), ptr(araw), ptr(d_sigma), ptr(dX5), Nv, K,
                                       ptr(dz), ptr(d_wc2), ptr(d_wa2), ptr(d_ba2), ptr(d_confc), stream()), "alpha_ksum_bwd_img")
    # the split image keeps 16 mantissa bits (1.5e-5 relative): per row 1e-4 x the row's max magnitude
    _grad_close(mlp_tc.image_to_dense(dz, rows, 256), rdz, "alpha_ksum_bwd_img dZ_3", rdz.abs().amax(1, keepdim=True))
    hd_mag = (Hj.double().abs().view(Nv, K, 256) * dX5[:, None, :256].double().abs()).sum(-1)
    sp = torch.nn.functional.softplus(rraw2.detach() - 1).view(Nv, K) * d_sigma.double()
    _grad_close(d_wc2, wcj.grad, "alpha_ksum_bwd_img d_wc", sp.abs() + hd_mag)
    _grad_close(d_wa2, waj.grad, "alpha_ksum_bwd_img d_walpha")
    _grad_close(d_ba2, baj.grad, "alpha_ksum_bwd_img d_balpha")
    # d conf_coefficient = d_wc * weight at the vlist samples' rows; every other row untouched
    rdc = torch.zeros(S, K, device="cuda", dtype=D)
    rdc[vl] = wcj.grad * weight[vl].double()
    _grad_close(d_confc[vl], rdc[vl], "alpha_ksum_bwd_img d_confc", (sp.abs() + hd_mag) * weight[vl].double())
    others = torch.ones(S, dtype=torch.bool, device="cuda")
    others[vl] = False
    if bool(others.any()):
        assert float(d_confc[others].abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------- image gather
def _down(x):
    return (x - 1) // 2 + 1


def _level_shapes(V, H, W):
    hs, ws = [H], [W]
    for _ in range(3):
        hs.append(_down(hs[-1]))
        ws.append(_down(ws[-1]))
    return [(V, h, w, c) for h, w, c in zip(hs, ws, (3, 6, 12, 24))]


def _misaligned(t):
    """the same values one float past the allocator's aligned base: the launchers' alignment check then takes the scalar kernel"""
    buf = torch.zeros(t.numel() + 4, device=t.device, dtype=t.dtype)
    v = buf[1:1 + t.numel()].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


def _gather_coords(g, V, S, H, W, vlist):
    """uniform in [-3, W+3] x [-3, H+3], plus exact integers, -0.999 (truncates to 0: valid), -1 (invalid), W - 2^-10, exactly W and
    H, and the zeroed (0,0) slot, each on a block of vlist samples"""
    xy = torch.stack([torch.rand(V, S, device="cuda", generator=g) * (W + 6) - 3, torch.rand(V, S, device="cuda", generator=g) * (H + 6) - 3], -1)
    Nv = vlist.shape[0]
    blk = max(1, Nv // 40)
    ix = lambda hi: torch.randint(0, hi, (V, blk), device="cuda", generator=g).float()
    specials = [(ix(W), ix(H)), (torch.full((V, blk), -0.999, device="cuda"), ix(H)), (ix(W), torch.full((V, blk), -0.999, device="cuda")),
                (torch.full((V, blk), -1.0, device="cuda"), ix(H)), (ix(W), torch.full((V, blk), -1.0, device="cuda")),
                (torch.full((V, blk), W - 2.0 ** -10, device="cuda"), ix(H)), (ix(W), torch.full((V, blk), H - 2.0 ** -10, device="cuda")),
                (torch.full((V, blk), float(W), device="cuda"), ix(H)), (ix(W), torch.full((V, blk), float(H), device="cuda")),
                (torch.rand(V, blk, device="cuda", generator=g), torch.rand(V, blk, device="cuda", generator=g))]
    for i, (x, y) in enumerate(specials):
        sl = vlist.long()[(i * blk) % Nv:(i * blk) % Nv + blk]
        xy[:, sl, 0], xy[:, sl, 1] = x[:, :sl.numel()], y[:, :sl.numel()]
    return xy.contiguous()


@pytest.mark.parametrize("ld", [45, 48])
@pytest.mark.parametrize("path", ["vector", "scalar"])
@pytest.mark.parametrize("V,H,W", [(8, 480, 640), (3, 37, 51), (2, 9, 7), (1, 1, 1)])
def test_image_gather_match_fp64(V, H, W, path, ld):
    """hnr_image_gather_fwd and hnr_image_gather_bwd_ld vs fp64 F.interpolate (bilinear, align_corners=False) + truncated lookup + the
    zeroed pixel, and its autograd.  8x480x640 is the benchmark (~80k samples x 8 views into a 60x80 level 3: heavy contention on the
    vector reductions); at 9x7 level 3 is 2x1, at 1x1 every level is 1x1 and every in-bounds pair reads the zeroed pixel.  The scalar
    kernels are forced by level (gradient) tensors one float off their aligned base; they take 45-wide forward rows only, so with
    ld 48 only their backward reads 48-wide rows"""
    g = _gen(V * H * W + (path == "scalar") + ld)
    Nv = 80000 if H == 480 else 3000
    S = Nv + Nv // 4
    shapes = _level_shapes(V, H, W)
    hw = [x for s in shapes for x in s[1:3]]
    lv = [torch.randn(s, device="cuda", generator=g) for s in shapes]
    vlist = torch.randperm(S, device="cuda", generator=g)[:Nv].to(torch.int32)
    xy = _gather_coords(g, V, S, H, W, vlist)
    fwd_ld = 45 if path == "scalar" else ld
    levels = lv if path == "vector" else [lv[0]] + [_misaligned(t) for t in lv[1:]]
    delta = torch.randn(V, S, 3, device="cuda", generator=g) if fwd_ld == 48 else None
    aux = torch.full((V, Nv, fwd_ld), float("nan"), device="cuda")
    ok = torch.full((V, Nv), float("nan"), device="cuda")
    check(lib().hnr_image_gather_fwd(ptr_array(levels), i64_array(hw), ptr(xy), ptr(vlist), V, S, Nv, ptr(aux), ptr(ok), fwd_ld, ptr(delta),
                                     stream()), "image_gather_fwd")
    lvd = [t.double().requires_grad_(True) for t in lv]
    raux, rok = ref_image_gather(lvd, xy.double(), vlist)
    assert torch.equal(ok, rok.float())                                       # validity flags: exact
    assert 0 < int(rok.sum()) < rok.numel() or H == 1
    if delta is not None:
        assert torch.equal(aux[..., 45:], delta[:, vlist.long()])              # copied through
    zeroed = ~rok | ((xy[:, vlist.long()].to(torch.int32) == 0).all(-1))
    assert float(aux[..., :45][zeroed].abs().max()) == 0.0                   # out of bounds and pixel (0,0): exactly 0
    # tap weights come from the fp32 source coordinate scale * (dst + 0.5) - 0.5.  Where every in/out size ratio is a power of two
    # (480x640, 1x1) it is exact and the only rounding is the 4-tap sum (atol 1e-6); otherwise it is off by up to ~2 ulp of a coordinate
    # < the level size, which moves the value by that times the spread of the taps: atol 1e-6 + 2^-22 x max level size x 2 max |level|
    exact = all((H // s[1]) * s[1] == H and (W // s[2]) * s[2] == W and (H // s[1]) & (H // s[1] - 1) == 0 and (W // s[2]) & (W // s[2] - 1) == 0
                for s in shapes[1:])
    atol = 1e-6 if exact else 1e-6 + 2.0 ** -22 * max(hw[2:]) * 2 * max(float(t.abs().max()) for t in lv[1:])
    _close(aux[..., :45], raux, 1e-5, atol, f"image_gather_fwd {path} {V}x{H}x{W}")
    # backward: level 0 and zeroed pairs receive nothing; columns 45..47 of 48-wide gradient rows are data and are never read
    d_aux = torch.randn(V, Nv, ld, device="cuda", generator=g)
    if ld == 48:
        d_aux[..., 45:] = float("nan")
    grads = [torch.zeros(s, device="cuda") for s in shapes]
    if path == "scalar":
        grads = [grads[0]] + [_misaligned(t) for t in grads[1:]]
    check(lib().hnr_image_gather_bwd_ld(ptr_array(grads), i64_array(hw), ptr(xy), ptr(vlist), ptr(d_aux), ld, V, S, Nv, stream()),
          "image_gather_bwd_ld")
    (raux * d_aux[..., :45].double()).sum().backward()
    assert float(grads[0].abs().max()) == 0.0
    for l in (1, 2, 3):
        _grad_close(grads[l], lvd[l].grad, f"image_gather_bwd {path} {V}x{H}x{W} level {l}")
    if ld == 45 and path == "vector":                                         # the 45-wide entry point is the same kernel
        g45 = [torch.zeros(s, device="cuda") for s in shapes]
        check(lib().hnr_image_gather_bwd(ptr_array(g45), i64_array(hw), ptr(xy), ptr(vlist), ptr(d_aux), V, S, Nv, stream()), "image_gather_bwd")
        for l in (1, 2, 3):
            _grad_close(g45[l], lvd[l].grad, f"image_gather_bwd (45) {V}x{H}x{W} level {l}")


# ---------------------------------------------------------------------------------------------------------- blend
@pytest.mark.parametrize("ld", [45, 48])
@pytest.mark.parametrize("keep", [False, True])
@pytest.mark.parametrize("V", [1, 2, 8])
def test_blend_match_fp64(V, keep, ld):
    """hnr_blend_fwd and hnr_blend_bwd(_ld) vs fp64 autograd of keep * num / (den + 1e-6): a sample whose views are all invalid
    (den = 1e-6: merged 0, d_sig 0), a sample whose blend weights are ~0 in every view (den ~1e-6: d_sig ~1e6), keep NULL and given,
    45- and 48-wide rows (padding columns of merged and d_aux exactly 0; columns 45..47 of aux are never read)"""
    g = _gen(100 * V + 10 * keep + ld)
    Nv = 3000
    aux = torch.randn(V, Nv, ld, device="cuda", generator=g)
    if ld == 48:
        aux[..., 45:] = float("nan")
    sig = torch.rand(V, Nv, device="cuda", generator=g) * 0.98 + 0.01
    ok = (torch.rand(V, Nv, device="cuda", generator=g) > 0.25).float()
    ok[:, 0] = 0.0
    sig[:, 1], ok[:, 1] = 1e-12, 1.0
    kp = (torch.rand(Nv, device="cuda", generator=g) > 0.3).to(torch.uint8) if keep else None
    if kp is not None:
        kp[:2] = 1
    merged = torch.full((Nv, ld), float("nan"), device="cuda")
    check(lib().hnr_blend_fwd(ptr(aux), ptr(sig), ptr(ok), ptr(kp), V, Nv, ld, ptr(merged), ld, stream()), "blend_fwd")
    ad, sd = aux[..., :45].double().requires_grad_(True), sig.double().requires_grad_(True)
    rm = ref_blend(ad, sd, ok.double(), kp)
    # V-term weighted sums of O(1) values over a sum of the weights: rtol 1e-5, atol 1e-6
    _close(merged[:, :45], rm, 1e-5, 1e-6, f"blend_fwd V={V}")
    assert float(merged[:, 45:].abs().max() if ld == 48 else 0.0) == 0.0    # padding: exactly 0
    assert float(merged[0].abs().max()) == 0.0                                # no valid view: num = 0 exactly
    if kp is not None:
        assert float(merged[kp == 0].abs().max()) == 0.0
    dm = torch.randn(Nv, 45, device="cuda", generator=g)
    (rm * dm.double()).sum().backward()
    d_aux = torch.full((V, Nv, ld), float("nan"), device="cuda")
    d_sig = torch.full((V * Nv,), float("nan"), device="cuda")
    if ld == 45:
        check(lib().hnr_blend_bwd(ptr(aux), ptr(sig), ptr(ok), ptr(kp), ptr(dm), V, Nv, ptr(d_aux), ptr(d_sig), stream()), "blend_bwd")
    else:
        check(lib().hnr_blend_bwd_ld(ptr(aux), ld, ptr(sig), ptr(ok), ptr(kp), ptr(dm), V, Nv, ptr(d_aux), ld, ptr(d_sig), stream()), "blend_bwd_ld")
    d_sig = d_sig.view(V, Nv)
    assert float(d_aux[..., 45:].abs().max() if ld == 48 else 0.0) == 0.0   # padding: exactly 0
    assert float(d_sig[ok == 0].abs().max()) == 0.0                           # invalid views: d_sig exactly 0
    assert float(d_aux[:, 0, :45].abs().max()) == 0.0
    # d_sig of sample 1 is ~1e6 x the others'.  d_aux: per sample 1e-4 x its max magnitude over views and channels.  d_sig =
    # ok / (den + 1e-6) x sum_c dm_c (aux_c - merged_c) cancels where one view dominates (aux - merged ~ 1e-6 aux for V = 1), in fp32 as
    # in any evaluation of this gradient: per element 1e-4 x the magnitude of those terms
    _grad_close(d_aux[..., :45], ad.grad, f"blend_bwd d_aux V={V}", ad.grad.abs().amax((0, 2))[None, :, None])
    rmd = rm.detach()
    if kp is not None:
        rmd = ref_blend(ad.detach(), sd.detach(), ok.double(), None)
    dmk = dm.double() * (kp.double()[:, None] if kp is not None else 1.0)
    terms = (dmk.abs()[None] * (ad.detach().abs() + rmd.abs()[None])).sum(-1) * ok.double() / ((sd.detach() * ok.double()).sum(0) + 1e-6)
    _grad_close(d_sig, sd.grad, f"blend_bwd d_sig V={V}", terms)


# ---------------------------------------------------------------------------------------------------------- pyramid
PYRAMID_CH = ((3, 6), (6, 6), (6, 12), (12, 12), (12, 24), (24, 24))


def _rows_per_block(V, Ho, Wo):
    """output rows per conv_bwd_weight block, as pyramid.cu's launch_bwd computes it"""
    strips = (Wo + 63) // 64
    return max(1, -(-(strips * Ho * V) // (4 * NUM_SMS)))


@pytest.mark.parametrize("ext", ["dlev", "null"])
@pytest.mark.parametrize("V,H,W", [(8, 480, 640), (1, 1, 1), (2, 5, 3), (3, 9, 130), (1, 2, 200)])
def test_pyramid_match_fp64(V, H, W, ext):
    """hnr_pyramid_fwd / hnr_pyramid_bwd vs fp64 conv2d: all six activations and all 12 weight / bias gradients, with the gradients
    of levels 1 and 2 given or NULL.  8x480x640 is the benchmark's shape and the only one whose weight-gradient blocks walk several
    output rows (rb > 1, bias sums carried across rows); Wo > 64 with a partial last strip (130, 200); levels of one pixel (1x1, 2x5)"""
    g = _gen(V * H * W + (ext == "null"))
    shapes = _level_shapes(V, H, W)
    outs = [shapes[1 + i // 2][1:3] for i in range(6)]
    rb = [_rows_per_block(V, ho, wo) for ho, wo in outs]
    assert (max(rb) > 1) == ((V, H, W) == (8, 480, 640)), rb
    ws = [torch.randn(co, ci, 3, 3, device="cuda", generator=g) * 0.3 for ci, co in PYRAMID_CH]
    bs = [torch.randn(co, device="cuda", generator=g) * 0.1 for _, co in PYRAMID_CH]
    img = torch.rand(V, H, W, 3, device="cuda", generator=g)
    act = [torch.full((V, ho, wo, co), float("nan"), device="cuda") for (ho, wo), (_, co) in zip(outs, PYRAMID_CH)]
    check(lib().hnr_pyramid_fwd(ptr(img), ptr_array(ws), ptr_array(bs), ptr_array(act), V, H, W, stream()), "pyramid_fwd")
    ref = ref_pyramid(img.double(), [w.double() for w in ws], [b.double() for b in bs])
    for i in range(6):
        r = ref[i].permute(0, 2, 3, 1)
        # fp32 sums of up to 9 x 24 products: rtol 1e-5, atol 2e-6 x the activation's max magnitude
        _close(act[i], r, 1e-5, 2e-6 * float(r.abs().max()), f"pyramid_fwd act{i} {V}x{H}x{W}")
    dlev = [torch.randn(s, device="cuda", generator=g) for s in shapes[1:]]
    dlev[0][:, ::3] = 0                                      # sparse, like the image gather's scatter
    dl = [dlev[0] if ext == "dlev" else None, dlev[1] if ext == "dlev" else None, dlev[2]]
    dws, dbs = [torch.zeros_like(w) for w in ws], [torch.zeros_like(b) for b in bs]
    scratch = [torch.empty_like(act[i]) for i in (4, 3, 2, 1, 0)]
    check(lib().hnr_pyramid_bwd(ptr(img), ptr_array(ws), ptr_array(act), ptr_array(dl), ptr_array(dws), ptr_array(dbs), ptr_array(scratch), V, H, W,
                                stream()), "pyramid_bwd")
    # fp64 adjoint, LeakyReLU' taken from the product's activation signs (a pre-activation within rounding of 0 may sit on either side)
    ins = [img.double().permute(0, 3, 1, 2)] + ref[:5]
    up = dl[2].double().permute(0, 3, 1, 2)
    for i in range(5, -1, -1):
        gz = up * torch.where(act[i].permute(0, 3, 1, 2) > 0, 1.0, 0.01).double()
        rdw = torch.nn.grad.conv2d_weight(ins[i], ws[i].shape, gz, stride=PYRAMID_STRIDES[i], padding=1)
        _grad_close(dws[i], rdw, f"pyramid_bwd dW{i} {V}x{H}x{W}")
        _grad_close(dbs[i], gz.sum((0, 2, 3)), f"pyramid_bwd db{i} {V}x{H}x{W}")
        if i:
            up = torch.nn.grad.conv2d_input(ins[i].shape, ws[i].double(), gz, stride=PYRAMID_STRIDES[i], padding=1)
            lvl = {3: dl[1], 1: dl[0]}.get(i - 1)
            if lvl is not None:
                up = up + lvl.double().permute(0, 3, 1, 2)
