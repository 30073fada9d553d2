"""GPU parity of the blur module (csrc/blur.cu, csrc/blur_learn.cu and their wrappers in ops.py / blur.py) against the fp64
oracle: the kernels alone over patch sizes 1..16 and kernel sizes 1..15 with planted winners, exact ties and 0/0 borders in the
pre-defined banks, every learnable norm / mode / boundary combination, and whole blur training steps (render -> fill_invalid ->
blur -> MSE -> backward into the point tables, the aggregator and the blur-kernel predictor)."""
import numpy as np
import pytest
import torch

from helpers import T, assert_close, blur_predictor, cuda, grad_atol
from oracle import render_oracle as ro

pytestmark = pytest.mark.gpu
RTOL_FWD, ATOL_FWD = 1e-5, 1e-6       # outputs
RTOL = 1e-4                           # gradients: rtol 1e-4 + grad_atol
NEAR_TIE = 1e-6                       # relative gap under which two candidates' fp64 errors count as tied to rounding

# (patch_num, patch_size, kernel_size, number of kernels): PS 1 / 3 / 5 leave lanes of the warp idle, PS 12 / 16 need 5 / 8 warps,
# KS 15 has more taps than a 96-thread block, KS 9 on 3x3 patches reaches past the patch from every pixel.  The 36-kernel rows use
# the shipped bank; 4x8 is BASELINE configs[3], 7x8 the shipped scripts' raster.
SELECT_CASES = [(1, 1, 1, 1), (2, 3, 9, 5), (3, 5, 3, 7), (4, 8, 9, 36), (7, 8, 9, 36), (2, 12, 15, 4), (2, 16, 15, 3)]
NAN_CASES = [c for c in SELECT_CASES if c[2] > 1]         # a corner tap needs a kernel wider than 1
LEARN_GEOMS = [(7, 8, 9), (4, 8, 9), (1, 1, 1), (2, 3, 9), (3, 5, 3), (2, 12, 15), (2, 16, 15)]
LEARN_COMBOS = [(norm, mode, bnd) for norm in (0, 1) for mode in (0, 4) for bnd in (0, 1, 2)]


def _gid(v):
    return "x".join(str(x) for x in v)


# ----------------------------------------------------------------------------------------------
# pre-defined kernels
# ----------------------------------------------------------------------------------------------
def _bank(rng, Nk, KS):
    if Nk == 36:
        from hybridneuralrendering_b200.blur import predefined_blur_kernels
        return predefined_blur_kernels(3)
    if KS == 1:
        return np.full((Nk, 1, 1), 0.5, np.float32)               # w p / w == p exactly: ties with the identity
    return rng.uniform(0.05, 1.0, (Nk, KS, KS)).astype(np.float32)


def _raster(rng, PN, PS):
    return rng.random(((PN * PS) ** 2, 3), dtype=np.float32)


def _plant(pred, gt, kernels, PN, PS, plan):
    """gt of patch p := the fp64 candidate plan[p] of pred (the blur with kernel j, or pred itself for j == Nk), rounded to fp32"""
    cand, _ = ro.blur_candidates(T(pred).double()[None], T(gt).double()[None], T(kernels).double()[None], PN, PS)
    g = gt.copy().reshape(PN, PS, PN, PS, 3)
    for p, j in plan.items():
        g[p // PN, :, p % PN, :, :] = cand[p, :, j].permute(1, 2, 0).numpy()
    return g.reshape(-1, 3)


def _check_selection(sel, err, msg):
    """the product's pick `sel` vs the fp64 argmin of `err` (P2,Nk+1): equal, except in at most one patch whose two candidates'
    fp64 errors differ, but by no more than NEAR_TIE relative (there either is right).  Errors that are exactly equal in fp64 come
    from candidates that are equal (a duplicated kernel, a delta and the identity) and so tie exactly in fp32 too: the lower index
    must win."""
    sel = sel.cpu().long()
    ref = torch.argmin(err, dim=1)
    off = torch.nonzero(sel != ref).flatten().tolist()
    for p in off:
        a, b = float(err[p, sel[p]]), float(err[p, ref[p]])
        assert np.isfinite(a) and np.isfinite(b) and a != b and abs(a - b) <= NEAR_TIE * max(abs(a), abs(b)), \
            f"{msg}: patch {p} picks {int(sel[p])} (err {a!r}), fp64 argmin {int(ref[p])} (err {b!r})"
    assert len(off) <= 1, f"{msg}: {len(off)} near-tied patches"
    return ref


def _run_select(pred, gt, kernels, PN, PS, rng, msg):
    """product blur_select (forward + backward under a random upstream gradient) vs the fp64 oracle with the product's pick.
    Returns (product pick, fp64 argmin) as CPU tensors."""
    from hybridneuralrendering_b200.blur import blur_select
    S2 = (PN * PS) ** 2
    G = rng.standard_normal((S2, 3)).astype(np.float32)
    pc = cuda(pred).clone().requires_grad_(True)
    out, sel = blur_select(pc[None], cuda(gt)[None], cuda(kernels)[None], PN, PS)
    assert sel.dtype == torch.int32 and sel.shape == (PN * PN,)
    (out[0] * cuda(G)).sum().backward()
    k64 = T(kernels).double()[None]
    p64 = T(pred).double().requires_grad_(True)
    _, err = ro.blur_candidates(p64.detach()[None], T(gt).double()[None], k64, PN, PS)
    ref_sel = _check_selection(sel, err, msg)
    ref, _ = ro.blur_select(p64[None], T(gt).double()[None], k64, PN, PS, select=sel.cpu())
    nan = torch.isnan(ref[0])
    assert torch.equal(torch.isnan(out[0]).cpu(), nan), f"{msg}: NaN positions"
    assert_close(out[0], ref[0], RTOL_FWD, ATOL_FWD, f"select out | {msg}")
    # backward on the patches whose selected error is finite (a 0/0 border makes the whole patch NaN on both sides)
    fin = torch.isfinite(err[torch.arange(PN * PN), sel.cpu().long()])
    if bool(fin.any()):
        (ref[0] * T(G).double()).sum().backward()
        pix = fin.reshape(PN, 1, PN, 1).expand(PN, PS, PN, PS).reshape(-1)
        r = p64.grad[pix]
        assert_close(pc.grad[pix.cuda()], r, RTOL, grad_atol(r), f"select d pred | {msg}")
    return sel.cpu().long(), ref_sel


@pytest.mark.parametrize("PN,PS,KS,Nk", SELECT_CASES, ids=[_gid(c) for c in SELECT_CASES])
def test_blur_select_planted_winners_vs_fp64(PN, PS, KS, Nk):
    """every candidate, the last kernel and the identity included, wins some patch: gt there is the fp64 candidate itself"""
    rng = np.random.default_rng(PN * 1000 + PS * 100 + KS)
    K = _bank(rng, Nk, KS)
    P2 = PN * PN
    order = list(range(Nk + 1))
    won = set()
    for r in range(0, Nk + 1, P2):                                 # as many rasters as it takes to plant every index once
        plan = dict(zip(rng.permutation(P2).tolist(), order[r:r + P2]))
        pred = _raster(rng, PN, PS)
        gt = _plant(pred, _raster(rng, PN, PS), K, PN, PS, plan)
        sel, ref_sel = _run_select(pred, gt, K, PN, PS, rng, f"{_gid((PN, PS, KS, Nk))} raster {r // P2}")
        won |= set(ref_sel.tolist())
        if KS > 1:
            for p, j in plan.items():
                assert int(sel[p]) == j, (p, j, int(sel[p]))
    if KS > 1:
        assert won == set(order)
    else:
        assert won == {0}                                          # a 1x1 kernel is the identity: the lower index wins every tie


@pytest.mark.parametrize("PN,PS,KS,Nk", SELECT_CASES, ids=[_gid(c) for c in SELECT_CASES])
def test_blur_select_exact_ties_pick_the_lower_index(PN, PS, KS, Nk):
    """a centred delta kernel ties exactly with the identity, a duplicated kernel with its copy: strict <, first minimum wins, on
    both sides"""
    rng = np.random.default_rng(PN * 1000 + PS * 100 + KS + 1)
    K = _bank(rng, Nk, KS)
    delta = np.zeros((KS, KS), np.float32)
    delta[KS // 2, KS // 2] = 1.0
    d = 1 if Nk >= 3 else 0
    K[d] = delta
    plan = {0: Nk}                                                 # gt == pred: delta and identity both have error 0
    expect = {0: d}
    if Nk >= 3:
        K[Nk - 1] = K[0]
        if PN * PN > 1:
            plan[1], expect[1] = 0, 0                              # kernel 0 and its copy at Nk - 1 tie
    pred = _raster(rng, PN, PS)
    gt = _plant(pred, _raster(rng, PN, PS), K, PN, PS, plan)
    sel, ref_sel = _run_select(pred, gt, K, PN, PS, rng, f"ties {_gid((PN, PS, KS, Nk))}")
    for p, j in expect.items():
        assert int(sel[p]) == j and int(ref_sel[p]) == j, (p, j, int(sel[p]), int(ref_sel[p]))


@pytest.mark.parametrize("PN,PS,KS,Nk", NAN_CASES, ids=[_gid(c) for c in NAN_CASES])
def test_blur_select_zero_mass_border_is_nan_and_wins(PN, PS, KS, Nk):
    """a single corner tap leaves border pixels with no in-bounds mass: 0/0 = NaN error, which wins (as torch.argmin) over every
    finite error, the first NaN kernel over a later one; NaN positions of the output match"""
    rng = np.random.default_rng(PN * 1000 + PS * 100 + KS + 2)
    K = _bank(rng, Nk, KS)
    s1 = 1 if Nk >= 2 else 0
    K[s1] = 0.0
    K[s1, 0, 0] = 1.0
    if Nk - 1 > s1:
        K[Nk - 1] = 0.0
        K[Nk - 1, -1, -1] = 1.0                                    # a second NaN kernel, later in the bank
    pred = _raster(rng, PN, PS)
    gt = _plant(pred, _raster(rng, PN, PS), K, PN, PS, {0: 0} if s1 else {})     # kernel 0 fits patch 0 exactly, yet loses
    sel, ref_sel = _run_select(pred, gt, K, PN, PS, rng, f"nan {_gid((PN, PS, KS, Nk))}")
    assert (sel == s1).all() and (ref_sel == s1).all()


# ----------------------------------------------------------------------------------------------
# learnable kernels
# ----------------------------------------------------------------------------------------------
def _raw(rng, N, KK, mode):
    """predictor outputs in (0, 1) as from the sigmoid; every other row has a quarter of its taps near 0; for mode 4 combine weights
    of exactly 0 and exactly 1"""
    raw = rng.uniform(0.05, 0.95, (N, KK + (mode == 4))).astype(np.float32)
    for r in range(0, N, 2):
        raw[r, rng.choice(KK, max(1, KK // 4), replace=False)] = rng.uniform(1e-7, 1e-5)
    if mode == 4 and N >= 3:
        raw[1, KK], raw[2, KK] = 0.0, 1.0
    return raw


@pytest.mark.parametrize("norm,mode,bnd", LEARN_COMBOS, ids=[f"n{n}m{m}b{b}" for n, m, b in LEARN_COMBOS])
@pytest.mark.parametrize("PN,PS,KS", LEARN_GEOMS, ids=[_gid(g) for g in LEARN_GEOMS])
def test_learnable_blur_kernel_vs_fp64(PN, PS, KS, norm, mode, bnd):
    """BlurLearnFn on raw predictor rows: output, d pred, d raw (taps and the combine weight) vs fp64 autograd of the oracle"""
    from hybridneuralrendering_b200 import ops
    rng = np.random.default_rng(PN * 10000 + PS * 1000 + KS * 10 + 100 * norm + 10 * mode + bnd)
    N, KK = PN * PN, KS * KS
    msg = f"{_gid((PN, PS, KS))} norm {norm} mode {mode} boundary {bnd}"
    pred, raw = _raster(rng, PN, PS), _raw(rng, N, KK, mode)
    G = rng.standard_normal(pred.shape).astype(np.float32)
    pc, rc = cuda(pred).requires_grad_(True), cuda(raw).requires_grad_(True)
    out = ops.BlurLearnFn.apply(pc, rc, PN, PS, KS, norm, mode, bnd)
    (out * cuda(G)).sum().backward()
    p64, r64 = T(pred).double().requires_grad_(True), T(raw).double().requires_grad_(True)
    ref = ro.learnable_blur_apply(p64[None], r64, PN, PS, KS, mode, norm, bnd)[0]
    (ref * T(G).double()).sum().backward()
    assert_close(out, ref, RTOL_FWD, ATOL_FWD, f"learn out | {msg}")
    assert_close(pc.grad, p64.grad, RTOL, grad_atol(p64.grad), f"learn d pred | {msg}")
    assert_close(rc.grad, r64.grad, RTOL, grad_atol(r64.grad), f"learn d raw | {msg}")
    if mode == 4:
        wc = r64.grad[:, KK]
        assert KS == 1 or float(wc.abs().max()) > 0                # a 1x1 kernel is the identity whatever the combine weight
        assert_close(rc.grad[:, KK], wc, RTOL, grad_atol(wc), f"learn d combine weight | {msg}")


def _predictor_ref(params, pred, gt, PN, PS, KS, mode, norm, bnd, G):
    """fp64 learnable_blur with leaf copies of the predictor weights; also the smallest |pre-activation| of its LeakyReLUs"""
    W64 = [(W.double().requires_grad_(True), b.double().requires_grad_(True)) for W, b in params]
    p64 = T(pred).double().requires_grad_(True)
    ro.KINK_TAP = []
    try:
        ref, raw = ro.learnable_blur(p64[None], T(gt).double()[None], W64, PN, PS, KS, mode, norm, bnd)
        kink = min(float(t.min()) for t in ro.KINK_TAP)
    finally:
        ro.KINK_TAP = None
    (ref[0] * T(G).double()).sum().backward()
    return ref[0], raw, p64.grad, W64, kink


@pytest.mark.parametrize("norm,mode,bnd", LEARN_COMBOS, ids=[f"n{n}m{m}b{b}" for n, m, b in LEARN_COMBOS])
@pytest.mark.parametrize("PN,PS,KS", LEARN_GEOMS, ids=[_gid(g) for g in LEARN_GEOMS])
def test_learnable_blur_with_predictor_vs_fp64(PN, PS, KS, norm, mode, bnd):
    """learnable_blur end to end: gray features -> predictor MLP (the dense-layer kernels at M = PN^2 rows, K = 2 PS^2) -> kernel
    -> blur, and back: output, raw, d pred (both paths: the blur and the predictor input) and the 8 predictor gradients"""
    from hybridneuralrendering_b200.blur import learnable_blur
    rng = np.random.default_rng(PN * 10000 + PS * 1000 + KS * 10 + 100 * norm + 10 * mode + bnd + 7)
    msg = f"{_gid((PN, PS, KS))} norm {norm} mode {mode} boundary {bnd}"
    pred, gt = _raster(rng, PN, PS), _raster(rng, PN, PS)
    G = rng.standard_normal(pred.shape).astype(np.float32)
    # predictor weights whose hidden units all stay >= 1e-5 from the LeakyReLU kink on these inputs (LeakyReLU' jumps there, so
    # fp32 and fp64 may take different slopes)
    for seed in range(20):
        params = ro.blur_predictor_params(1000 * PN + 100 * PS + KS + 17 * seed, PS, KS, mode)
        ref, raw_ref, gp_ref, W64, kink = _predictor_ref(params, pred, gt, PN, PS, KS, mode, norm, bnd, G)
        if kink > 1e-5:
            break
    assert kink > 1e-5
    blk = blur_predictor(params)
    pc = cuda(pred).requires_grad_(True)
    out, raw = learnable_blur(pc[None], cuda(gt)[None], blk, PN, PS, KS, mode, norm, bnd)
    (out[0] * cuda(G)).sum().backward()
    assert_close(raw, raw_ref, RTOL_FWD, ATOL_FWD, f"predictor raw | {msg}")
    assert_close(out[0], ref, RTOL_FWD, ATOL_FWD, f"learn out | {msg}")
    assert_close(pc.grad, gp_ref, RTOL, grad_atol(gp_ref), f"learn+predictor d pred | {msg}")
    for li, (W, b) in enumerate(W64):
        lin = blk[2 * li]
        assert_close(lin.weight.grad, W.grad, RTOL, grad_atol(W.grad), f"predictor dW{li} | {msg}")
        assert_close(lin.bias.grad, b.grad, RTOL, grad_atol(b.grad), f"predictor db{li} | {msg}")


# ----------------------------------------------------------------------------------------------
# whole blur training steps (benchmarks.blur_train_step_benchmark at BASELINE configs[3]'s raster, on a small scene)
# ----------------------------------------------------------------------------------------------
def _blur_training_step_vs_oracle(learnable: bool, seed: int):
    """forward -> fill_invalid -> blur -> MSE against gt_image -> backward, compared with the same step on the fp64 oracle (the
    product's query positions, projections and blur pick).  Rays with a hidden unit within 1e-5 of a LeakyReLU kink keep their
    colour but pass no gradient, on both sides (the blur mixes neighbouring pixels, so they cannot be masked out of the loss)."""
    from test_gpu_e2e import _build, _check_projections, _frame_cuda, _product_projections
    from hybridneuralrendering_b200 import make_opt
    from hybridneuralrendering_b200 import synthetic as syn
    from hybridneuralrendering_b200.blur import blur_select, learnable_blur, predefined_blur_kernels
    from hybridneuralrendering_b200.neural_points_volumetric_model import fill_invalid
    from oracle import pipeline_oracle as po
    PN, PS, KS = 4, 8, 9
    opt = make_opt("scannet", use_nearest=2, SR=24, is_train=True, drop_ratio=0.5, dilation_setup="4_8_1_8",
                   learnable_blur_kernel=int(learnable), boundary_mode=1)
    xyz = syn.room_scene(30000, seed)
    att = syn.point_attributes(np.random.default_rng(seed), len(xyz))
    fr = syn.room_frame(H=480, W=640, V=2, patch_num=PN, patch_size=PS, seed=seed)
    P = ro.random_params(seed)
    net = _build(opt, xyz, att, P)
    blk = net.aggregator.learn_blur_kernel_block
    if learnable:
        with torch.no_grad():                                      # taps far from uniform
            for li, (W, b) in enumerate(ro.blur_predictor_params(seed, PS, KS, 4)):
                blk[2 * li].weight.copy_(W)
                blk[2 * li].bias.copy_(b)
    R = fr["raydir"].shape[1]
    assert R == (PN * PS) ** 2
    torch.manual_seed(seed)
    st = torch.cuda.get_rng_state()
    ts = net.neural_points.querier.candidate_ts(R, 0.1, 8.0, "cuda")       # the jittered draw the forward will repeat
    torch.cuda.set_rng_state(st)
    out = net(**_frame_cuda(fr))

    # fp64 oracle of the render on the product's query and projections
    pts = dict(xyz=xyz, **att)
    mask = out["ray_mask"][0] > 0
    q = po.query(pts, fr, opt, ts.cpu().numpy().reshape(R, -1))
    np.testing.assert_array_equal(out["ray_mask"].cpu().numpy(), q["ray_mask"])
    xy, delta = _product_projections(net, fr, q["sample_loc_w"])
    cfg = ro.AggCfg(use_nearest=2, is_train=True, drop_ratio=0.5, dilation_setup="4_8_1_8")
    ref = po.render(P, cfg, pts, fr, opt, None, dtype=torch.float64, params_grad=True, q=q, xy_override=xy.cpu(), kink_eps=1e-5)
    _check_projections(xy, delta, ref)
    assert int(mask.sum()) == ref["ray_color"].shape[1] > 200
    keep = ref["kink_free"].to(torch.float64)[None, :, None]
    assert float(keep.mean()) > 0.5

    # product: kinked rays detached, scattered to the raster, blurred, MSE
    kp = keep.float().cuda()
    c = out["coarse_raycolor"]
    full = fill_invalid(dict(out, coarse_raycolor=kp * c + (1 - kp) * c.detach()), cuda(fr["bg_color"]), net.last_extras.ray_ids)
    gt = cuda(fr["gt_image"])
    K = predefined_blur_kernels(3)
    if learnable:
        blurred, _ = learnable_blur(full["coarse_raycolor"], gt, out["blur_predictor"], PN, PS, KS, 4, 0, 1)
    else:
        blurred, sel = blur_select(full["coarse_raycolor"], gt, cuda(K)[None], PN, PS)
    loss = torch.nn.functional.mse_loss(blurred, gt)
    loss.backward()

    # oracle: the same, in fp64
    c64 = ref["ray_color"]
    c64 = keep * c64 + (1 - keep) * c64.detach()
    full64 = T(fr["bg_color"]).double().reshape(1, 1, 3).expand(1, R, 3).index_copy(1, torch.nonzero(mask.cpu()).flatten(), c64)
    gt64 = T(fr["gt_image"]).double()
    if learnable:
        W64 = [(blk[2 * li].weight.detach().cpu().double().requires_grad_(True), blk[2 * li].bias.detach().cpu().double().requires_grad_(True))
               for li in range(4)]
        ro.KINK_TAP = []
        try:
            blurred64, _ = ro.learnable_blur(full64, gt64, W64, PN, PS, KS, 4, 0, 1)
            assert min(float(t.min()) for t in ro.KINK_TAP) > 1e-5    # no predictor unit on its kink
        finally:
            ro.KINK_TAP = None
    else:
        K64 = T(K).double()[None]
        _, err = ro.blur_candidates(full64.detach(), gt64, K64, PN, PS)
        _check_selection(sel, err, "training step")
        assert len(set(sel.tolist())) > 1
        blurred64, _ = ro.blur_select(full64, gt64, K64, PN, PS, select=sel.cpu())
    assert_close(blurred, blurred64, RTOL_FWD, ATOL_FWD, "training blurred raster")
    rloss = torch.nn.functional.mse_loss(blurred64, gt64)
    rloss.backward()
    assert_close(loss, rloss, RTOL, 1e-7, "training loss")

    npts = net.neural_points
    for name, leaf in (("points_embeding", "emb"), ("points_conf", "conf"), ("points_color", "color"), ("points_dir", "dir")):
        g, r = getattr(npts, name).grad[0], ref["leaf"][leaf].grad
        assert int((r.abs().sum(-1) > 0).sum()) > 50
        assert_close(g, r, RTOL, grad_atol(r), f"training {name}")
    n = 0
    for k, p in net.aggregator.named_parameters():
        r = ref["params"][k].grad if k in ref["params"] else None
        if r is None or float(r.abs().max()) == 0:
            continue
        assert_close(p.grad, r, RTOL, grad_atol(r), f"training {k}")
        n += 1
    assert n >= 40
    if learnable:
        for li, (W, b) in enumerate(W64):
            assert_close(blk[2 * li].weight.grad, W.grad, RTOL, grad_atol(W.grad), f"training predictor dW{li}")
            assert_close(blk[2 * li].bias.grad, b.grad, RTOL, grad_atol(b.grad), f"training predictor db{li}")


def test_blur_select_training_step_matches_oracle():
    """the 36-kernel bank, as train_blur"""
    _blur_training_step_vs_oracle(False, 21)


def test_learnable_blur_training_step_matches_oracle():
    """mode 4, norm 0, boundary 1, as train_blur_learnable"""
    _blur_training_step_vs_oracle(True, 22)
