"""Pin the CPU oracle against outputs of the unmodified reference (tests/golden/*.npz, made by
tests/golden/make_golden.py in the build container).  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import render_oracle as ro
from hybridneuralrendering_b200 import synthetic as syn
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

T = torch.from_numpy


def _load(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))


def _agg_inputs(meta, empty_frac=0.4):
    R, SR, V, H, W, is_train, seed = [int(x) for x in meta]
    d = syn.render_stage_inputs(seed=seed, N=600, R=R, SR=SR, K=8, V=V, H=H, W=W, empty_frac=empty_frac)
    return d, syn.gather_neighbours(d), (R, SR, V, H, W, bool(is_train), seed)


def _run_oracle(d, g, P, cfg, dtype=torch.float32, grad=False):
    c = lambda a: T(a).to(dtype)
    leaf = {k: c(g[k]).clone().requires_grad_(grad) for k in ("sampled_embedding", "sampled_color", "sampled_dir", "sampled_conf")}
    Pd = {k: v.to(dtype).clone().requires_grad_(grad) for k, v in P.items()}
    out = ro.aggregate(Pd, cfg, leaf["sampled_color"], torch.eye(3, dtype=dtype), leaf["sampled_dir"], leaf["sampled_conf"],
                       leaf["sampled_embedding"], c(g["sampled_xyz_pers"]), c(g["sampled_xyz"]), T(g["sample_pnt_mask"]),
                       c(d["sample_loc"]), c(d["sample_loc_w"]), c(d["sample_ray_dirs"]), img_n=c(d["images_nearest"]),
                       sample_loc_i_n=c(d["sample_loc_i_n"]), delta_viewdir_n=c(d["delta_viewdir_n"]))
    return out, leaf, Pd


def test_agg_eval_matches_reference():
    G = _load("agg_eval")
    d, g, (R, SR, V, H, W, is_train, seed) = _agg_inputs(G["meta"])
    P = ro.random_params(seed=seed + 100)
    cfg = ro.AggCfg(use_nearest=V, is_train=False)
    (decoded, valid, w, cc), _, _ = _run_oracle(d, g, P, cfg)
    assert np.array_equal(valid.numpy(), G["ray_valid"])
    np.testing.assert_allclose(decoded.numpy(), G["decoded"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(w.numpy(), G["weight"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(cc.numpy(), G["conf_coefficient"], rtol=0, atol=0)
    rd = ro.ray_dist_from_depth(T(d["sample_loc"])[..., 2], valid, float(d["vsize"][2]))
    np.testing.assert_array_equal(rd.numpy(), G["ray_dist"])
    o = ro.ray_march(rd, valid, decoded, torch.ones(1, 3))
    np.testing.assert_allclose(o[0].numpy(), G["ray_color"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(o[2].numpy(), G["opacity"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(o[3].numpy(), G["acc_transmission"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(o[4].numpy(), G["blend_weight"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(o[5].numpy(), G["bg_transmission"], rtol=1e-5, atol=1e-7)


def test_agg_train_grads_match_reference():
    G = _load("agg_train")
    d, g, (R, SR, V, H, W, is_train, seed) = _agg_inputs(G["meta"])
    assert is_train
    P = ro.random_params(seed=seed + 100)
    cfg = ro.AggCfg(use_nearest=V, is_train=True, drop_ratio=float(G["drop_ratio"]), dilation_setup=str(G["dilation_setup"]))
    (decoded, valid, w, cc), leaf, Pd = _run_oracle(d, g, P, cfg, grad=True)
    np.testing.assert_allclose(decoded.detach().numpy(), G["decoded"], rtol=1e-5, atol=1e-6)
    rd = ro.ray_dist_from_depth(T(d["sample_loc"])[..., 2], valid, float(d["vsize"][2]))
    color = ro.ray_march(rd, valid, decoded, torch.ones(1, 3))[0]
    v = cc.clamp(1e-3, 1 - 1e-3)
    loss = torch.nn.functional.mse_loss(color, T(G["gt"])) + 1e-4 * torch.mean(torch.log(v) + torch.log(1 - v))
    np.testing.assert_allclose(loss.item(), float(G["loss"]), rtol=1e-5)
    loss.backward()
    for k, t in leaf.items():
        ref = G["grad_" + k]
        np.testing.assert_allclose(t.grad.numpy(), ref, rtol=2e-4, atol=1e-7 + 1e-4 * np.abs(ref).max(), err_msg=k)
    n = 0
    for k, p in Pd.items():
        key = "gradP_" + k
        if key not in G:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        ref = G[key]
        np.testing.assert_allclose(p.grad.numpy(), ref, rtol=2e-4, atol=1e-7 + 2e-4 * np.abs(ref).max(), err_msg=k)
        n += 1
    assert n >= 40


def test_posenc_raygen_raymarch_match_reference():
    G = _load("misc")
    x = T(G["pe_x"])
    np.testing.assert_array_equal(ro.pos_enc(x, 3).numpy(), G["pe_pe3"])
    np.testing.assert_array_equal(ro.pos_enc(x[:, :3], 4, ori=True).numpy(), G["pe_pe4_ori"])
    from oracle import query_oracle as qo
    rp0, ts0 = qo.ray_candidates(G["gen_campos"], G["gen_raydir"], 40, 0.1, 8.0, None)
    np.testing.assert_array_equal(ts0, G["gen_ts0"])
    np.testing.assert_array_equal(rp0, G["gen_raypos0"])
    rp1, ts1 = qo.ray_candidates(G["gen_campos"], G["gen_raydir"], 40, 2.0, 6.0, G["gen_noise"], jitter=0.3)
    np.testing.assert_array_equal(ts1, G["gen_ts1"])
    np.testing.assert_array_equal(rp1, G["gen_raypos1"])
    f = T(G["rm_feats"]).clone().requires_grad_(True)
    o = ro.ray_march(T(G["rm_dist"]), T(G["rm_valid"]), f, T(G["rm_bg"]))
    np.testing.assert_allclose(o[0].detach().numpy(), G["rm_ray_color"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(o[5].detach().numpy(), G["rm_bgT"], rtol=1e-6, atol=1e-12)
    (o[0] * T(G["rm_G"])).sum().backward()
    np.testing.assert_allclose(f.grad.numpy(), G["rm_grad_feats"], rtol=1e-5, atol=1e-7)


def test_projection_matches_reference():
    G = _load("proj")
    xy = ro.project_to_views(T(G["loc_w"])[0], T(G["intrinsic"]), T(G["c2w_n"]))
    np.testing.assert_allclose(xy.numpy(), G["xy"], rtol=1e-6, atol=1e-4)
    dv = ro.delta_viewdirs(T(G["loc_w"])[0], T(G["campos"])[0], T(G["campos_n"]))
    np.testing.assert_allclose(dv.numpy(), G["delta_view"], rtol=1e-6, atol=1e-7)


def test_blur_matches_reference():
    G = _load("blur")
    PN, PS, Nk = [int(v) for v in G["meta"]]
    pred = T(G["pred"]).clone().requires_grad_(True)
    out, sel = ro.blur_select(pred, T(G["gt"]), T(G["kernels"]), PN, PS)
    np.testing.assert_allclose(out.detach().numpy(), G["out"], rtol=1e-6, atol=1e-7)
    (out * T(G["G"])).sum().backward()
    np.testing.assert_allclose(pred.grad.numpy(), G["grad_pred"], rtol=1e-5, atol=1e-7)
    assert len(set(sel.tolist())) > 1, "fixture should exercise more than one candidate"


def test_learnable_blur_matches_reference():
    """N3: oracle restatement of learnable_blur_update_output vs the unmodified reference, all option branches of the fixture
    (outputs, gradient w.r.t. the rendered colours and every predictor weight)."""
    G = _load("blur_learn")
    PN, PS, KS = [int(v) for v in G["meta"]]
    for ci, (mode, norm, bmode) in enumerate(G["cases"].tolist()):
        W = [(w.clone().requires_grad_(True), b.clone().requires_grad_(True)) for w, b in ro.blur_predictor_params(100 + ci, PS, KS, mode)]
        pred = T(G["pred"]).clone().requires_grad_(True)
        out, raw = ro.learnable_blur(pred, T(G["gt"]), W, PN, PS, KS, mode, norm, bmode)
        np.testing.assert_allclose(out.detach().numpy(), G[f"c{ci}_out"], rtol=1e-5, atol=1e-6)
        (out * T(G["G"])).sum().backward()
        ref = G[f"c{ci}_grad_pred"]
        np.testing.assert_allclose(pred.grad.numpy(), ref, rtol=1e-4, atol=1e-5 * np.abs(ref).max())
        for li, (w, b) in enumerate(W):
            for got, key in ((w.grad, f"c{ci}_gW{li}"), (b.grad, f"c{ci}_gb{li}")):
                np.testing.assert_allclose(got.numpy(), G[key], rtol=1e-4, atol=1e-4 * np.abs(G[key]).max() + 1e-12)
        assert raw.std() > 0.05, "fixture should predict non-uniform kernels"


def _frame_oracle_item(name, split, idx, over, seed, bg):
    import random
    from oracle import frame_oracle as fo
    images, c2w, vids, K, train_ids, test_ids = syn.frame_scene()
    random.seed(seed)
    np.random.seed(seed)
    it = fo.frame_item(images, c2w, vids, K, train_ids if split == "train" else test_ids, train_ids, idx, split=split, bg_color=bg,
                       total_num_image=vids[-1] + 1, **over)
    return it, np.array([random.random(), np.random.rand()])


def test_frame_producer_matches_reference():
    """N4: oracle restatement of ScannetFtDataset.__getitem__ vs the unmodified method (tests/golden/frame.npz): chosen views,
    pixel grid, ground-truth lookup and camera entries exact; ray directions to 1 ulp-ish (BLAS vs numpy summation order);
    both RNG streams end in the same state."""
    from frame_cases import FRAME_CASES, FRAME_CASES_CPU
    G = _load("frame")
    for name, split, idx, over, seed, bg in FRAME_CASES + FRAME_CASES_CPU:
        it, after = _frame_oracle_item(name, split, idx, over, seed, bg)
        assert np.float32(np.abs(it["images_nearest"]).max()) == G[f"{name}_images_nearest_absmax"]
        assert it["vid_nearest"].tolist() == G[f"{name}_vid_nearest"].tolist(), name
        assert [it["vid"], it["h"], it["w"]] == G[f"{name}_meta"][:3].tolist()
        for k in ("pixel_idx", "gt_image", "c2w_nearest", "campos_nearest", "camrotc2w_nearest", "c2w", "campos", "camrotc2w", "bg_color"):
            np.testing.assert_array_equal(np.asarray(it[k], np.float32), G[f"{name}_{k}"].astype(np.float32), err_msg=f"{name}:{k}")
        np.testing.assert_allclose(it["raydir"], G[f"{name}_raydir"], rtol=0, atol=3e-7, err_msg=name)
        np.testing.assert_allclose(it["vid_angle_nearest"], G[f"{name}_vid_angle_nearest"], rtol=1e-12)
        np.testing.assert_allclose(it["middle"], G[f"{name}_middle"].reshape(()), rtol=1e-6)
        np.testing.assert_array_equal(after, G[f"{name}_after"])


# ---------------------------------------------------------------------------------------------------------------------
# shipped shapes (SR 80 / V 4 eval; SR 24 / V 8 / dilation_setup 7_8_1_8 / drop 0.5 training with the out-of-range drop quirk):
# outputs of the unmodified reference with the POINT TABLES as differentiable leaves (make_golden.agg_case_tables)
# ---------------------------------------------------------------------------------------------------------------------
def _tables_case(G):
    R, SR, V, H, W, is_train, seed, N = [int(x) for x in G["meta"]]
    d = syn.render_stage_inputs(seed=seed, N=N, R=R, SR=SR, K=8, V=V, H=H, W=W, empty_frac=float(G["empty_frac"]))
    return d, syn.gather_neighbours(d), (R, SR, V, H, W, bool(is_train), seed)


def _run_oracle_tables(d, g, P, cfg, grad):
    tab = {k: T(d[k]).clone().requires_grad_(grad) for k in ("emb", "color", "dir", "conf")}
    idx = T(np.maximum(d["sample_pidx"], 0)).long()
    Pd = {k: v.clone().requires_grad_(grad) for k, v in P.items()}
    out = ro.aggregate(Pd, cfg, tab["color"][idx], torch.eye(3), tab["dir"][idx], tab["conf"][idx], tab["emb"][idx], T(g["sampled_xyz_pers"]),
                       T(g["sampled_xyz"]), T(g["sample_pnt_mask"]), T(d["sample_loc"]), T(d["sample_loc_w"]), T(d["sample_ray_dirs"]),
                       img_n=T(d["images_nearest"]), sample_loc_i_n=T(d["sample_loc_i_n"]), delta_viewdir_n=T(d["delta_viewdir_n"]))
    return out, tab, Pd


def test_agg_eval_shipped_shape_matches_reference():
    G = _load("agg_eval_sr80")
    d, g, (R, SR, V, H, W, is_train, seed) = _tables_case(G)
    assert (SR, V) == (80, 4) and int(G["ray_valid"].sum()) >= 2000
    cfg = ro.AggCfg(use_nearest=V, is_train=False)
    with torch.no_grad():
        (decoded, valid, w, cc), _, _ = _run_oracle_tables(d, g, ro.random_params(seed=seed + 100), cfg, False)
    assert np.array_equal(valid.numpy(), G["ray_valid"])
    np.testing.assert_allclose(decoded.numpy(), G["decoded"], rtol=1e-5, atol=1e-6)
    rd = ro.ray_dist_from_depth(T(d["sample_loc"])[..., 2], valid, float(d["vsize"][2]))
    o = ro.ray_march(rd, valid, decoded, torch.ones(1, 3))
    np.testing.assert_allclose(o[0].numpy(), G["ray_color"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(o[2].numpy(), G["opacity"], rtol=1e-5, atol=1e-7)


def test_agg_train_shipped_shape_grads_match_reference():
    G = _load("agg_train_sr24")
    d, g, (R, SR, V, H, W, is_train, seed) = _tables_case(G)
    assert (SR, V, str(G["dilation_setup"])) == (24, 8, "7_8_1_8") and int(G["ray_valid"].sum()) >= 2000
    cfg = ro.AggCfg(use_nearest=V, is_train=True, drop_ratio=float(G["drop_ratio"]), dilation_setup=str(G["dilation_setup"]))
    torch.set_num_threads(8)
    (decoded, valid, w, cc), tab, Pd = _run_oracle_tables(d, g, ro.random_params(seed=seed + 100), cfg, True)
    np.testing.assert_allclose(decoded.detach().numpy(), G["decoded"], rtol=1e-5, atol=1e-6)
    rd = ro.ray_dist_from_depth(T(d["sample_loc"])[..., 2], valid, float(d["vsize"][2]))
    color = ro.ray_march(rd, valid, decoded, torch.ones(1, 3))[0]
    v = cc.clamp(1e-3, 1 - 1e-3)
    # rays with a hidden unit on a LeakyReLU kink (|pre-activation| < 1e-5 in the reference's forward) are masked out of the colour
    # loss: their slopes may legitimately differ between fp32 implementations (make_golden._fragile_rays)
    keep = T(G["keep"])
    loss = torch.nn.functional.mse_loss(color * keep, T(G["gt"]) * keep) + 1e-4 * torch.mean(torch.log(v) + torch.log(1 - v))
    np.testing.assert_allclose(loss.item(), float(G["loss"]), rtol=1e-5)
    loss.backward()
    for k, t in tab.items():
        ref = G["gradT_" + k]
        np.testing.assert_allclose(t.grad.numpy(), ref, rtol=2e-4, atol=1e-7 + 1e-4 * np.abs(ref).max(), err_msg=k)
    n = 0
    for k, p in Pd.items():
        key = "gradP_" + k
        if key not in G:
            continue
        ref = G[key]
        np.testing.assert_allclose(p.grad.numpy(), ref, rtol=2e-4, atol=1e-7 + 1e-4 * np.abs(ref).max(), err_msg=k)
        n += 1
    assert n >= 40


def test_kernel_references_match_oracle(monkeypatch):
    """the fp64 references of the per-kernel GPU tests (tests/helpers.py ref_*) against the oracle's own expressions on one small case:
    pos_enc, feature_pyramid, full_res_features + the truncated pixel lookup, and the weight, MLP-input, density-head / K-sum and blend
    expressions inside aggregate(), read off the inputs and outputs of its dense layers.  The oracle is pinned to the reference's
    goldens above, so this ties the yardstick of tests/test_gpu_aggregate_kernels.py to them too."""
    import helpers as h
    dt = torch.float64
    R, SR, K, V = 7, 6, 8, 2
    S = R * SR
    d = syn.render_stage_inputs(seed=5, N=300, R=R, SR=SR, K=K, V=V, H=19, W=27, empty_frac=0.3)
    g = syn.gather_neighbours(d)
    P = ro.random_params(seed=6, dtype=dt)
    c = lambda a: T(a).to(dt)
    a, b = 0.7, -0.4                                         # a world->camera rotation that is not the identity
    rz = torch.tensor([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], dtype=dt)
    rx = torch.tensor([[1, 0, 0], [0, np.cos(b), -np.sin(b)], [0, np.sin(b), np.cos(b)]], dtype=dt)
    rw2c = rz @ rx
    taps, lin = {}, ro._lin

    def tap(x, P_, name):
        y = lin(x, P_, name)
        taps.setdefault(name, []).append((x, y))
        return y
    monkeypatch.setattr(ro, "_lin", tap)
    out, valid, w, cc = ro.aggregate(P, ro.AggCfg(use_nearest=V), c(g["sampled_color"]), rw2c, c(g["sampled_dir"]), c(g["sampled_conf"]),
                                     c(g["sampled_embedding"]), c(g["sampled_xyz_pers"]), c(g["sampled_xyz"]), T(g["sample_pnt_mask"]),
                                     c(d["sample_loc"]), c(d["sample_loc_w"]), c(d["sample_ray_dirs"]), img_n=c(d["images_nearest"]),
                                     sample_loc_i_n=c(d["sample_loc_i_n"]), delta_viewdir_n=c(d["delta_viewdir_n"]))
    monkeypatch.undo()
    close = lambda x, y, atol=1e-12: np.testing.assert_allclose(x.detach().numpy(), y.detach().numpy(), rtol=1e-10, atol=atol)
    pidx = T(d["sample_pidx"]).reshape(S, K)
    loc_w, loc_pers, rays = c(d["sample_loc_w"]).reshape(S, 3), c(d["sample_loc"]).reshape(S, 3), c(d["sample_ray_dirs"]).reshape(S, 3)
    cam = torch.cat([c(d["campos"]).reshape(3), c(d["camrotc2w"]).reshape(9), rw2c.t().reshape(9)])
    # weights, clamped confidence, validity
    rw, rc, rv = h.ref_nbr_weights(c(d["xyz"]), c(d["conf"]), pidx, None, loc_w)
    assert torch.equal(rv, valid.reshape(-1)) and 0 < int(rv.sum()) < S
    close(rw, w.reshape(S, K))
    close(rc, cc.reshape(S, K), atol=1e-11)                  # the oracle clamps at 1e-4, the kernel (and ref) at float32(1e-4)
    # MLP input rows of the live slots of the valid samples (the oracle's rows, in its order)
    vlist = rv.nonzero()[:, 0].to(torch.int32)
    live = pidx[vlist.long()].reshape(-1) >= 0
    X0, E = h.ref_nbr_features(c(d["xyz"]), c(d["xyz_pers"]), c(d["emb"]), c(d["color"]), c(d["dir"]), pidx, vlist, loc_w, loc_pers, rays, cam)
    close(X0[live], taps["block1.0"][0][0])
    close(E[live], taps["block3.0"][0][0][:, 256:])
    # without the table the perspective coordinates come from cam: equal up to the table's fp32 rounding (x 2^4 in the encoding)
    X0c, _ = h.ref_nbr_features(c(d["xyz"]), None, c(d["emb"]), c(d["color"]), c(d["dir"]), pidx, vlist, loc_w, loc_pers, rays, cam)
    close(X0c, X0, atol=1e-5)
    # density head + weighted K-sum from the oracle's layer-3 outputs (zero rows for masked slots)
    H = torch.zeros(len(live), 256, dtype=dt)
    H[live] = torch.nn.functional.leaky_relu(taps["block3.2"][0][1], 0.01)
    s = vlist.long()
    sigma, X5, _ = h.ref_alpha_ksum(H, (rw * rc)[s], P["alpha_branch.0.weight"], P["alpha_branch.0.bias"], rays[s] @ cam[12:21].reshape(3, 3))
    close(X5, taps["color_feature_branch.0"][0][0])
    close(sigma, out.reshape(S, 4)[s, 0])
    # pyramid, upsample + truncated lookup, blend
    img = c(d["images_nearest"])[0]
    ws = [P[f"aux_block_s{i}.{j}.weight"] for i in (1, 2, 3) for j in (0, 2)]
    bs = [P[f"aux_block_s{i}.{j}.bias"] for i in (1, 2, 3) for j in (0, 2)]
    acts = h.ref_pyramid(img, ws, bs)
    lv = ro.feature_pyramid(img, P)
    for i in (1, 2, 3):
        close(acts[2 * i - 1], lv[i])
    aux, ok = h.ref_image_gather([img] + [acts[i].permute(0, 2, 3, 1) for i in (1, 3, 5)], c(d["sample_loc_i_n"]).reshape(V, S, 2), vlist)
    assert 0 < int(ok.sum()) < ok.numel()
    full = ro.full_res_features(lv)
    for v in range(V):
        close(aux[v], taps["aux_merge_weight_block.0"][v][0][:, :45])
        px, py = [t.long() for t in c(d["sample_loc_i_n"]).reshape(V, S, 2)[v, s].to(torch.int32).unbind(-1)]
        px, py = torch.where(ok[v], px, 0), torch.where(ok[v], py, 0)
        close(aux[v], full[v][:, py, px].t())
    sig = torch.stack([torch.sigmoid(taps["aux_merge_weight_block.6"][v][1][:, 0]) for v in range(V)])
    close(h.ref_blend(aux, sig, ok.to(dt), None), taps["color_mixup_block.0"][0][0][:, 45:])
    x = torch.randn(50, 6, dtype=dt)
    close(h.ref_pos_enc(x, 5), ro.pos_enc(x, 5))
    close(h.ref_view_enc(x[:, :3], 4), ro.pos_enc(x[:, :3], 4, ori=True)[:, 3:])
