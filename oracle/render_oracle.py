"""CPU oracle for the differentiable half of the per-ray sample pipeline.

TEST INFRASTRUCTURE ONLY.  Nothing in the product package imports this file; it is used by
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs of
``bench.py`` as the checker / CPU arm.

It is a plain-torch (CPU, fp32 or fp64) restatement of what the reference computes after the
neighbour query, written from the equations in SURVEY.md Appendix B/D:

  * projection into the reference views + delta view dirs
        (reference: models/neural_points_volumetric_model.py:248-255, :287-310)
  * distance features, inverse-distance weights, confidence clamp
        (reference: models/aggregators/point_aggregators.py:1427-1522, :825-833, :1422-1424)
  * per-neighbour MLP, weighted K-sum, per-sample colour-feature MLP
        (reference: point_aggregators.py:892-1037, models/helpers/networks.py:175-189)
  * conv feature pyramid, nearest-pixel lookup, learned multi-view blend, drop, mix-up, colour head
        (reference: point_aggregators.py:1042-1344)
  * ray_dist prologue and alpha compositing
        (reference: neural_points_volumetric_model.py:331-339, models/rendering/diff_ray_marching.py:508-557)
  * patch blur module
        (reference: models/base_rendering_model.py:677-786)

Parity pinning: the reference ships no tests / golden vectors for this path.  The oracle is pinned
against outputs of the reference itself, generated in the build container by
``tests/golden/make_golden.py`` (which imports the unmodified reference from /root/reference) and
committed under ``tests/golden/*.npz``; ``tests/test_oracle_golden.py`` checks every function here
against those fixtures.

Gradients come from torch autograd through this restatement.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

LRELU_SLOPE = 0.01  # nn.LeakyReLU default, reference act_type="LeakyReLU"


@dataclass
class AggCfg:
    """Hyper-parameters the shipped scripts fix (SURVEY.md §8d)."""
    K: int = 8
    feat_dim: int = 32
    num_feat_freqs: int = 3
    dist_xyz_freq: int = 5
    num_viewdir_freqs: int = 4
    use_nearest: int = 4
    is_train: bool = False
    drop_ratio: float = 0.0
    drop_patch: int = 1
    dilation_setup: str = "7_8_1_8"
    return_weights: bool = True   # zero_one_loss_items contains conf_coefficient


# ----------------------------------------------------------------------------------------------
# small helpers
# ----------------------------------------------------------------------------------------------
def pos_enc(x: torch.Tensor, freqs: int, ori: bool = False) -> torch.Tensor:
    """helpers/networks.py:175-189.  Non-``ori``: per channel d, per freq f: [sin, cos] interleaved.
    ``ori``: [x, all sines (d-major, f-minor), all cosines]."""
    bands = (2.0 ** torch.arange(freqs, dtype=torch.float32)).to(x)
    ang = (x.unsqueeze(-1) * bands).flatten(-2)          # (..., D*F), index d*F+f
    if ori:
        return torch.cat([x, torch.sin(ang), torch.cos(ang)], dim=-1)
    return torch.stack([torch.sin(ang), torch.cos(ang)], dim=-1).flatten(-2)


def _lin(x, P, name):
    return F.linear(x, P[name + ".weight"], P[name + ".bias"])


KINK_TAP = None      # tests set this to a list: every LeakyReLU then records min |pre-activation| per row (see kink_free_rays)


def _act(x):
    if KINK_TAP is not None:
        KINK_TAP.append(x.detach().abs().amin(dim=-1).reshape(-1))
    return F.leaky_relu(x, LRELU_SLOPE)


def kink_free_rays(taps, sample_pnt_mask: torch.Tensor, ray_valid: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """(R,) bool: rays none of whose hidden units has a pre-activation within `eps` of the LeakyReLU kink.  LeakyReLU' jumps by a
    factor 100 at 0, so two correct fp32 implementations that sum in a different order may take different slopes for such a unit;
    gradient parity tests mask those rays out of the colour loss (their gradient paths are then exactly zero on both sides).
    taps: the KINK_TAP list of one aggregate() call; rows are compacted valid neighbours (block1 / block3) or valid samples."""
    B, R, SR, K = sample_pnt_mask.shape
    nbr_ray = torch.nonzero(sample_pnt_mask.reshape(-1)).reshape(-1) // (SR * K)
    smp_ray = torch.nonzero(ray_valid.reshape(-1)).reshape(-1) // SR
    ok = torch.ones(R, dtype=torch.bool)
    for mn in taps:
        if mn.numel() == nbr_ray.numel():
            rows = nbr_ray
        elif mn.numel() == smp_ray.numel():
            rows = smp_ray
        else:
            continue            # activations of the image pyramid (per pixel, not per ray)
        ok[rows[mn < eps]] = False
    return ok


def drop_patch_positions(patch_size: int, patch_num: int, drop_ratio: float) -> np.ndarray:
    """point_aggregators.py:14-23: raster positions (on the S x S patch raster) of the first
    floor(P^2*ratio) patches in row-major patch order."""
    S = patch_size * patch_num
    n = int(patch_num * patch_num * drop_ratio)
    rows, cols = divmod(n, patch_num)
    flag = np.zeros((S, S), dtype=bool)
    flag[: rows * patch_size, :] = True
    flag[rows * patch_size: (rows + 1) * patch_size, : cols * patch_size] = True
    return np.nonzero(flag.reshape(-1))[0]


# ----------------------------------------------------------------------------------------------
# P1: projection into reference views, delta view directions
# ----------------------------------------------------------------------------------------------
def project_to_views(sample_loc_w: torch.Tensor, intrinsic: torch.Tensor, c2w_n: torch.Tensor) -> torch.Tensor:
    """sample_loc_w (R,SR,3), intrinsic (3,3), c2w_n (V,4,4) -> pixel xy (V,R,SR,2).
    neural_points_volumetric_model.py:248-255 (no half-pixel offset, divide by z+1e-10)."""
    out = []
    ones = torch.ones_like(sample_loc_w[..., :1])
    xh = torch.cat([sample_loc_w, ones], dim=-1)
    for v in range(c2w_n.shape[0]):
        w2c_t = torch.inverse(c2w_n[v]).t()
        xc = xh @ w2c_t
        xi = xc[..., :3] @ intrinsic.t()
        out.append((xi / (xi[..., 2:3] + 1e-10))[..., :2])
    return torch.stack(out)


def delta_viewdirs(sample_loc_w: torch.Tensor, campos: torch.Tensor, campos_n: torch.Tensor) -> torch.Tensor:
    """(R,SR,3), (3,), (V,3) -> (V,R,SR,3).  neural_points_volumetric_model.py:296-310."""
    cur = sample_loc_w - campos
    cur = cur / (torch.linalg.norm(cur, dim=-1, keepdim=True) + 1e-6)
    out = []
    for v in range(campos_n.shape[0]):
        d = sample_loc_w - campos_n[v]
        d = d / (torch.linalg.norm(d, dim=-1, keepdim=True) + 1e-6)
        out.append(d - cur)
    return torch.stack(out)


# ----------------------------------------------------------------------------------------------
# I1: feature pyramid
# ----------------------------------------------------------------------------------------------
def feature_pyramid(img_nhwc: torch.Tensor, P: Dict[str, torch.Tensor]):
    """img (V,H,W,3) -> (rgb NCHW, s1, s2, s3).  point_aggregators.py:1047-1063."""
    x = img_nhwc.permute(0, 3, 1, 2)
    lv = [x]
    for name in ("aux_block_s1", "aux_block_s2", "aux_block_s3"):
        x = _act(F.conv2d(x, P[name + ".0.weight"], P[name + ".0.bias"], stride=2, padding=1))
        x = _act(F.conv2d(x, P[name + ".2.weight"], P[name + ".2.bias"], stride=1, padding=1))
        lv.append(x)
    return lv


def full_res_features(levels) -> torch.Tensor:
    """bilinear-upsample (align_corners=False) each level to HxW and concat -> (V,45,H,W);
    pixel (0,0) zeroed as the invalid slot.  point_aggregators.py:1064-1067, :1089."""
    H, W = levels[0].shape[-2:]
    full = torch.cat([levels[0]] + [F.interpolate(l, size=[H, W], mode="bilinear") for l in levels[1:]], dim=1)
    keep = torch.ones(1, 1, H, W, dtype=full.dtype, device=full.device)
    keep[..., 0, 0] = 0.0
    return full * keep


# ----------------------------------------------------------------------------------------------
# A1-A4 + I2-I5: the aggregator
# ----------------------------------------------------------------------------------------------
def aggregate(P: Dict[str, torch.Tensor], cfg: AggCfg,
              sampled_color, sampled_Rw2c, sampled_dir, sampled_conf, sampled_embedding,
              sampled_xyz_pers, sampled_xyz, sample_pnt_mask, sample_loc, sample_loc_w,
              sample_ray_dirs, img_n=None, sample_loc_i_n=None, delta_viewdir_n=None):
    """Same argument meaning as PointAggregator.forward (point_aggregators.py:1427).
    Shapes: sampled_* (1,R,SR,K,C); sample_pnt_mask (1,R,SR,K) bool; sample_loc* (1,R,SR,3);
    img_n (1,V,H,W,3); sample_loc_i_n (V,R,SR,2); delta_viewdir_n (V,R,SR,3).
    Returns decoded (1,R,SR,4), ray_valid (1,R,SR) bool, weight (1,R,SR,K), conf_coefficient."""
    B, R, SR, K = sample_pnt_mask.shape
    dt = sampled_embedding.dtype
    valid = sample_pnt_mask.any(dim=-1).reshape(-1)            # per-sample validity
    if valid.numel() == 0 or int(valid.sum()) == 0:
        return torch.zeros(B, R, SR, 4, dtype=dt), valid.view(B, R, SR), None, None

    # distance features (agg_dist_pers == 20), :1472-1480
    zk, zs = sampled_xyz_pers[..., 2], sample_loc[..., None, 2]
    d_pers = torch.stack([sampled_xyz_pers[..., 0] * zk - sample_loc[..., None, 0] * zs,
                          sampled_xyz_pers[..., 1] * zk - sample_loc[..., None, 1] * zs,
                          zk - zs], dim=-1)
    d_world = sampled_xyz - sample_loc_w[..., None, :]
    dists = torch.cat([d_world, d_pers], dim=-1)               # (1,R,SR,K,6)

    # inverse-distance weights (linear), normalisation, confidence, :825-833, :1500-1508
    maskf = sample_pnt_mask.to(dt)
    w = maskf / torch.clamp(torch.linalg.norm(dists[..., :3], dim=-1), min=1e-6)
    w = w / torch.clamp(w.sum(dim=-1, keepdim=True), min=1e-8)
    conf = sampled_conf[..., 0]
    conf_coef = conf - (conf - conf.clamp(1e-4, 1.0)).detach()
    wc = w * conf_coef

    Rt = sampled_Rw2c.transpose(-1, -2)
    mflat = sample_pnt_mask.reshape(-1)

    # per-neighbour branch
    dflat = dists.reshape(-1, 6)[mflat].clone()
    dflat = torch.cat([dflat[:, :3] @ Rt, dflat[:, 3:]], dim=-1)
    d_enc = pos_enc(dflat, cfg.dist_xyz_freq)
    e = sampled_embedding.reshape(-1, cfg.feat_dim)[mflat]
    x = torch.cat([e, pos_enc(e, cfg.num_feat_freqs), d_enc], dim=-1)
    x = _act(_lin(x, P, "block1.0"))
    x = _act(_lin(x, P, "block1.2"))
    view_all = sample_ray_dirs.reshape(-1, 3) @ Rt              # (R*SR,3) unnormalised
    view_enc_all = pos_enc(view_all, cfg.num_viewdir_freqs, ori=True)
    ori_view = view_enc_all[:, :3].unsqueeze(1).expand(-1, K, -1).reshape(-1, 3)[mflat]
    col = sampled_color.reshape(-1, 3)[mflat]
    pdir = sampled_dir.reshape(-1, 3)[mflat] @ Rt
    x = torch.cat([x, col, pdir - ori_view, (pdir * ori_view).sum(-1, keepdim=True)], dim=-1)
    x = _act(_lin(x, P, "block3.0"))
    h = _act(_lin(x, P, "block3.2"))
    alpha = F.softplus(_lin(h, P, "alpha_branch.0") - 1.0)

    wcf = wc.reshape(-1, K, 1)
    a_full = torch.zeros(B * R * SR * K, 1, dtype=dt).index_put((mflat.nonzero()[:, 0],), alpha)
    h_full = torch.zeros(B * R * SR * K, h.shape[-1], dtype=dt).index_put((mflat.nonzero()[:, 0],), h)
    sigma = (a_full.view(-1, K, 1) * wcf).sum(dim=1)[valid]
    feat = (h_full.view(-1, K, h.shape[-1]) * wcf).sum(dim=1)[valid]

    # per-sample colour feature branch
    g = torch.cat([feat, view_enc_all[valid, 3:]], dim=-1)
    g = _act(_lin(g, P, "color_feature_branch.0"))
    g = _act(_lin(g, P, "color_feature_branch.2"))
    g = _act(_lin(g, P, "color_feature_branch.4"))

    C_aux = 45
    V = cfg.use_nearest
    if V > 0:
        levels = feature_pyramid(img_n[0], P)
        full = full_res_features(levels)                       # (V,45,H,W)
        H1, W1 = full.shape[-2:]
        xy = sample_loc_i_n.reshape(V, -1, 2)[:, valid, :]
        px = xy[..., 0].to(torch.int32).long()                 # truncation toward zero
        py = xy[..., 1].to(torch.int32).long()
        bad = (px < 0) | (px >= W1) | (py < 0) | (py >= H1)
        px = torch.where(bad, torch.zeros_like(px), px)
        py = torch.where(bad, torch.zeros_like(py), py)
        ok = (~bad).to(dt)
        dv = delta_viewdir_n.reshape(V, -1, 3)[:, valid, :]
        num, den = 0.0, 0.0
        for v in range(V):
            a_v = full[v][:, py[v], px[v]].t()                 # (Nv,45)
            t = torch.cat([a_v, g, dv[v]], dim=-1)
            t = _act(_lin(t, P, "aux_merge_weight_block.0"))
            t = _act(_lin(t, P, "aux_merge_weight_block.2"))
            t = _act(_lin(t, P, "aux_merge_weight_block.4"))
            wv = torch.sigmoid(_lin(t, P, "aux_merge_weight_block.6")) * ok[v][:, None]
            num = num + a_v * wv
            den = den + wv
        merged = num / (den + 1e-6)
        if cfg.is_train and cfg.drop_ratio > 0:
            toks = cfg.dilation_setup.split("_")
            pos = drop_patch_positions(int(toks[1]), int(toks[0]), cfg.drop_ratio)
            flag = np.zeros((R, SR), dtype=bool)
            flag[pos, :] = True        # IndexError if a raster position >= R (same as the reference)
            dropped = torch.from_numpy(flag.reshape(-1))[valid]
            merged = merged * (~dropped).to(dt)[:, None]
    else:
        merged = torch.zeros(g.shape[0], C_aux, dtype=dt)

    gi, gv = g[:, :C_aux], g[:, C_aux:]
    m = torch.cat([gi, merged], dim=-1)
    m = _act(_lin(m, P, "color_mixup_block.0"))
    m = _act(_lin(m, P, "color_mixup_block.2"))
    m = _lin(m, P, "color_mixup_block.4") + gi
    rgb = torch.sigmoid(_lin(torch.cat([m, gv], dim=-1), P, "color_final_block.0")) * 1.002 - 0.001

    out = torch.zeros(B * R * SR, 4, dtype=dt).index_put((valid.nonzero()[:, 0],), torch.cat([sigma, rgb], dim=-1))
    return out.view(B, R, SR, 4), valid.view(B, R, SR), w, conf_coef


# ----------------------------------------------------------------------------------------------
# C1, C2: compositing
# ----------------------------------------------------------------------------------------------
def ray_dist_from_depth(sample_z: torch.Tensor, ray_valid: torch.Tensor, vsize_z: float, unit_mode: bool = True):
    """(1,R,SR) camera depth -> segment lengths.  neural_points_volumetric_model.py:331-339."""
    m = torch.cummax(sample_z, dim=-1)[0]
    last = torch.full_like(m[..., :1], vsize_z)
    d = torch.cat([m[..., 1:] - m[..., :-1], last], dim=-1)
    bad = d < 1e-8
    if unit_mode:
        bad = bad | (d > 2 * vsize_z)
    badf = bad.to(d.dtype)
    d = d * (1.0 - badf) + badf * vsize_z
    return d * ray_valid.to(d.dtype)


def ray_march(ray_dist, ray_valid, feats, bg_color=None):
    """diff_ray_marching.py:508-557 with radiance_render + alpha_blend.
    Returns ray_color (1,R,3), point_color, opacity, acc_transmission, blend_weight (…,1),
    background_transmission (1,R,1), background_blend_weight."""
    sigma = feats[..., 0] * ray_valid.to(feats.dtype)
    opacity = 1 - torch.exp(-sigma * ray_dist)
    a = 1.0 - opacity + 1e-10
    T_incl = torch.cumprod(a, dim=-1)
    bg_T = T_incl[..., -1:]
    T = torch.cat([torch.ones_like(bg_T), T_incl[..., :-1]], dim=-1)
    bw = (opacity * T).unsqueeze(-1)
    color = (feats[..., 1:] * bw).sum(dim=-2)
    if bg_color is not None:
        color = color + bg_color.view(-1, 1, 3).to(color) * bg_T
    return color, feats[..., 1:], opacity, T, bw, bg_T, bg_T


# ----------------------------------------------------------------------------------------------
# B1: blur module
# ----------------------------------------------------------------------------------------------
def blur_select(pred: torch.Tensor, gt: torch.Tensor, kernels: torch.Tensor, patch_num: int, patch_size: int, select=None):
    """pred, gt (1,S*S,3) on an S x S raster of patch_num^2 patches; kernels (1,Nk,kh,kw).
    Returns (new_pred (1,S*S,3), select_index (patch_num^2,)).  base_rendering_model.py:677-786.
    `select` (patch_num^2,): use these candidates instead of the argmin (tests pass the product's pick where two candidates'
    errors tie to rounding)."""
    cand, err = blur_candidates(pred, gt, kernels, patch_num, patch_size)
    sel = torch.argmin(err, dim=1) if select is None else torch.as_tensor(select).long().reshape(-1)
    best = cand[torch.arange(cand.shape[0]), :, sel]                   # (P2,3,p,p)
    S = patch_num * patch_size
    img = best.reshape(patch_num, patch_num, 3, patch_size, patch_size).permute(2, 0, 3, 1, 4).reshape(3, S, S)
    return img.permute(1, 2, 0).reshape(1, S * S, 3), sel


def blur_candidates(pred: torch.Tensor, gt: torch.Tensor, kernels: torch.Tensor, patch_num: int, patch_size: int):
    """every candidate of blur_select: (cand (P2,3,Nk+1,p,p) -- the Nk border-renormalised blurs, then the patch itself --,
    err (P2,Nk+1) the L1 distance of each candidate to the ground truth)"""
    Nk, kh = kernels.shape[1], kernels.shape[2]
    xp, gp = _blur_patches(pred, patch_num, patch_size), _blur_patches(gt, patch_num, patch_size)
    flat = xp.reshape(-1, 1, patch_size, patch_size)
    k = kernels[0].unsqueeze(1).to(flat)
    norm = F.conv2d(torch.ones_like(flat), k, padding=kh // 2)
    blurred = F.conv2d(flat, k, padding=kh // 2) / norm               # (P2*3,Nk,p,p)
    cand = torch.cat([blurred, flat], dim=1).reshape(-1, 3, Nk + 1, patch_size, patch_size)
    err = (cand - gp.unsqueeze(2)).abs().sum(dim=(1, 3, 4))            # (P2,Nk+1)
    return cand, err


# ----------------------------------------------------------------------------------------------
# N3: learnable blur-kernel branch
# ----------------------------------------------------------------------------------------------
def learnable_blur(pred: torch.Tensor, gt: torch.Tensor, weights, patch_num: int, patch_size: int, kernel_size: int = 9,
                   kernel_mode: int = 4, kernel_norm: int = 0, boundary_mode: int = 0):
    """pred, gt (1,S*S,3) on the patch raster; weights = [(W,b)] * 4 of learn_blur_kernel_block (point_aggregators.py:715-749).
    Returns (new_pred (1,S*S,3), raw predictor output (N, ks^2 [+1])).  base_rendering_model.py:827-1020 with
    learnable_blur_kernel_conv=0."""
    N = patch_num * patch_num
    xp, gp = _blur_patches(pred, patch_num, patch_size), _blur_patches(gt, patch_num, patch_size)
    x = torch.cat([gp.mean(dim=1).reshape(N, -1), xp.mean(dim=1).reshape(N, -1)], dim=-1)          # :887-889
    for i, (W, b) in enumerate(weights):
        x = F.linear(x, W, b)
        x = torch.sigmoid(x) if i == len(weights) - 1 else _act(x)
    return learnable_blur_apply(pred, x, patch_num, patch_size, kernel_size, kernel_mode, kernel_norm, boundary_mode), x


def _blur_patches(x, patch_num, patch_size):
    """(1,S*S,3) patch raster -> (patch_num^2,3,p,p), patches in row-major order"""
    S = patch_num * patch_size
    x = x.reshape(S, S, 3).permute(2, 0, 1).reshape(3, patch_num, patch_size, patch_num, patch_size)
    return x.permute(1, 3, 0, 2, 4).reshape(patch_num * patch_num, 3, patch_size, patch_size)


def learnable_blur_apply(pred: torch.Tensor, raw: torch.Tensor, patch_num: int, patch_size: int, kernel_size: int = 9,
                         kernel_mode: int = 4, kernel_norm: int = 0, boundary_mode: int = 0):
    """the part of learnable_blur after the predictor: raw predictor output (N, ks^2 [+1]) -> per-patch kernel -> blurred
    patch raster (1,S*S,3).  base_rendering_model.py:895-1005."""
    S, N, KK = patch_num * patch_size, patch_num * patch_num, kernel_size * kernel_size
    xp = _blur_patches(pred, patch_num, patch_size)
    if kernel_norm == 0:                                                                             # :895-899
        k = raw[:, :KK].view(N, 1, kernel_size, kernel_size)
        k = k / k.sum(dim=(2, 3), keepdim=True)
    else:
        k = F.softmax(raw[:, :KK], dim=-1).view(N, 1, kernel_size, kernel_size)
    if kernel_mode == 4:                                                                             # :904-909
        wc = raw[:, -1][:, None, None, None]
        ident = torch.zeros_like(k)
        ident[:, :, kernel_size // 2, kernel_size // 2] = 1.0
        k = wc * k + (1 - wc) * ident
        k = k / k.sum(dim=(2, 3), keepdim=True)
    elif kernel_mode != 0:
        raise NotImplementedError
    xin = xp.permute(1, 0, 2, 3)                                                                     # (3,N,p,p): groups = patches
    pad = kernel_size // 2
    if boundary_mode == 0:                                                                           # :915-923
        m = F.conv2d(torch.ones_like(xin), k, padding=pad, groups=N)
        y = F.conv2d(xin, k, padding=pad, groups=N) / (m + 1e-10)
    elif boundary_mode in (1, 2):
        m = F.conv2d(torch.ones_like(xin), k if boundary_mode == 1 else k.detach(), padding=pad, groups=N)
        y = F.conv2d(xin, k, padding=pad, groups=N) + (1 - m) * xin
    else:
        raise NotImplementedError
    best = y.permute(1, 0, 2, 3)                                                                     # (N,3,p,p)
    img = best.reshape(patch_num, patch_num, 3, patch_size, patch_size).permute(2, 0, 3, 1, 4).reshape(3, S, S)
    return img.permute(1, 2, 0).reshape(1, S * S, 3)


def blur_predictor_params(seed: int, patch_size: int = 8, kernel_size: int = 9, kernel_mode: int = 4):
    """seeded weights [(W,b)]*4 of learn_blur_kernel_block (numpy PCG64; larger than init_seq's so the predicted taps are far
    from uniform).  Used by tests/golden/make_golden.py and by the tests, so the fixtures store only reference OUTPUTS."""
    rng = np.random.default_rng(seed)
    sizes = [2 * patch_size * patch_size, 128, 128, 128, kernel_size * kernel_size + (1 if kernel_mode in (2, 4) else 0)]
    out = []
    for i in range(4):
        W = (rng.standard_normal((sizes[i + 1], sizes[i])) * (2.5 / np.sqrt(sizes[i]))).astype(np.float32)
        b = (rng.standard_normal((sizes[i + 1],)) * 0.5).astype(np.float32)
        out.append((torch.from_numpy(W), torch.from_numpy(b)))
    return out


# ----------------------------------------------------------------------------------------------
# weights
# ----------------------------------------------------------------------------------------------
# the seeded weight generator lives with the other synthetic-input generators (product side, no oracle import needed by bench.py);
# re-exported here because the tests and the golden generator call it through the oracle
from hybridneuralrendering_b200.synthetic import CONV_SHAPES, LAYER_SHAPES, random_aggregator_params as random_params  # noqa: E402,F401
