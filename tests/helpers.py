"""shared helpers for the GPU parity tests (the oracle is the checker, never the thing measured)."""
import os

import numpy as np
import torch

from hybridneuralrendering_b200 import make_opt
from hybridneuralrendering_b200 import synthetic as syn
from oracle import render_oracle as ro

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
T = torch.from_numpy


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))


def cuda(x):
    return (T(x) if isinstance(x, np.ndarray) else x).cuda()


def build_aggregator(P, **opt_over):
    from hybridneuralrendering_b200 import PointAggregator
    agg = PointAggregator(make_opt(**opt_over)).cuda()
    missing = agg.load_state_dict(P, strict=False)
    assert not missing.unexpected_keys
    return agg


def blur_predictor(params):
    """learn_blur_kernel_block with the given [(W,b)]*4, built by the product's own aggregator so the state_dict names are the
    checkpoint's (learn_blur_kernel_block.{0,2,4,6})."""
    from hybridneuralrendering_b200 import PointAggregator
    KK1, K0 = params[-1][0].shape[0], params[0][0].shape[1]
    ks = int(np.sqrt(KK1))
    agg = PointAggregator(make_opt(is_train=True, learnable_blur_kernel=1, learnable_blur_kernel_size=ks,
                                   learnable_blur_patch_size=int(np.sqrt(K0 // 2)), learnable_blur_kernel_mode=4 if KK1 > ks * ks else 0)).cuda()
    sd = {}
    for li, (W, b) in enumerate(params):
        sd[f"learn_blur_kernel_block.{2 * li}.weight"], sd[f"learn_blur_kernel_block.{2 * li}.bias"] = W, b
    missing = agg.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys
    return agg.learn_blur_kernel_block


def run_dropin(agg, d, g, grad=False):
    """call the drop-in forward with the gathered tensors of synthetic case (d, g)"""
    leaf = {k: cuda(g[k]).clone().requires_grad_(grad) for k in ("sampled_embedding", "sampled_color", "sampled_dir", "sampled_conf")}
    out = agg(leaf["sampled_color"], torch.eye(3).cuda(), leaf["sampled_dir"], leaf["sampled_conf"], leaf["sampled_embedding"],
              cuda(g["sampled_xyz_pers"]), cuda(g["sampled_xyz"]), cuda(g["sample_pnt_mask"]), cuda(d["sample_loc"]), cuda(d["sample_loc_w"]),
              cuda(d["sample_ray_dirs"]), d["vsize"], 0, img_n=cuda(d["images_nearest"]), sample_loc_i_n=cuda(d["sample_loc_i_n"]),
              delta_viewdir_n=cuda(d["delta_viewdir_n"]))
    return out, leaf


def run_oracle(d, g, P, cfg, dtype=torch.float32, grad=False):
    c = lambda a: T(a).to(dtype)
    leaf = {k: c(g[k]).clone().requires_grad_(grad) for k in ("sampled_embedding", "sampled_color", "sampled_dir", "sampled_conf")}
    Pd = {k: v.to(dtype).clone().requires_grad_(grad) for k, v in P.items()}
    out = ro.aggregate(Pd, cfg, leaf["sampled_color"], torch.eye(3, dtype=dtype), leaf["sampled_dir"], leaf["sampled_conf"],
                       leaf["sampled_embedding"], c(g["sampled_xyz_pers"]), c(g["sampled_xyz"]), T(g["sample_pnt_mask"]),
                       c(d["sample_loc"]), c(d["sample_loc_w"]), c(d["sample_ray_dirs"]), img_n=c(d["images_nearest"]),
                       sample_loc_i_n=c(d["sample_loc_i_n"]), delta_viewdir_n=c(d["delta_viewdir_n"]))
    return out, leaf, Pd


def assert_close(a, b, rtol, atol, msg=""):
    a = a.detach().cpu().double().numpy() if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = b.detach().cpu().double().numpy() if torch.is_tensor(b) else np.asarray(b, np.float64)
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=msg)


def grad_atol(ref, scale=1e-4):
    """gradients span many orders of magnitude: rtol 1e-4 plus an atol of 1e-4 x the tensor's max
    magnitude (stated tolerance for tiny-magnitude entries, SURVEY.md §7.3)."""
    r = ref.detach().cpu().numpy() if torch.is_tensor(ref) else np.asarray(ref)
    return float(np.abs(r).max()) * scale + 1e-12


# ------------------------------------------------------------------------------------------------------------------------------
# Plain references of the aggregation glue and image-branch kernels (csrc/aggregate.cu, csrc/pyramid.cu), written from the formulas
# of oracle/render_oracle.py (aggregate(), pos_enc, feature_pyramid, full_res_features) but shaped like the kernels' arguments:
# point tables + neighbour ids instead of gathered (1,R,SR,K,C) tensors, NHWC levels.  Device- and dtype-agnostic (the GPU tests
# run them in fp64 on the GPU; test_oracle_golden checks them against the oracle on the CPU).  cam is the 21-float block of
# ops.make_cam: [campos 3 | camrot 9 (c2w) | Rw2c^T 9], each 3x3 row-major; the kernels' rot3(m, v) is v @ m.
# ------------------------------------------------------------------------------------------------------------------------------
CONF_LO = float(np.float32(1e-4))        # the kernel clamps with the fp32 constant 1e-4f


def ref_pos_enc(x, freqs):
    """per channel d, per frequency 2^f: [sin, cos] interleaved, index (d * freqs + f) * 2 (networks.py:175-189, not `ori`)"""
    ang = (x.unsqueeze(-1) * 2.0 ** torch.arange(freqs, dtype=x.dtype, device=x.device)).flatten(-2)
    return torch.stack([ang.sin(), ang.cos()], -1).flatten(-2)


def ref_view_enc(v, freqs):
    """the `ori=True` encoding without its raw 3 columns: all sines (d-major, f-minor), then all cosines"""
    ang = (v.unsqueeze(-1) * 2.0 ** torch.arange(freqs, dtype=v.dtype, device=v.device)).flatten(-2)
    return torch.cat([ang.sin(), ang.cos()], -1)


def ref_nbr_weights(xyz, conf, pidx, mask, loc_w):
    """inverse-distance weights of the live slots normalised per sample, clamped confidence (straight-through: differentiable as
    the identity) and per-sample validity.  pidx (S,K) int; mask (S,K) u8 or None (then live = pidx >= 0); masked slots read point
    0 (clamp(pidx, 0)).  -> weight (S,K), confc (S,K), valid (S,) bool"""
    live = (mask != 0) if mask is not None else (pidx >= 0)
    g = pidx.long().clamp_min(0)
    u = live.to(xyz.dtype) / (xyz[g] - loc_w[:, None, :]).norm(dim=-1).clamp_min(1e-6)
    w = u / u.sum(-1, keepdim=True).clamp_min(1e-8)
    if conf is None:
        confc = torch.ones_like(w)
    else:
        c = conf.reshape(-1)[g]
        confc = c - (c - c.clamp(CONF_LO, 1.0)).detach()
    return w, confc, live.any(-1)


def ref_nbr_features(xyz, xyz_pers, emb, color, dirs, pidx, vlist, loc_w, loc_pers, raydirs, cam):
    """MLP input rows of every (vlist sample, slot): X0 (Nv*K, 284) = [emb 32 | PE(emb, 3) 192 | PE(d, 5) 60], d = [world offset
    rotated by Rw2c | perspective offset (agg_dist_pers 20)]; E (Nv*K, 7) = [colour | dirR - viewR | <dirR, viewR>].  xyz_pers None:
    the point's perspective coordinates are computed from cam.  Masked slots read point 0 like the kernel (their rows are never used)."""
    K = pidx.shape[1]
    s = vlist.long().repeat_interleave(K)
    g = pidx[vlist.long()].long().clamp_min(0).reshape(-1)
    rt, p = cam[12:21].reshape(3, 3), xyz[g]
    if xyz_pers is None:
        c = (p - cam[:3]) @ cam[3:12].reshape(3, 3)
        q = torch.stack([c[:, 0] / c[:, 2], c[:, 1] / c[:, 2], c[:, 2]], -1)
    else:
        q = xyz_pers[g]
    sp = loc_pers[s]
    d_pers = torch.stack([q[:, 0] * q[:, 2] - sp[:, 0] * sp[:, 2], q[:, 1] * q[:, 2] - sp[:, 1] * sp[:, 2], q[:, 2] - sp[:, 2]], -1)
    e = emb[g]
    X0 = torch.cat([e, ref_pos_enc(e, 3), ref_pos_enc(torch.cat([(p - loc_w[s]) @ rt, d_pers], -1), 5)], -1)
    view, dr = raydirs[s] @ rt, dirs[g] @ rt
    E = torch.cat([color[g], dr - view, (dr * view).sum(-1, keepdim=True)], -1)
    return X0, E


def ref_alpha_ksum(H, wc, w_alpha, b_alpha, view):
    """density head + weighted K-sum: H (Nv*K, 256) layer-3 outputs, wc (Nv, K) = weight * confc of the vlist samples, view (Nv, 3)
    rotated ray directions.  -> sigma (Nv,) = sum_k wc softplus(raw - 1), X5 (Nv, 280) = [sum_k wc H | view encoding 24],
    raw (Nv*K,) = H w_alpha + b_alpha"""
    K = wc.shape[1]
    raw = H @ w_alpha.reshape(-1) + b_alpha.reshape(())
    sigma = (torch.nn.functional.softplus(raw - 1.0).reshape(-1, K) * wc).sum(-1)
    feat = (H.reshape(-1, K, H.shape[1]) * wc[..., None]).sum(1)
    return sigma, torch.cat([feat, ref_view_enc(view, 4)], -1), raw


def ref_image_gather(levels, xy, vlist):
    """levels NHWC (V,H,W,3), (V,h1,w1,6), (V,h2,w2,12), (V,h3,w3,24); xy (V,S,2) pixel coordinates.  Every level bilinearly
    upsampled to H x W (align_corners=False), then the pixel at the truncated coordinates; out-of-bounds pairs and pixel (0,0) read
    zeros.  -> aux (V,Nv,45), ok (V,Nv) bool (in bounds)"""
    V, H, W = levels[0].shape[:3]
    full = torch.cat([levels[0]] + [torch.nn.functional.interpolate(l.permute(0, 3, 1, 2), size=(H, W), mode="bilinear",
                                                                    align_corners=False).permute(0, 2, 3, 1) for l in levels[1:]], -1)
    p = xy[:, vlist.long()]
    px, py = p[..., 0].to(torch.int32).long(), p[..., 1].to(torch.int32).long()        # truncation toward zero
    ok = (px >= 0) & (px < W) & (py >= 0) & (py < H)
    keep = ok & ~((px == 0) & (py == 0))
    vi = torch.arange(V, device=xy.device)[:, None]
    aux = full[vi, torch.where(ok, py, 0), torch.where(ok, px, 0)] * keep[..., None].to(full.dtype)
    return aux, ok


def ref_blend(aux, sig, ok, keep):
    """learned multi-view blend: aux (V,Nv,45), sig, ok (V,Nv), keep (Nv,) or None -> merged (Nv,45) = keep * num / (den + 1e-6),
    num = sum_v aux_v w_v, den = sum_v w_v, w_v = sig_v ok_v"""
    w = (sig * ok)[..., None]
    m = (aux * w).sum(0) / (w.sum(0) + 1e-6)
    return m * keep.to(m.dtype)[:, None] if keep is not None else m


PYRAMID_STRIDES = (2, 1, 2, 1, 2, 1)


def ref_pyramid(img, ws, bs):
    """img (V,H,W,3) NHWC -> the six LeakyReLU(conv3x3) activations NCHW of s1.conv0, s1.conv1, s2.conv0, ... (levels: 1, 3, 5)"""
    x, acts = img.permute(0, 3, 1, 2), []
    for w, b, st in zip(ws, bs, PYRAMID_STRIDES):
        x = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(x, w, b, stride=st, padding=1), 0.01)
        acts.append(x)
    return acts
