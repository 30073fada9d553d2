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
