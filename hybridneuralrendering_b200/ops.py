"""torch.autograd.Function wrappers around the libhnr kernels.

Every function here launches hand-written CUDA through the C ABI (``_lib``); there is no torch
fallback.  torch is used for allocation, streams and the autograd tape only.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import check, i64_array, lib, ptr, ptr_array, require_cuda, stream

ACT_NONE, ACT_LRELU, ACT_SIGMOID, ACT_COLOR = 0, 1, 2, 3
X0_W, E_W, HID, X5_W, AUX_C = 284, 7, 256, 280, 45
X0_GRAD_W = 224      # leading columns of the layer-0 input that carry a gradient: [emb 32 | sin/cos(2^j emb) 192]

# counts kernels launched through the C ABI (bench.py reports it as gpu_launches)
LAUNCHES = 0


def _count(n: int = 1):
    global LAUNCHES
    LAUNCHES += n


# Range guard of the split-fp16 tensor-core kernels: they saturate instead of overflowing and set a bit in this device word;
# the host looks at it at its next natural synchronisation point (the query's count read-back) and raises.
_STATUS = {}


def status_word(dev) -> torch.Tensor:
    key = torch.device(dev).index or 0
    if key not in _STATUS:
        _STATUS[key] = (torch.zeros(1, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32).pin_memory())
    return _STATUS[key][0]


def status_fetch_async(dev) -> None:
    """queue the copy of the status word to pinned host memory (call BEFORE a stream synchronisation)"""
    key = torch.device(dev).index or 0
    if key in _STATUS:
        _STATUS[key][1].copy_(_STATUS[key][0], non_blocking=True)


def status_check(dev) -> None:
    """after the synchronisation: raise if a tensor-core kernel had to saturate a value"""
    key = torch.device(dev).index or 0
    if key in _STATUS and int(_STATUS[key][1][0]) != 0:
        bits = int(_STATUS[key][1][0])
        _STATUS[key][0].zero_()
        _STATUS[key][1].zero_()
        raise RuntimeError(f"hybridneuralrendering_b200: a split-fp16 tensor-core kernel saturated an activation (status {bits}: "
                           "1 = per-neighbour MLP activation, 2 = per-sample chain value, 4 = weight beyond the fixed training scale); "
                           "hidden activations beyond +-1000 (weights beyond +-58 in training) do not fit the x64-scaled fp16 split of the fused "
                           "kernels; nothing was applied from this step (the fused Adam skips a flagged step on the device)")


# optional per-launch device timing (CUDA events on the launching stream); used by profiling.py / bench.py
TIMERS = None          # None = off, else a list of (tag, start_event, end_event)
_TAG = ["untagged"]


class tag:
    """`with ops.tag("nbr_mlp"):` labels the launches issued inside for the timers"""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        _TAG.append(self.name)

    def __exit__(self, *a):
        _TAG.pop()


class _launch:
    def __init__(self, n=1, name=None):
        self.n, self.name = n, name

    def __enter__(self):
        _count(self.n)
        if TIMERS is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.e = torch.cuda.Event(enable_timing=True)
            self.s.record()

    def __exit__(self, *a):
        if TIMERS is not None:
            self.e.record()
            TIMERS.append((_TAG[-1] if self.name is None else f"{_TAG[-1]}/{self.name}", self.s, self.e))


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _rows2d(t: torch.Tensor) -> torch.Tensor:
    """2-D fp32 view with unit inner stride (row stride may exceed the width)."""
    assert t.dim() == 2
    if t.dtype != torch.float32 or t.stride(1) != 1:
        t = t.float().contiguous()
    return t


def make_cam(campos: torch.Tensor, camrot: torch.Tensor, rw2c: Optional[torch.Tensor]) -> torch.Tensor:
    """21-float device block [campos(3), camrot(9) c2w rotation, rt(9) = Rw2c^T]; built with device
    ops only (no host sync)."""
    dev = campos.device
    rt = rw2c.detach().float().t().reshape(-1) if rw2c is not None else torch.eye(3, device=dev).reshape(-1)
    return torch.cat([campos.detach().float().reshape(-1)[:3], camrot.detach().float().reshape(-1)[:9], rt.to(dev)]).contiguous()


# --------------------------------------------------------------------------------------------
# dense layer
# --------------------------------------------------------------------------------------------
# forward engine of ops.linear: "tc" = tcgen05 3xTF32 kernel (csrc/linear_tc.cu) for layers with >= 16 outputs,
# "simt" = exact-fp32 FFMA kernel (csrc/linear_simt.cu).  Backward always uses the exact-fp32 kernels.
import os as _os
LINEAR_ENGINE = _os.environ.get("HNR_LINEAR_ENGINE", "tc")


def pack_linear(W: torch.Tensor):
    """(N,K) fp32 -> (uint8 image, Npad, Kp): zero-pad to Npad % 16 == 0, Kp % 8 == 0, split into TF32 hi (13 low
    mantissa bits cleared) and lo = w - hi, tile per 8-column chunk as [hi | lo], each part
    [k half (2)][row group (Npad/8)][row (8)][4 floats] -- the canonical no-swizzle K-major UMMA layout."""
    W = W.detach().float()
    N, K = W.shape
    Npad, Kp = (N + 15) // 16 * 16, (K + 7) // 8 * 8
    Wp = torch.zeros((Npad, Kp), device=W.device, dtype=torch.float32)
    Wp[:N, :K] = W
    hi = (Wp.view(torch.int32) & -8192).view(torch.float32)
    lo = Wp - hi
    tile = lambda x: x.view(Npad // 8, 8, Kp // 8, 2, 4).permute(2, 3, 0, 1, 4)
    img = torch.stack([tile(hi), tile(lo)], dim=1).contiguous().view(torch.uint8).reshape(-1)
    assert img.numel() == lib().hnr_linear_tc_packed_bytes(Npad, Kp)
    return img, Npad, Kp


def _packed_linear(W: torch.Tensor):
    """packed image cached ON the weight tensor object (a cache keyed by data_ptr would hand a stale image to a
    new tensor that the caching allocator placed at a recycled address)"""
    ent = getattr(W, "_hnr_pack", None)
    if ent is None or ent[0] != W._version:
        ent = (W._version, pack_linear(W))
        try:
            W._hnr_pack = ent
        except Exception:
            pass
    return ent[1]


def _packed_linear_T(W: torch.Tensor):
    """images of W^T for the tensor-core data gradient, one per slice of <= 256 input columns: [(k0, (image, Kpad, Np))];
    cached on the weight tensor like _packed_linear"""
    ent = getattr(W, "_hnr_packT", None)
    if ent is None or ent[0] != W._version:
        K = W.shape[1]
        packs = [(k0, pack_linear(W.detach()[:, k0:k0 + 256].t().contiguous())) for k0 in range(0, K, 256)]
        ent = (W._version, packs)
        try:
            W._hnr_packT = ent
        except Exception:
            pass
    return ent[1]


class LinearFn(torch.autograd.Function):
    """y = act(concat(srcs) W^T + b [+ res]).  `mods[i] > 0`: source i has mods[i] rows reused by
    every block of mods[i] output rows."""

    @staticmethod
    def forward(ctx, W, b, res, act: int, M: int, mods: Tuple[int, ...], *srcs):
        srcs = [_rows2d(s) for s in srcs]
        assert 1 <= len(srcs) <= 3
        W = _f32c(W)
        N, K = W.shape
        ks = [s.shape[1] for s in srcs] + [0] * (3 - len(srcs))
        assert sum(ks) == K, (ks, K)
        require_cuda(W, *srcs)
        Y = torch.empty((M, N), device=W.device, dtype=torch.float32)
        padded = list(srcs) + [None] * (3 - len(srcs))
        lds = [s.stride(0) if s is not None else 0 for s in padded]
        modl = list(mods) + [0] * (3 - len(mods))
        resv = _rows2d(res) if res is not None else None
        bc = _f32c(b) if b is not None else None
        if LINEAR_ENGINE == "tc" and N >= 16 and M >= 128:
            wpack, Npad, Kp = _packed_linear(W)
            with _launch(name=f"linear_tc_fwd[{M}x{N}x{K}]" if TIMERS is not None else None):
                check(lib().hnr_linear_tc_fwd(ptr_array(padded), i64_array(lds), i64_array(ks), i64_array(modl), ptr(wpack), Npad, Kp,
                                              ptr(bc), ptr(resv), resv.stride(0) if resv is not None else 0, ptr(Y), N, M, N, K, act,
                                              None, None, 0, None, stream()), "linear_tc_fwd")
        else:
            with _launch():
                check(lib().hnr_linear_fwd(ptr_array(padded), i64_array(lds), i64_array(ks), i64_array(modl), ptr(W), ptr(bc), ptr(resv),
                                           resv.stride(0) if resv is not None else 0, ptr(Y), N, M, N, K, act, stream()), "linear_fwd")
        ctx.act, ctx.M, ctx.mods, ctx.nsrc, ctx.has_res, ctx.has_b = act, M, modl, len(srcs), res is not None, b is not None
        ctx.save_for_backward(W, Y, *srcs)
        return Y

    @staticmethod
    def backward(ctx, dY):
        W, Y, *srcs = ctx.saved_tensors
        need_src = [ctx.needs_input_grad[6 + i] for i in range(ctx.nsrc)]
        need_w = ctx.needs_input_grad[0] or (ctx.has_b and ctx.needs_input_grad[1])
        d_srcs, dW, db = linear_backward(W, Y, srcs, ctx.mods, dY, ctx.act, need_src, need_w, ctx.has_b, M=ctx.M)
        d_res = dY if ctx.has_res else None
        return (dW, db, d_res, None, None, None, *d_srcs)


# narrowest layer whose backward runs on the tensor-core kernels.  The 64-wide blend-weight net spends 3.6 ms per training step there for
# ~0.5 ms of traffic (DESIGN.md 7): HNR_TC_BWD_MIN_N=65 sends it to the exact-fp32 SIMT kernels instead -- an A/B switch for round 2,
# the default (16) is the measured and validated configuration.
TC_BWD_MIN_N = int(os.environ.get("HNR_TC_BWD_MIN_N", "16"))


def linear_backward(W, Y, srcs, mods, dY, act: int, need_src, need_w: bool = True, has_b: bool = True, M: Optional[int] = None,
                    k_need: Optional[int] = None):
    """gradients of y = act(concat(srcs) W^T + b) given dY and the saved output Y: ([d_src_i | None], dW | None, db | None).
    Tensor-core kernels (3xTF32: gated data gradient, TMEM-resident weight gradient) for layers with >= 16 outputs and
    >= 128 rows, exact-fp32 SIMT kernels otherwise.  `k_need`: only the first k_need input columns of the data gradient are
    consumed by the caller (the rest of the returned buffer is left unwritten) -- a column slice nobody reads costs a full pass
    over dY."""
    srcs = [_rows2d(s) for s in srcs]
    nsrc = len(srcs)
    dY, Y = _rows2d(dY), _rows2d(Y)
    N, K = W.shape
    if M is None:
        M = dY.shape[0]
    mods = list(mods) + [0] * (3 - len(mods))
    ks = [s.shape[1] for s in srcs] + [0] * (3 - nsrc)
    padded = list(srcs) + [None] * (3 - nsrc)
    lds = [s.stride(0) if s is not None else 0 for s in padded]
    d_srcs: List[Optional[torch.Tensor]] = [None] * nsrc
    use_tc = LINEAR_ENGINE == "tc" and M >= 128 and N >= TC_BWD_MIN_N
    if any(need_src) and M > 0:
        if use_tc:
            # tensor-core data gradient: dX = (dY * act'(Y)) . W in column slices of <= 256, then views per source
            ldx = (K + 3) // 4 * 4                      # 16-byte aligned rows: the consumers of the column views load float4
            dX = torch.empty((M, ldx), device=W.device, dtype=torch.float32)
            kn = K if k_need is None else min(K, int(k_need))
            Wc = _f32c(W)
            narrow_ok = N in (128, 256) and dY.stride(0) % 4 == 0 and Y.stride(0) % 4 == 0 and dY.data_ptr() % 16 == 0 and Y.data_ptr() % 16 == 0
            for k0, (wpackT, Kpad, Np) in _packed_linear_T(W):
                if k0 >= kn:
                    continue
                kout = min(256, kn - k0)
                if kout <= 8 and narrow_ok:
                    # a slice of a few columns (the 7 extra inputs of block3): HBM-bound SIMT kernel, one read of dY / Y
                    with _launch(name=f"linear_bwd_data_narrow[{M}x{N}x{kout}]" if TIMERS is not None else None):
                        check(lib().hnr_linear_bwd_data_narrow(ptr(dY), dY.stride(0), ptr(Y), Y.stride(0), act, ptr(Wc), Wc.stride(0), k0, kout,
                                                               ptr(dX[:, k0:]), ldx, M, N, stream()), "linear_bwd_data_narrow")
                    continue
                with _launch(name=f"linear_tc_bwd_data[{M}x{N}x{K}]" if TIMERS is not None else None):
                    check(lib().hnr_linear_tc_bwd_data(ptr(dY), dY.stride(0), ptr(Y), Y.stride(0), act, ptr(wpackT), Kpad, Np,
                                                       ptr(dX[:, k0:]), ldx, M, N, kout, stream()), "linear_tc_bwd_data")
            outs, off = [], 0
            for i in range(nsrc):
                outs.append(dX[:, off:off + ks[i]] if need_src[i] else None)
                off += ks[i]
        else:
            outs = [torch.empty((M, ks[i]), device=W.device, dtype=torch.float32) if need_src[i] else None for i in range(nsrc)]
            outs_p = outs + [None] * (3 - nsrc)
            with _launch(name="linear_bwd_data"):
                check(lib().hnr_linear_bwd_data(ptr(dY), dY.stride(0), ptr(Y), Y.stride(0), ptr(W), ptr_array(outs_p),
                                                i64_array([o.stride(0) if o is not None else 0 for o in outs_p]), i64_array(ks), M, N, K, act,
                                                stream()), "linear_bwd_data")
        for i in range(nsrc):
            if outs[i] is not None and mods[i] > 0:
                outs[i] = outs[i].reshape(-1, mods[i], ks[i]).sum(dim=0)
            d_srcs[i] = outs[i]
    elif any(need_src):
        d_srcs = [torch.zeros_like(s) if n else None for s, n in zip(srcs, need_src)]
    dW = db = None
    if need_w:
        dW = torch.zeros_like(W)
        db = torch.zeros(N, device=W.device, dtype=torch.float32) if has_b else None
        if M > 0:
            if use_tc and (K + 1 + 31) // 32 * 32 <= 320:
                with _launch(name=f"linear_tc_bwd_weight[{M}x{N}x{K}]" if TIMERS is not None else None):
                    check(lib().hnr_linear_tc_bwd_weight(ptr(dY), dY.stride(0), ptr(Y), Y.stride(0), ptr_array(padded), i64_array(lds),
                                                         i64_array(ks), i64_array(mods), ptr(dW), ptr(db), M, N, K, act, stream()),
                          "linear_tc_bwd_weight")
            else:
                with _launch(name="linear_bwd_weight"):
                    check(lib().hnr_linear_bwd_weight(ptr(dY), dY.stride(0), ptr(Y), Y.stride(0), ptr_array(padded), i64_array(lds),
                                                      i64_array(ks), i64_array(mods), ptr(dW), ptr(db), M, N, K, act, stream()),
                          "linear_bwd_weight")
    return d_srcs, dW, db


def linear_head_backward(head_W: torch.Tensor, h: torch.Tensor, y: torch.Tensor, dH: torch.Tensor, act: int):
    """gradients of the one-output layer h = act(y . w + b): (dY (M,K), dW (1,K), db (1,)) in ONE pass over y (csrc/linear_simt.cu
    linear_head_bwd_kernel) when K is 64 or 128 and the rows are 16-byte aligned; the generic kernels otherwise."""
    y, dH, h = _rows2d(y), _f32c(dH), _f32c(h)
    M, K = y.shape
    w = _f32c(head_W).view(-1)
    if K in (64, 128) and y.stride(0) % 4 == 0 and y.data_ptr() % 16 == 0 and M > 0:
        dY = torch.empty((M, K), device=y.device, dtype=torch.float32)
        g = torch.zeros(K + 4, device=y.device, dtype=torch.float32)          # dW | db in one zero fill (16-byte aligned views)
        with _launch(name="linear_head_bwd"):
            check(lib().hnr_linear_head_bwd(ptr(dH), ptr(h), int(act), ptr(w), ptr(y), y.stride(0), M, K, ptr(dY), K, ptr(g), ptr(g[K:]),
                                            stream()), "linear_head_bwd")
        return dY, g[:K].view(1, K), g[K:K + 1]
    (dY,), dW, db = linear_backward(head_W, h, [y], (), dH, act, [True])
    return dY, dW, db


def linear_head(srcs: Sequence[torch.Tensor], W, b, act: int, head_W, head_b, head_act: int, mods: Sequence[int] = (),
                M: Optional[int] = None) -> torch.Tensor:
    """no-grad fusion of a dense layer with a following 1-output layer: head_act(act(cat(srcs) W^T + b) head_W^T + head_b)
    -> (M,1); the hidden layer's output never reaches memory (tensor-core epilogue).  Inference only."""
    assert not torch.is_grad_enabled() and LINEAR_ENGINE == "tc"
    srcs = [_rows2d(s) for s in srcs]
    if M is None:
        M = srcs[0].shape[0]
    W = _f32c(W)
    N, K = W.shape
    ks = [s.shape[1] for s in srcs] + [0] * (3 - len(srcs))
    assert sum(ks) == K and head_W.numel() == N
    require_cuda(W, *srcs)
    padded = list(srcs) + [None] * (3 - len(srcs))
    lds = [s.stride(0) if s is not None else 0 for s in padded]
    modl = list(mods) + [0] * (3 - len(mods))
    out = torch.empty((M, 1), device=W.device, dtype=torch.float32)
    wpack, Npad, Kp = _packed_linear(W)
    hw, hb, bc = _f32c(head_W).view(-1), _f32c(head_b).view(-1), _f32c(b)
    with _launch():
        check(lib().hnr_linear_tc_fwd(ptr_array(padded), i64_array(lds), i64_array(ks), i64_array(modl), ptr(wpack), Npad, Kp, ptr(bc), None, 0,
                                      None, N, M, N, K, act, ptr(hw), ptr(hb), head_act, ptr(out), stream()), "linear_tc_fwd(head)")
    return out


def linear(srcs: Sequence[torch.Tensor], W, b, act: int = ACT_NONE, res=None, mods: Sequence[int] = (), M: Optional[int] = None):
    if M is None:
        M = srcs[0].shape[0]
    mods = tuple(mods) if mods else tuple([0] * len(srcs))
    return LinearFn.apply(W, b, res, act, M, mods, *srcs)


# --------------------------------------------------------------------------------------------
# neighbour weights / features
# --------------------------------------------------------------------------------------------
class NbrWeightsFn(torch.autograd.Function):
    """-> weight (S,K) [no grad], conf_coefficient (S,K) [straight-through grad to conf], valid (S) u8."""

    @staticmethod
    def forward(ctx, xyz, conf, pidx, mask, loc_w):
        S, K = pidx.shape
        require_cuda(xyz, pidx, loc_w)
        weight = torch.empty((S, K), device=xyz.device, dtype=torch.float32)
        confc = torch.empty((S, K), device=xyz.device, dtype=torch.float32)
        valid = torch.empty((S,), device=xyz.device, dtype=torch.uint8)
        with _launch():
            check(lib().hnr_nbr_weights(ptr(xyz), ptr(conf), ptr(pidx), ptr(mask), ptr(loc_w), S, K, ptr(weight), ptr(confc), ptr(valid),
                                        stream()), "nbr_weights")
        ctx.save_for_backward(pidx)
        ctx.conf_shape = conf.shape if conf is not None else None
        ctx.mark_non_differentiable(weight, valid)
        return weight, confc, valid

    @staticmethod
    def backward(ctx, g_weight, g_confc, g_valid):
        (pidx,) = ctx.saved_tensors
        d_conf = None
        if ctx.needs_input_grad[1] and g_confc is not None:
            S, K = pidx.shape
            g = _f32c(g_confc)
            d_conf = torch.zeros(ctx.conf_shape, device=pidx.device, dtype=torch.float32)
            with _launch(name="conf_bwd"):
                check(lib().hnr_conf_bwd(None, None, None, ptr(pidx), ptr(g), 0, S, K, ptr(d_conf), stream()), "conf_bwd")
        return None, d_conf, None, None, None


class NbrFeaturesFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, emb, color, dirs, xyz, xyz_pers, pidx, mask, vlist, loc_w, loc_pers, raydirs, cam):
        Nv, K = vlist.shape[0], pidx.shape[1]
        require_cuda(emb, color, dirs, xyz, pidx, vlist)
        X0 = torch.empty((Nv * K, X0_W), device=emb.device, dtype=torch.float32)
        E = torch.empty((Nv * K, E_W), device=emb.device, dtype=torch.float32)
        with _launch():
            check(lib().hnr_nbr_features(ptr(xyz), ptr(xyz_pers), ptr(emb), ptr(color), ptr(dirs), ptr(pidx), ptr(vlist), ptr(loc_w),
                                         ptr(loc_pers), ptr(raydirs), ptr(cam), Nv, K, emb.shape[-1], ptr(X0), ptr(E), stream()), "nbr_features")
        ctx.cam, ctx.Nv, ctx.K = cam, Nv, K
        ctx.shapes = (emb.shape, color.shape, dirs.shape)
        ctx.save_for_backward(emb, pidx, mask if mask is not None else torch.empty(0, device=emb.device), vlist, raydirs)
        ctx.has_mask = mask is not None
        return X0, E

    @staticmethod
    def backward(ctx, dX0, dE):
        emb, pidx, mask, vlist, raydirs = ctx.saved_tensors
        dX0, dE = _f32c(dX0), _f32c(dE)
        ne, nc, nd = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        d_emb = torch.zeros(ctx.shapes[0], device=emb.device, dtype=torch.float32) if ne else None
        d_col = torch.zeros(ctx.shapes[1], device=emb.device, dtype=torch.float32) if nc else None
        d_dir = torch.zeros(ctx.shapes[2], device=emb.device, dtype=torch.float32) if nd else None
        if ne or nc or nd:
            with _launch(name="nbr_features_bwd"):
                check(lib().hnr_nbr_features_bwd(ptr(dX0), ptr(dE), ptr(emb), ptr(pidx), ptr(mask) if ctx.has_mask else None, ptr(vlist),
                                                 ptr(raydirs), ptr(ctx.cam), ctx.Nv, ctx.K, ptr(d_emb), ptr(d_col), ptr(d_dir), stream()),
                      "nbr_features_bwd")
        return d_emb, d_col, d_dir, None, None, None, None, None, None, None, None, None


class AlphaKSumFn(torch.autograd.Function):
    """H (Nv*K,256), weight (S,K), confc (S,K) -> sigma (Nv,1), X5 (Nv,280)."""

    @staticmethod
    def forward(ctx, H, confc, w_alpha, b_alpha, weight, vlist, raydirs, cam):
        Nv, K = vlist.shape[0], weight.shape[1]
        H = _f32c(H)
        w_alpha_c, b_alpha_c, confc_c = _f32c(w_alpha).view(-1), _f32c(b_alpha).view(-1), _f32c(confc)
        sigma = torch.empty((Nv, 1), device=H.device, dtype=torch.float32)
        X5 = torch.empty((Nv, X5_W), device=H.device, dtype=torch.float32)
        araw = torch.empty((Nv * K,), device=H.device, dtype=torch.float32)
        with _launch():
            check(lib().hnr_alpha_ksum_fwd(ptr(H), ptr(weight), ptr(confc_c), ptr(vlist), ptr(w_alpha_c), ptr(b_alpha_c), ptr(raydirs), ptr(cam),
                                           Nv, K, H.shape[1], ptr(sigma), ptr(X5), ptr(araw), stream()), "alpha_ksum_fwd")
        ctx.save_for_backward(H, confc_c, w_alpha_c, weight, vlist, araw)
        ctx.wshape, ctx.bshape = w_alpha.shape, b_alpha.shape
        return sigma, X5

    @staticmethod
    def backward(ctx, d_sigma, dX5):
        H, confc, w_alpha, weight, vlist, araw = ctx.saved_tensors
        Nv, K = vlist.shape[0], weight.shape[1]
        d_sigma, dX5 = _f32c(d_sigma), _f32c(dX5)
        dH = torch.empty_like(H)
        d_wc = torch.empty((Nv, K), device=H.device, dtype=torch.float32)
        d_wa = torch.zeros(HID, device=H.device, dtype=torch.float32)
        d_ba = torch.zeros(1, device=H.device, dtype=torch.float32)
        with _launch(name="alpha_ksum_bwd"):
            check(lib().hnr_alpha_ksum_bwd(ptr(H), ptr(weight), ptr(confc), ptr(vlist), ptr(w_alpha), ptr(araw), ptr(d_sigma), ptr(dX5), Nv, K,
                                           H.shape[1], ptr(dH), ptr(d_wc), ptr(d_wa), ptr(d_ba), stream()), "alpha_ksum_bwd")
        d_confc = None
        if ctx.needs_input_grad[1]:
            vl = vlist.long()
            d_confc = torch.zeros_like(confc)
            d_confc.index_copy_(0, vl, d_wc * weight.index_select(0, vl))
        return dH, d_confc, d_wa.view(ctx.wshape), d_ba.view(ctx.bshape), None, None, None, None


class NbrMlpFusedFn(torch.autograd.Function):
    """Training forward of the whole per-neighbour stage (gather, encodings, block1, block3, density head, weighted K-sum)
    through the fused tensor-core kernel (csrc/nbr_mlp_f16.cu) with the four layers' activations saved for the backward
    pass; the backward runs layer by layer on the tensor-core gradient kernels.  Same arithmetic and the same gradients as
    NbrFeaturesFn -> 4 x LinearFn -> AlphaKSumFn.  -> sigma (Nv,1), X5 (Nv,280)."""

    @staticmethod
    def forward(ctx, emb, color, dirs, confc, W1, b1, W2, b2, W3, b3, W4, b4, w_alpha, b_alpha, aux):
        from . import mlp_tc
        xyz, xyz_pers, pidx, vlist, loc_w, loc_pers, raydirs, cam, weight, pack = aux
        Nv, K = vlist.shape[0], pidx.shape[1]
        X0 = torch.empty((Nv * K, X0_W), device=emb.device, dtype=torch.float32)
        E = torch.empty((Nv * K, E_W), device=emb.device, dtype=torch.float32)
        with _launch():
            check(lib().hnr_nbr_features(ptr(xyz), ptr(xyz_pers), ptr(emb), ptr(color), ptr(dirs), ptr(pidx), ptr(vlist), ptr(loc_w),
                                         ptr(loc_pers), ptr(raydirs), ptr(cam), Nv, K, emb.shape[-1], ptr(X0), ptr(E), stream()), "nbr_features")
        confc_c = _f32c(confc)
        sigma, X5, H, araw = mlp_tc.forward_f16((xyz, xyz_pers, emb, color, dirs, None), pidx, vlist, loc_w, loc_pers, raydirs, cam, weight,
                                                confc_c, pack, w_alpha, b_alpha, debug=True)
        ctx.save_for_backward(emb, confc_c, W1, W2, W3, W4, _f32c(w_alpha).view(-1), X0, E, H, araw, pidx, vlist, raydirs, weight)
        ctx.cam, ctx.Nv, ctx.K = cam, Nv, K
        ctx.shapes = (emb.shape, color.shape, dirs.shape, w_alpha.shape, b_alpha.shape)
        return sigma, X5

    @staticmethod
    def backward(ctx, d_sigma, dX5):
        emb, confc, W1, W2, W3, W4, w_alpha, X0, E, H, araw, pidx, vlist, raydirs, weight = ctx.saved_tensors
        Nv, K = ctx.Nv, ctx.K
        d_sigma, dX5 = _f32c(d_sigma), _f32c(dX5)
        dH4 = torch.empty_like(H[3])
        d_wc = torch.empty((Nv, K), device=H.device, dtype=torch.float32)
        d_wa = torch.zeros(HID, device=H.device, dtype=torch.float32)
        d_ba = torch.zeros(1, device=H.device, dtype=torch.float32)
        with _launch(name="alpha_ksum_bwd"):
            check(lib().hnr_alpha_ksum_bwd(ptr(H[3]), ptr(weight), ptr(confc), ptr(vlist), ptr(w_alpha), ptr(araw), ptr(d_sigma), ptr(dX5), Nv, K,
                                           HID, ptr(dH4), ptr(d_wc), ptr(d_wa), ptr(d_ba), stream()), "alpha_ksum_bwd")
        d_confc = None
        if ctx.needs_input_grad[3]:
            vl = vlist.long()
            d_confc = torch.zeros_like(confc)
            d_confc.index_copy_(0, vl, d_wc * weight.index_select(0, vl))
        (dH3,), dW4, db4 = linear_backward(W4, H[3], [H[2]], (), dH4, ACT_LRELU, [True])
        (dH2, dE), dW3, db3 = linear_backward(W3, H[2], [H[1], E], (), dH3, ACT_LRELU, [True, True])
        (dH1,), dW2, db2 = linear_backward(W2, H[1], [H[0]], (), dH2, ACT_LRELU, [True])
        # of layer 0's 284 inputs only [emb 32 | PE(emb) 192] carry a gradient (the 60 distance encodings depend on positions,
        # xyz_grad = 0; nbr_features_bwd reads columns < 224 only): one 224-column slice instead of 256 + 28
        (dX0,), dW1, db1 = linear_backward(W1, H[0], [X0], (), dH1, ACT_LRELU, [True], k_need=X0_GRAD_W)
        ne, nc, nd = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        d_emb = torch.zeros(ctx.shapes[0], device=emb.device, dtype=torch.float32) if ne else None
        d_col = torch.zeros(ctx.shapes[1], device=emb.device, dtype=torch.float32) if nc else None
        d_dir = torch.zeros(ctx.shapes[2], device=emb.device, dtype=torch.float32) if nd else None
        if ne or nc or nd:
            dX0c, dEc = _f32c(dX0), _f32c(dE)
            with _launch(name="nbr_features_bwd"):
                check(lib().hnr_nbr_features_bwd(ptr(dX0c), ptr(dEc), ptr(emb), ptr(pidx), None, ptr(vlist), ptr(raydirs), ptr(ctx.cam), Nv, K,
                                                 ptr(d_emb), ptr(d_col), ptr(d_dir), stream()), "nbr_features_bwd")
        return (d_emb, d_col, d_dir, d_confc, dW1, db1, dW2, db2, dW3, db3, dW4, db4, d_wa.view(ctx.shapes[3]), d_ba.view(ctx.shapes[4]), None)


# Deferred gradient tails.  The weight-gradient launches (wgrad_img: ~1.4 ms per step) and the tail of the image branch
# (image_gather_bwd -> pyramid_bwd: ~1.1 ms) depend on nothing that follows them in the backward pass and nothing in the backward pass
# depends on them: they only produce parameter gradients.  Inside `with defer_weight_gradients() as d:` the backward functions hand
# autograd their (zeroed) gradient buffers at once and park the launch in `d`; the training loop runs `d.run()` after loss.backward()
# returned -- a data-parallel loop first starts the all-reduce of the point tables, so that the collective overlaps with these kernels
# instead of being exposed (parallel.train_step).  Jobs of lane 1 (the image-branch tail: small grids, latency / atomics bound) are
# issued on a side stream and run CONCURRENTLY with lane 0 (wgrad_img: HBM bound, 192-thread CTAs with few registers).
_DEFER = None
_SIDE = {}
SIDE_LANE = True        # False: the image-branch tail runs on the main stream behind the weight gradients (clean per-kernel timings)


def side_stream(dev) -> "torch.cuda.Stream":
    key = torch.device(dev).index or 0
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=dev)
    return _SIDE[key]


class defer_weight_gradients:
    def __init__(self, side: bool = True):
        self.jobs = []          # (launch closure, [(parameter, gradient buffer)], lane)
        self.side = side and SIDE_LANE and os.environ.get("HNR_SIDE_STREAM", "1") != "0"

    def __enter__(self):
        global _DEFER
        self._prev, _DEFER = _DEFER, self
        return self

    def __exit__(self, *a):
        global _DEFER
        _DEFER = self._prev

    def run(self):
        lane1 = [j for j in self.jobs if j[2] == 1]
        lane0 = [j for j in self.jobs if j[2] == 0]
        main = torch.cuda.current_stream()
        side = None
        if lane1 and self.side and lane0:
            side = side_stream(main.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                for fn, _, _ in lane1:
                    fn()
        else:
            lane0 = self.jobs
        for fn, _, _ in lane0:
            fn()
        if side is not None:
            # every buffer the side lane touched was allocated on `main` and is still referenced by self.jobs here: nothing can be
            # recycled before the join below
            main.wait_stream(side)
        for _, pairs, _ in self.jobs:
            for p, buf in pairs:
                # autograd normally adopts the returned buffer as p.grad (same storage: nothing to do); if it cloned it instead (the clone
                # was taken before the launch above filled the buffer), add the result to the clone
                if p.grad is not None and p.grad.data_ptr() != buf.data_ptr():
                    p.grad.add_(buf.view_as(p.grad))
        self.jobs = []


def alias(t: torch.Tensor) -> torch.Tensor:
    """another tensor object on the same memory, NOT a view of `t`: a parked launch must not keep the gradient tensor itself alive, or
    autograd (which adopts a returned gradient as p.grad only when nobody else references it) would clone it before it is filled"""
    return torch.empty(0, dtype=t.dtype, device=t.device).set_(t.untyped_storage(), t.storage_offset(), t.size(), t.stride())


def _wgrad_launch(fn, pairs, lane: int = 0):
    if _DEFER is not None:
        _DEFER.jobs.append((fn, pairs, lane))
    else:
        fn()


class NbrMlpTrainFn(torch.autograd.Function):
    """Fully fused training path of the per-neighbour stage (round 2).  Forward: nbr_mlp_f16 in save mode -- the layer-0 input,
    the block3 extras and the four layers' outputs go to HBM as split bf16 images (csrc/img_common.cuh).  Backward: three
    launches instead of 4 x (data gradient + weight gradient): density-head / K-sum backward writing the gated gradient image
    dZ_3, the fused data-gradient chain (csrc/nbr_bwd_f16.cu: dZ_3 -> dZ_2 -> dZ_1 -> dZ_0 -> dX0, gradient tile resident on the
    SM), and ONE weight-gradient launch for all four layers that bulk-copies the images as MN-major UMMA operands
    (csrc/wgrad_img.cu).  Same gradients as NbrMlpFusedFn (autograd over point_aggregators.py:921-1026 of the reference).
    -> sigma (Nv,1), X5 (Nv,280)."""

    @staticmethod
    def forward(ctx, emb, color, dirs, confc, W1, b1, W2, b2, W3, b3, W4, b4, w_alpha, b_alpha, aux):
        from . import mlp_tc
        xyz, xyz_pers, pidx, vlist, loc_w, loc_pers, raydirs, cam, weight, pack, packT = aux
        Nv, K = vlist.shape[0], pidx.shape[1]
        confc_c = _f32c(confc)
        sigma, X5, imgs, araw = mlp_tc.forward_f16_train((xyz, xyz_pers, emb, color, dirs, None), pidx, vlist, loc_w, loc_pers, raydirs, cam,
                                                         weight, confc_c, pack, w_alpha, b_alpha)
        ctx.save_for_backward(emb, confc_c, W3, _f32c(w_alpha).view(-1), araw, pidx, vlist, raydirs, weight, packT, imgs["x0"], imgs["e"],
                              imgs["h0"], imgs["h1"], imgs["h2"], imgs["h3"])
        ctx.wparams = (W1, b1, W2, b2, W3, b3, W4, b4)
        ctx.cam, ctx.Nv, ctx.K = cam, Nv, K
        ctx.shapes = (emb.shape, color.shape, dirs.shape, w_alpha.shape, b_alpha.shape)
        return sigma, X5

    @staticmethod
    def backward(ctx, d_sigma, dX5):
        from . import mlp_tc
        emb, confc, W3, w_alpha, araw, pidx, vlist, raydirs, weight, packT, x0img, eimg, h0, h1, h2, h3 = ctx.saved_tensors
        Nv, K = ctx.Nv, ctx.K
        rows = Nv * K
        dev = emb.device
        d_sigma, dX5 = _f32c(d_sigma), _f32c(dX5)
        dz = [mlp_tc.image_empty(rows, HID, dev) for _ in range(4)]                 # dZ_0 .. dZ_3
        d_wc = torch.empty((Nv, K), device=dev, dtype=torch.float32)
        # ONE zero fill for every small gradient of this stage: d_walpha | d_balpha | dW1, db1, ... dW4, db4 (parameter-shaped views; the
        # weight-gradient kernel accumulates straight into them through its column maps)
        shapes = [(HID, X0_W), (HID,), (HID, HID), (HID,), (HID, HID + E_W), (HID,), (HID, HID), (HID,)]
        sizes = [HID, 1] + [int(torch.Size(sh).numel()) for sh in shapes]
        pad4 = lambda n_: (n_ + 3) // 4 * 4                       # 16-byte aligned views: the fused Adam takes its vector path
        small = torch.zeros(sum(pad4(n_) for n_ in sizes), device=dev, dtype=torch.float32)
        views, o = [], 0
        for n_ in sizes:
            views.append(small[o:o + n_]); o += pad4(n_)
        d_wa, d_ba = views[0], views[1]
        gW = [views[2 + i].view(shapes[i]) for i in range(8)]
        # the gradient of conf_coefficient (S,K) is written by the same kernel at the valid samples' rows (was: long + gather + mul + index_copy)
        d_confc = torch.zeros_like(confc) if ctx.needs_input_grad[3] else None
        with _launch(name="alpha_ksum_bwd"):
            check(lib().hnr_alpha_ksum_bwd_img(ptr(h3), ptr(weight), ptr(confc), ptr(vlist), ptr(w_alpha), ptr(araw), ptr(d_sigma), ptr(dX5),
                                               Nv, K, ptr(dz[3]), ptr(d_wc), ptr(d_wa), ptr(d_ba), ptr(d_confc), stream()), "alpha_ksum_bwd_img")
        dX0 = torch.empty((rows, X0_GRAD_W), device=dev, dtype=torch.float32)
        with _launch(name="nbr_bwd_chain"):
            check(lib().hnr_nbr_bwd_f16(ptr(dz[3]), ptr(h2), ptr(h1), ptr(h0), ptr(dz[2]), ptr(dz[1]), ptr(dz[0]), ptr(dX0), X0_GRAD_W,
                                        X0_GRAD_W, ptr(packT), rows, stream()), "nbr_bwd_f16")
        dE = torch.empty((rows, E_W), device=dev, dtype=torch.float32)
        W3c = _f32c(W3)
        with _launch(name="dz_extras_bwd"):
            check(lib().hnr_dz_extras_bwd(ptr(dz[2]), ptr(W3c), W3c.stride(0), HID, rows, ptr(dE), stream()), "dz_extras_bwd")
        x0map, e3map = _wgrad_colmaps(dev)
        rows_pad = mlp_tc.rows_padded(rows)
        ga = [alias(t) for t in gW]             # the parked launch refers to aliases only (see alias())

        def launch_wgrad():
            with _launch(name="wgrad_img"):
                check(lib().hnr_wgrad_img_jobs(4, ptr_array(dz), i64_array([HID] * 4), ptr_array([x0img, h0, h1, h2]), ptr_array([None, None, eimg, None]),
                                               i64_array([mlp_tc.X0_IMG_W, HID, HID, HID]), i64_array([0, 0, mlp_tc.E_IMG_W, 0]),
                                               ptr_array([ga[0], ga[2], ga[4], ga[6]]), ptr_array([ga[1], ga[3], ga[5], ga[7]]),
                                               ptr_array([x0map, None, e3map, None]), i64_array([HID] * 4), i64_array([X0_W, HID, HID + E_W, HID]),
                                               i64_array([rows_pad] * 4), stream()), "wgrad_img_jobs")
        _wgrad_launch(launch_wgrad, list(zip(ctx.wparams, ga)))
        dW1, db1, dW2, db2, dW3, db3, dW4, db4 = gW
        ne, nc, nd = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        d_emb = torch.zeros(ctx.shapes[0], device=dev, dtype=torch.float32) if ne else None
        d_col = torch.zeros(ctx.shapes[1], device=dev, dtype=torch.float32) if nc else None
        d_dir = torch.zeros(ctx.shapes[2], device=dev, dtype=torch.float32) if nd else None
        if ne or nc or nd:
            with _launch(name="nbr_features_bwd"):
                check(lib().hnr_nbr_features_bwd_ld(ptr(dX0), X0_GRAD_W, ptr(dE), ptr(emb), ptr(pidx), None, ptr(vlist), ptr(raydirs),
                                                    ptr(ctx.cam), Nv, K, ptr(d_emb), ptr(d_col), ptr(d_dir), stream()), "nbr_features_bwd_ld")
        return (d_emb, d_col, d_dir, d_confc, dW1, db1, dW2, db2, dW3, db3, dW4, db4, d_wa.view(ctx.shapes[3]), d_ba.view(ctx.shapes[4]), None)


_WG_MAPS = {}


def _wgrad_colmaps(dev):
    """device int32 column maps of hnr_wgrad_img_jobs for the per-neighbour MLP, cached per device: layer 0 (288 kernel-order
    columns -> reference column of the 284-wide block1 input, -1 = padding) and layer 2 ([H_1 256 | extras 16] -> 263 columns)"""
    key = str(dev)
    if key not in _WG_MAPS:
        from . import mlp_tc
        _WG_MAPS[key] = (torch.tensor(mlp_tc.layer1_column_order_f16(), device=dev, dtype=torch.int32),
                         torch.tensor(list(range(HID + E_W)) + [-1] * (mlp_tc.E_IMG_W - E_W), device=dev, dtype=torch.int32))
    return _WG_MAPS[key]


_X0_COLS = {}


def _x0_cols(dev):
    """(reference column, kernel-order column) of every real column of the layer-0 input, cached per device (index tensors, not a
    boolean mask: mask indexing reads its count back from the device, i.e. a host synchronisation in the middle of backward)"""
    key = str(dev)
    if key not in _X0_COLS:
        from . import mlp_tc
        cols = mlp_tc.layer1_column_order_f16()
        _X0_COLS[key] = (torch.tensor([c for c in cols if c >= 0], device=dev, dtype=torch.long),
                         torch.tensor([k for k, c in enumerate(cols) if c >= 0], device=dev, dtype=torch.long))
    return _X0_COLS[key]


# --------------------------------------------------------------------------------------------
# image branch
# --------------------------------------------------------------------------------------------
TRAIN_LOSS_PARTIALS = 512        # HNR_TRAIN_LOSS_PARTIALS (include/hnr.h): scratch doubles of hnr_train_loss


class TrainLossFn(torch.autograd.Function):
    """training loss of the hot path (csrc/loss.cu): masked MSE (+1e-6) x frame_weight + zero-one regulariser on conf_coefficient;
    the gradients are computed by the same launch and only scaled in backward.  A second one-warp launch adds the block partials in a
    fixed order, so the value is the same in every run."""

    @staticmethod
    def forward(ctx, color, confc, gt, ray_ids, frame_weight: float, zero_one_weight: float):
        color = _f32c(color)
        gt2 = _f32c(gt).reshape(-1, 3)
        n_rays = color.numel() // 3
        cc = _f32c(confc) if confc is not None else None
        dev = color.device
        loss = torch.empty((), device=dev, dtype=torch.float32)
        partials = torch.empty(TRAIN_LOSS_PARTIALS, device=dev, dtype=torch.float64)
        d_color = torch.empty_like(color)
        d_cc = torch.empty_like(cc) if cc is not None else None
        with _launch(2, name="train_loss"):
            check(lib().hnr_train_loss(ptr(color), ptr(gt2), ptr(ray_ids), n_rays, ptr(cc), cc.numel() if cc is not None else 0, float(frame_weight),
                                       float(zero_one_weight), ptr(loss), ptr(partials), ptr(d_color), ptr(d_cc), stream()), "train_loss")
        ctx.save_for_backward(d_color, d_cc if d_cc is not None else torch.empty(0, device=dev))
        ctx.has_cc = cc is not None
        return loss

    @staticmethod
    def backward(ctx, g):
        d_color, d_cc = ctx.saved_tensors
        return d_color * g, (d_cc * g if ctx.has_cc else None), None, None, None, None


class PyramidFn(torch.autograd.Function):
    """feature pyramid of the image branch (csrc/pyramid.cu): img (V,H,W,3) NHWC + the 12 conv parameters of aux_block_s1/s2/s3 ->
    levels (V,H/2,W/2,6), (V,H/4,W/4,12), (V,H/8,W/8,24) NHWC.  Exact fp32, forward and backward on own kernels (no cuDNN, no
    layout conversions).  No gradient flows to the images."""

    @staticmethod
    def forward(ctx, img, *params):
        img = _f32c(img)
        require_cuda(img, *params)
        V, H, W, _ = img.shape
        ws = [_f32c(p) for p in params[0::2]]
        bs = [_f32c(p) for p in params[1::2]]
        d = lambda x: (x - 1) // 2 + 1
        hs, wd = [d(H)], [d(W)]
        for _ in range(2):
            hs.append(d(hs[-1])); wd.append(d(wd[-1]))
        chans = (6, 6, 12, 12, 24, 24)
        act = [torch.empty((V, hs[i // 2], wd[i // 2], chans[i]), device=img.device, dtype=torch.float32) for i in range(6)]
        with _launch(6, name="pyramid_fwd"):
            check(lib().hnr_pyramid_fwd(ptr(img), ptr_array(ws), ptr_array(bs), ptr_array(act), V, H, W, stream()), "pyramid_fwd")
        ctx.save_for_backward(img, *ws, *act)
        ctx.wparams = list(params)
        ctx.mark_non_differentiable(act[0], act[2], act[4])
        return act[1], act[3], act[5]

    @staticmethod
    def backward(ctx, d1, d2, d3):
        sv = ctx.saved_tensors
        img, ws, act = sv[0], list(sv[1:7]), list(sv[7:13])
        V, H, W, _ = img.shape
        dev = img.device
        flat = torch.zeros(sum(w.numel() + w.shape[0] for w in ws), device=dev, dtype=torch.float32)       # one fill for all 12 gradients
        dws, dbs, o = [], [], 0
        for w in ws:
            dws.append(flat[o:o + w.numel()].view_as(w)); o += w.numel()
            dbs.append(flat[o:o + w.shape[0]]); o += w.shape[0]
        scratch = [torch.empty_like(act[i]) for i in (4, 3, 2, 1, 0)]
        c = lambda t: _f32c(t) if t is not None else None
        if d3 is None:
            d3 = torch.zeros_like(act[5])
        ds = [c(d1), c(d2), c(d3)]
        aw, ab = [alias(t) for t in dws], [alias(t) for t in dbs]          # the parked launch refers to aliases only (see alias())

        def launch():
            with _launch(11, name="pyramid_bwd"):
                check(lib().hnr_pyramid_bwd(ptr(img), ptr_array(ws), ptr_array(act), ptr_array(ds), ptr_array(aw), ptr_array(ab),
                                            ptr_array(scratch), V, H, W, stream()), "pyramid_bwd")
        pairs = []
        for i in range(6):
            pairs += [(ctx.wparams[2 * i], aw[i]), (ctx.wparams[2 * i + 1], ab[i])]
        _wgrad_launch(launch, pairs, lane=1)
        del flat
        grads = []
        for dw, db in zip(dws, dbs):
            grads += [dw, db]
        return (None, *grads)


def project_views(loc_w: torch.Tensor, w2c: torch.Tensor, Kmat: torch.Tensor, campos: torch.Tensor, campos_n: torch.Tensor):
    """loc_w (S,3), w2c (V,4,4), Kmat (3,3), campos (3,), campos_n (V,3) -> xy (V,S,2), delta (V,S,3)."""
    S, V = loc_w.shape[0], w2c.shape[0]
    loc_w, w2c, Kmat, campos, campos_n = map(_f32c, (loc_w, w2c, Kmat, campos, campos_n))
    require_cuda(loc_w, w2c, Kmat, campos, campos_n)
    xy = torch.empty((V, S, 2), device=loc_w.device, dtype=torch.float32)
    delta = torch.empty((V, S, 3), device=loc_w.device, dtype=torch.float32)
    with _launch():
        check(lib().hnr_project_views(ptr(loc_w), ptr(w2c), ptr(Kmat), ptr(campos), ptr(campos_n), V, S, ptr(xy), ptr(delta), stream()),
              "project_views")
    return xy, delta


class ImageGatherFn(torch.autograd.Function):
    """levels NHWC (V,H,W,3),(V,h1,w1,6),(V,h2,w2,12),(V,h3,w3,24); xy (V,S,2) -> aux (V,Nv,45), ok (V,Nv).
    With `delta` (V,S,3): 48-wide rows [aux 45 | dview 3] (16-byte aligned: the blend-weight chain reads them with vector loads);
    the incoming gradient then has 48-wide rows too, of which columns 45..47 (the view-direction difference: data) are ignored."""

    @staticmethod
    def forward(ctx, l0, l1, l2, l3, xy, vlist, delta=None):
        lv = [_f32c(l) for l in (l0, l1, l2, l3)]
        require_cuda(*lv, xy, vlist)
        V, S, Nv = xy.shape[0], xy.shape[1], vlist.shape[0]
        hw = []
        for l in lv:
            hw += [l.shape[1], l.shape[2]]
        ld = AUX_C if delta is None else AUX_LD
        aux = torch.empty((V, Nv, ld), device=xy.device, dtype=torch.float32)
        ok = torch.empty((V, Nv), device=xy.device, dtype=torch.float32)
        d = _f32c(delta.reshape(V, S, 3)) if delta is not None else None
        with _launch():
            check(lib().hnr_image_gather_fwd(ptr_array(lv), i64_array(hw), ptr(xy), ptr(vlist), V, S, Nv, ptr(aux), ptr(ok), ld, ptr(d),
                                             stream()), "image_gather_fwd")
        ctx.hw, ctx.shapes, ctx.dims, ctx.ld = hw, [l.shape for l in lv], (V, S, Nv), ld
        ctx.save_for_backward(xy, vlist)
        ctx.mark_non_differentiable(ok)
        return aux, ok

    @staticmethod
    def backward(ctx, d_aux, d_ok):
        xy, vlist = ctx.saved_tensors
        V, S, Nv = ctx.dims
        grads = [None] + [torch.zeros(s, device=xy.device, dtype=torch.float32) for s in ctx.shapes[1:]]
        d_aux = _f32c(d_aux)
        hw, ld = ctx.hw, ctx.ld

        def launch():
            with _launch(name="image_gather_bwd"):
                check(lib().hnr_image_gather_bwd_ld(ptr_array(grads), i64_array(hw), ptr(xy), ptr(vlist), ptr(d_aux), ld, V, S, Nv, stream()),
                      "image_gather_bwd")
        # the pyramid gradients feed pyramid_bwd only, which is parked behind this launch on the same lane (in order)
        _wgrad_launch(launch, [], lane=1)
        return None, grads[1], grads[2], grads[3], None, None, None


AUX_LD = 48        # 16-byte aligned row stride of the no-grad image-branch tensors: [aux 45 | dview 3] and [merged 45 | 0 0 0]


def image_gather_padded(levels, xy, vlist, delta):
    """no-grad lookup into 48-wide rows with the view-direction difference in columns 45..47: the blend-weight net reads
    [aux | dview] as one aligned block.  -> aux48 (V,Nv,48), ok (V,Nv)"""
    lv = [_f32c(l) for l in levels]
    V, S, Nv = xy.shape[0], xy.shape[1], vlist.shape[0]
    hw = []
    for l in lv:
        hw += [l.shape[1], l.shape[2]]
    aux = torch.empty((V, Nv, AUX_LD), device=xy.device, dtype=torch.float32)
    ok = torch.empty((V, Nv), device=xy.device, dtype=torch.float32)
    d = _f32c(delta.reshape(V, S, 3))
    with _launch():
        check(lib().hnr_image_gather_fwd(ptr_array(lv), i64_array(hw), ptr(xy), ptr(vlist), V, S, Nv, ptr(aux), ptr(ok), AUX_LD, ptr(d),
                                         stream()), "image_gather_fwd")
    return aux, ok


def blend_padded(aux48, sig, ok, keep):
    """no-grad blend of 48-wide aux rows -> merged (Nv,48) with zero padding"""
    V, Nv = aux48.shape[0], aux48.shape[1]
    merged = torch.empty((Nv, AUX_LD), device=aux48.device, dtype=torch.float32)
    with _launch():
        check(lib().hnr_blend_fwd(ptr(aux48), ptr(_f32c(sig)), ptr(ok), ptr(keep), V, Nv, AUX_LD, ptr(merged), AUX_LD, stream()), "blend_fwd")
    return merged


class BlendFn(torch.autograd.Function):
    """aux (V,Nv,45 | 48), sig (V*Nv,1), ok (V,Nv), keep (Nv) u8|None -> merged (Nv,45)."""

    @staticmethod
    def forward(ctx, aux, sig, ok, keep):
        aux, sig = _f32c(aux), _f32c(sig)
        V, Nv, ld = aux.shape[0], aux.shape[1], aux.shape[2]
        merged = torch.empty((Nv, AUX_C), device=aux.device, dtype=torch.float32)
        with _launch():
            check(lib().hnr_blend_fwd(ptr(aux), ptr(sig), ptr(ok), ptr(keep), V, Nv, ld, ptr(merged), AUX_C, stream()), "blend_fwd")
        ctx.save_for_backward(aux, sig, ok, keep if keep is not None else torch.empty(0, device=aux.device))
        ctx.has_keep = keep is not None
        return merged

    @staticmethod
    def backward(ctx, d_merged):
        aux, sig, ok, keep = ctx.saved_tensors
        V, Nv, ld = aux.shape[0], aux.shape[1], aux.shape[2]
        d_aux = torch.empty_like(aux)
        d_sig = torch.empty_like(sig)
        with _launch(name="blend_bwd"):
            check(lib().hnr_blend_bwd_ld(ptr(aux), ld, ptr(sig), ptr(ok), ptr(keep) if ctx.has_keep else None, ptr(_f32c(d_merged)), V, Nv,
                                         ptr(d_aux), ld, ptr(d_sig), stream()), "blend_bwd")
        return d_aux, d_sig, None, None


class ScatterRowsFn(torch.autograd.Function):
    """out (S,C) = zeros; out[idx] = src (Nv,C): the decoded [sigma | rgb] rows of the valid samples scattered back to all sample
    slots.  Same result as zeros.index_copy(0, idx, src); its backward is an element-wise torch.gather instead of index_select's (and
    grad[idx]'s) one-block-per-row gather kernel (42 us for 75 k rows of 4 floats)."""

    @staticmethod
    def forward(ctx, src, idx, S: int):
        out = torch.zeros((S, src.shape[1]), device=src.device, dtype=src.dtype)
        out.index_copy_(0, idx, src)
        ctx.save_for_backward(idx)
        return out

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        return torch.gather(g, 0, idx.unsqueeze(1).expand(-1, g.shape[1])), None, None


# --------------------------------------------------------------------------------------------
# compositing
# --------------------------------------------------------------------------------------------
class CompositeFn(torch.autograd.Function):
    """feats (R,SR,4); valid (R,SR) u8; either z (R,SR) view with element stride (camera depth) or
    dist (R,SR).  -> ray_color (R,3), opacity, acc_transmission, blend_weight (R,SR), bg_T (R), dist."""

    @staticmethod
    def forward(ctx, feats, valid, z, z_stride: int, dist, bg, vsize_z: float, unit_mode: int):
        feats = _f32c(feats)
        R, SR = feats.shape[0], feats.shape[1]
        require_cuda(feats, valid)
        dev = feats.device
        color = torch.empty((R, 3), device=dev, dtype=torch.float32)
        opacity = torch.empty((R, SR), device=dev, dtype=torch.float32)
        accT = torch.empty((R, SR), device=dev, dtype=torch.float32)
        bw = torch.empty((R, SR), device=dev, dtype=torch.float32)
        bgT = torch.empty((R,), device=dev, dtype=torch.float32)
        dist_out = torch.empty((R, SR), device=dev, dtype=torch.float32)
        bgc = _f32c(bg).view(-1) if bg is not None else None
        with _launch():
            check(lib().hnr_composite_fwd(ptr(feats), ptr(valid), ptr(z), z_stride, ptr(dist), ptr(bgc), float(vsize_z), int(unit_mode), R, SR,
                                          ptr(color), ptr(opacity), ptr(accT), ptr(bw), ptr(bgT), ptr(dist_out), stream()), "composite_fwd")
        ctx.save_for_backward(feats, valid, dist_out, accT, bgT, bgc if bgc is not None else torch.empty(0, device=dev))
        ctx.has_bg = bgc is not None
        ctx.mark_non_differentiable(dist_out)
        return color, opacity, accT, bw, bgT, dist_out

    @staticmethod
    def backward(ctx, g_color, g_opacity, g_accT, g_bw, g_bgT, g_dist):
        feats, valid, dist, accT, bgT, bg = ctx.saved_tensors
        R, SR = feats.shape[0], feats.shape[1]
        g_feats = torch.empty_like(feats)
        c = lambda t: _f32c(t) if t is not None else None
        gc = c(g_color) if g_color is not None else torch.zeros((R, 3), device=feats.device)
        with _launch(name="composite_bwd"):
            check(lib().hnr_composite_bwd(ptr(feats), ptr(valid), ptr(dist), ptr(accT), ptr(bgT), ptr(bg) if ctx.has_bg else None, ptr(gc),
                                          ptr(c(g_opacity)), ptr(c(g_bgT)), ptr(c(g_bw)), ptr(c(g_accT)), R, SR, ptr(g_feats), stream()),
                  "composite_bwd")
        return g_feats, None, None, None, None, None, None, None


# --------------------------------------------------------------------------------------------
# blur
# --------------------------------------------------------------------------------------------
# The blur kernels index the raster from patch_num and patch_size alone, so a tensor of the wrong shape would be read and
# written out of bounds: the shapes are checked on the host before anything is launched.
def _check_raster(name: str, t: torch.Tensor, patch_num: int, patch_size: int) -> None:
    rows = (patch_num * patch_size) ** 2
    if t.dim() != 2 or t.shape[0] != rows or t.shape[1] != 3:
        raise ValueError(f"blur: {name} must be ((patch_num*patch_size)^2, 3) = ({rows}, 3) for patch_num {patch_num}, "
                         f"patch_size {patch_size}; got {tuple(t.shape)}")


def _check_kernel_bank(kernels: torch.Tensor) -> None:
    if kernels.dim() != 3 or kernels.shape[1] != kernels.shape[2] or kernels.shape[1] % 2 == 0:
        raise ValueError(f"blur: kernels must be (Nk, k, k) with k odd; got {tuple(kernels.shape)}")


def _check_raw(raw: torch.Tensor, patch_num: int) -> None:
    if raw.dim() != 2 or raw.shape[0] != patch_num * patch_num:
        raise ValueError(f"blur: raw predictor output must have patch_num^2 = {patch_num * patch_num} rows; got {tuple(raw.shape)}")


class BlurSelectFn(torch.autograd.Function):
    """pred, gt (S*S,3) on the patch raster; kernels (Nk,ks,ks) -> best candidate per patch."""

    @staticmethod
    def forward(ctx, pred, gt, kernels, patch_num: int, patch_size: int):
        _check_raster("pred", pred, patch_num, patch_size)
        _check_raster("gt", gt, patch_num, patch_size)
        _check_kernel_bank(kernels)
        pred, gt, kernels = _f32c(pred), _f32c(gt), _f32c(kernels)
        require_cuda(pred, gt, kernels)
        Nk, ks = kernels.shape[0], kernels.shape[1]
        out = torch.empty_like(pred)
        sel = torch.empty((patch_num * patch_num,), device=pred.device, dtype=torch.int32)
        with _launch(name="blur_select_fwd"):
            check(lib().hnr_blur_select_fwd(ptr(pred), ptr(gt), ptr(kernels), patch_num, patch_size, Nk, ks, ptr(out), ptr(sel), stream()),
                  "blur_select_fwd")
        ctx.save_for_backward(kernels, sel)
        ctx.geom = (patch_num, patch_size, Nk, ks)
        ctx.mark_non_differentiable(sel)
        return out, sel

    @staticmethod
    def backward(ctx, g_out, g_sel):
        kernels, sel = ctx.saved_tensors
        pn, ps, Nk, ks = ctx.geom
        g_out = _f32c(g_out)
        g_pred = torch.empty_like(g_out)
        with _launch(name="blur_select_bwd"):
            check(lib().hnr_blur_select_bwd(ptr(g_out), ptr(kernels), ptr(sel), pn, ps, Nk, ks, ptr(g_pred), stream()), "blur_select_bwd")
        return g_pred, None, None, None, None


class BlurGrayFn(torch.autograd.Function):
    """pred, gt (S*S,3) on the patch raster -> predictor input rows (N, 2*ps*ps) = [mean_c gt | mean_c pred]
    (base_rendering_model.py:887-889); gradient to pred only."""

    @staticmethod
    def forward(ctx, pred, gt, patch_num: int, patch_size: int):
        _check_raster("pred", pred, patch_num, patch_size)
        _check_raster("gt", gt, patch_num, patch_size)
        pred, gt = _f32c(pred), _f32c(gt)
        require_cuda(pred, gt)
        feat = torch.empty((patch_num * patch_num, 2 * patch_size * patch_size), device=pred.device, dtype=torch.float32)
        with _launch(name="blur_gray_fwd"):
            check(lib().hnr_blur_gray_fwd(ptr(pred), ptr(gt), patch_num, patch_size, ptr(feat), stream()), "blur_gray_fwd")
        ctx.geom = (patch_num, patch_size, tuple(pred.shape))
        return feat

    @staticmethod
    def backward(ctx, g_feat):
        pn, ps, shape = ctx.geom
        g_feat = _f32c(g_feat)
        g_pred = torch.empty(shape, device=g_feat.device, dtype=torch.float32)
        with _launch(name="blur_gray_bwd"):
            check(lib().hnr_blur_gray_bwd(ptr(g_feat), pn, ps, ptr(g_pred), stream()), "blur_gray_bwd")
        return g_pred, None, None, None


class BlurLearnFn(torch.autograd.Function):
    """pred (S*S,3) on the patch raster, raw (N, ks*ks [+1]) predictor outputs -> blurred pred (S*S,3)
    (base_rendering_model.py:893-1005); gradients to pred and raw."""

    @staticmethod
    def forward(ctx, pred, raw, patch_num: int, patch_size: int, kernel_size: int, norm_mode: int, mix_mode: int, boundary_mode: int):
        _check_raster("pred", pred, patch_num, patch_size)
        _check_raw(raw, patch_num)
        pred, raw = _f32c(pred), _f32c(raw)
        require_cuda(pred, raw)
        out = torch.empty_like(pred)
        with _launch(name="blur_learn_fwd"):
            check(lib().hnr_blur_learn_fwd(ptr(pred), ptr(raw), raw.shape[1], patch_num, patch_size, kernel_size, norm_mode, mix_mode,
                                           boundary_mode, ptr(out), stream()), "blur_learn_fwd")
        ctx.save_for_backward(pred, raw)
        ctx.geom = (patch_num, patch_size, kernel_size, norm_mode, mix_mode, boundary_mode)
        return out

    @staticmethod
    def backward(ctx, g_out):
        pred, raw = ctx.saved_tensors
        pn, ps, ks, nm, mm, bm = ctx.geom
        g_out = _f32c(g_out)
        g_pred = torch.empty_like(pred)
        g_raw = torch.zeros_like(raw)
        with _launch(name="blur_learn_bwd"):
            check(lib().hnr_blur_learn_bwd(ptr(pred), ptr(raw), raw.shape[1], ptr(g_out), pn, ps, ks, nm, mm, bm, ptr(g_pred), ptr(g_raw),
                                           stream()), "blur_learn_bwd")
        return g_pred, g_raw, None, None, None, None, None, None
