"""Thin Python wrappers over the libfdx C-ABI (one function per entry point).

Tensors are NHWC bf16 activations / HWIO conv kernels exactly as the reference's flax
modules store them (flaxdiff/models/common.py:166-172).  No arithmetic happens in
Python: each wrapper marshals pointers, shapes and the current CUDA stream.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

from . import _lib
from ._lib import GEMM_KK, GEMM_KMN, GEMM_MNMN, act, check, load, ptr, stream_ptr


def _opt_act(t: Optional[torch.Tensor], name: str):
    return None if t is None else ctypes.byref(act(t, name))


# --------------------------------------------------------------------------- conv
COLSTATS_SLOTS = 4
COLSTATS_MIN_PIXELS = 128     # the fused epilogue sums need one image per 128-pixel output tile


class ColStats:
    """Per-(image, channel) sum / sum-of-squares workspace of one activation BUFFER, filled by the epilogues
    of the convolutions that write into it (each at its channel offset) and turned into GroupNorm
    statistics by groupnorm_stats_from_cols."""

    def __init__(self, n: int, channels: int, device, slots: int = COLSTATS_SLOTS):
        self.ws = torch.zeros((slots, n, 2, channels), dtype=torch.float32, device=device)
        self.n, self.channels, self.slots = n, channels, slots

    def desc(self, channel_offset: int = 0):
        return _lib.fdx_colstats(self.ws.data_ptr() + 4 * channel_offset, self.slots, self.channels)


def groupnorm_stats_from_cols(cs: ColStats, groups: int, c0: int = 0, channels: Optional[int] = None) -> torch.Tensor:
    """fdx_groupnorm_stats' output for channels [c0, c0 + channels) of the buffer, from its epilogue sums."""
    channels = cs.channels - c0 if channels is None else channels
    stats = torch.empty((cs.n, groups, 2), dtype=torch.float32, device=cs.ws.device)
    check(load().fdx_groupnorm_stats_from_cols(ptr(cs.ws), ctypes.c_int(cs.slots), ctypes.c_int(cs.n),
                                               ctypes.c_int(cs.channels), ctypes.c_int(c0), ctypes.c_int(channels),
                                               ctypes.c_int(groups), ptr(stats), stream_ptr()),
          "groupnorm_stats_from_cols")
    return stats


def conv3x3_fwd(x: torch.Tensor, w_hwio: torch.Tensor, bias: Optional[torch.Tensor] = None,
                rowvec: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, stride: int = 1, colstats=None) -> torch.Tensor:
    """3x3 SAME conv, NHWC bf16, HWIO bf16 weights; out = conv + bias + rowvec[n] + res.
    colstats = (ColStats, channel offset): also accumulate the output's per-image channel sums."""
    n, h, w, cin = x.shape
    cout = w_hwio.shape[-1]
    assert w_hwio.dtype == torch.bfloat16 and w_hwio.is_contiguous()
    assert tuple(w_hwio.shape) == (3, 3, cin, cout), (w_hwio.shape, cin, cout)
    ho, wo = (h + stride - 1) // stride, (w + stride - 1) // stride
    if out is None:
        out = torch.empty((n, ho, wo, cout), dtype=torch.bfloat16, device=x.device)
    if colstats is not None:
        d = colstats[0].desc(colstats[1])
        check(load().fdx_conv3x3_fwd_stats(ctypes.byref(act(x, "x")), ptr(w_hwio), ptr(bias), ptr(rowvec),
                                           _opt_act(res, "res"), ctypes.byref(act(out, "out")),
                                           ctypes.c_int(stride), ctypes.byref(d), stream_ptr()),
              "conv3x3_fwd_stats")
        return out
    check(load().fdx_conv3x3_fwd(ctypes.byref(act(x, "x")), ptr(w_hwio), ptr(bias), ptr(rowvec),
                                 _opt_act(res, "res"), ctypes.byref(act(out, "out")),
                                 ctypes.c_int(stride), stream_ptr()), "conv3x3_fwd")
    return out


def conv3x3_dgrad(dy: torch.Tensor, w_hwio: torch.Tensor, dx: torch.Tensor, stride: int = 1,
                  accumulate: bool = False) -> torch.Tensor:
    check(load().fdx_conv3x3_dgrad(ctypes.byref(act(dy, "dy")), ptr(w_hwio),
                                   ctypes.byref(act(dx, "dx")), ctypes.c_int(stride),
                                   ctypes.c_int(1 if accumulate else 0), stream_ptr()),
          "conv3x3_dgrad")
    return dx


def conv3x3_wgrad(x: torch.Tensor, dy: torch.Tensor, dw_hwio: torch.Tensor, stride: int = 1) -> torch.Tensor:
    """Accumulates d(loss)/dw (f32 HWIO) into dw_hwio."""
    assert dw_hwio.dtype == torch.float32 and dw_hwio.is_contiguous()
    check(load().fdx_conv3x3_wgrad(ctypes.byref(act(x, "x")), ctypes.byref(act(dy, "dy")),
                                   ptr(dw_hwio), ctypes.c_int(stride), stream_ptr()),
          "conv3x3_wgrad")
    return dw_hwio


def conv1x1_fwd(x: torch.Tensor, w_io: torch.Tensor, bias: Optional[torch.Tensor] = None,
                res: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """1x1 conv in convolution geometry: x NHWC bf16, w_io bf16 [Cin, Cout] (flax (1,1,Cin,Cout))."""
    n, h, w, cin = x.shape
    cout = w_io.shape[-1]
    assert w_io.dtype == torch.bfloat16 and w_io.is_contiguous() and w_io.numel() == cin * cout
    if out is None:
        out = torch.empty((n, h, w, cout), dtype=torch.bfloat16, device=x.device)
    check(load().fdx_conv1x1_fwd(ctypes.byref(act(x, "x")), ptr(w_io), ptr(bias), _opt_act(res, "res"),
                                 ctypes.byref(act(out, "out")), stream_ptr()), "conv1x1_fwd")
    return out


def conv1x1_dgrad(dy: torch.Tensor, w_io: torch.Tensor, dx: torch.Tensor, accumulate: bool = False) -> torch.Tensor:
    check(load().fdx_conv1x1_dgrad(ctypes.byref(act(dy, "dy")), ptr(w_io), ctypes.byref(act(dx, "dx")),
                                   ctypes.c_int(1 if accumulate else 0), stream_ptr()), "conv1x1_dgrad")
    return dx


# --------------------------------------------------------------------------- gemm
def gemm(mode: int, A: torch.Tensor, B: torch.Tensor, D: torch.Tensor, M: int, N: int, K: int,
         a_ld: int, b_ld: int, d_ld: int, batch1: int = 1, batch2: int = 1,
         a_s=(0, 0), b_s=(0, 0), d_s=(0, 0), alpha: float = 1.0,
         bias: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None,
         r_ld: int = 0, r_s=(0, 0), atomic: bool = False, reduce_batch: bool = False) -> torch.Tensor:
    """Generic (batched) bf16 GEMM on the tcgen05 engine; see include/fdx.h fdx_gemm_desc."""
    g = _lib.fdx_gemm_desc()
    g.mode = mode
    g.M, g.N, g.K = M, N, K
    g.batch1, g.batch2 = batch1, batch2
    g.A, g.a_ld, g.a_s1, g.a_s2 = ptr(A), a_ld, a_s[0], a_s[1]
    g.B, g.b_ld, g.b_s1, g.b_s2 = ptr(B), b_ld, b_s[0], b_s[1]
    g.D, g.d_ld, g.d_s1, g.d_s2 = ptr(D), d_ld, d_s[0], d_s[1]
    g.d_f32 = 1 if D.dtype == torch.float32 else 0
    g.d_atomic = 1 if atomic else 0
    g.reduce_batch = 1 if reduce_batch else 0
    g.alpha = alpha
    g.bias = ptr(bias)
    g.res, g.r_ld, g.r_s1, g.r_s2 = ptr(res), r_ld, r_s[0], r_s[1]
    check(load().fdx_gemm(ctypes.byref(g), stream_ptr()), "gemm")
    return D


def linear_fwd(x2d: torch.Tensor, w_kn: torch.Tensor, out: Optional[torch.Tensor] = None,
               bias: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None,
               out_dtype=torch.bfloat16) -> torch.Tensor:
    """y[m][n] = x[m][k] @ w[k][n] (flax Dense kernel layout (in, out)); x row stride may exceed K."""
    M, K = x2d.shape
    Kw, N = w_kn.shape
    assert K == Kw and x2d.stride(1) == 1 and w_kn.is_contiguous()
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=x2d.device)
    return gemm(GEMM_KMN, x2d, w_kn, out, M, N, K, x2d.stride(0), N, out.stride(0), bias=bias,
                res=res, r_ld=(res.stride(0) if res is not None else 0))


# --------------------------------------------------------------------------- norms
def groupnorm_stats(x: torch.Tensor, groups: int) -> torch.Tensor:
    stats = torch.empty((x.shape[0], groups, 2), dtype=torch.float32, device=x.device)
    check(load().fdx_groupnorm_stats(ctypes.byref(act(x, "x")), ctypes.c_int(groups), ptr(stats),
                                     stream_ptr()), "groupnorm_stats")
    return stats


def groupnorm_apply(x, groups, stats, gamma, beta, eps: float, silu: bool, out=None) -> torch.Tensor:
    if out is None:
        out = torch.empty(tuple(x.shape), dtype=torch.bfloat16, device=x.device)
    check(load().fdx_groupnorm_apply(ctypes.byref(act(x, "x")), ctypes.c_int(groups), ptr(stats),
                                     ptr(gamma), ptr(beta), ctypes.c_float(eps),
                                     ctypes.c_int(1 if silu else 0), ctypes.byref(act(out, "out")),
                                     stream_ptr()), "groupnorm_apply")
    return out


def groupnorm_apply_cols(x, groups, cs: "ColStats", c0: int, gamma, beta, eps: float, silu: bool, out=None):
    """groupnorm_apply with the statistics read from the producers' epilogue column sums (no stats_from_cols
    launch) -> (y, stats[N][groups][2] for the backward)."""
    if out is None:
        out = torch.empty(tuple(x.shape), dtype=torch.bfloat16, device=x.device)
    stats = torch.empty((cs.n, groups, 2), dtype=torch.float32, device=x.device)
    check(load().fdx_groupnorm_apply_cols(ctypes.byref(act(x, "x")), ctypes.c_int(groups), ptr(cs.ws),
                                          ctypes.c_int(cs.slots), ctypes.c_int(cs.channels), ctypes.c_int(c0),
                                          ptr(gamma), ptr(beta), ctypes.c_float(eps), ctypes.c_int(1 if silu else 0),
                                          ctypes.byref(act(out, "out")), ptr(stats), stream_ptr()),
          "groupnorm_apply_cols")
    return out, stats


def groupnorm_bwd(x, dy, groups, stats, gamma, beta, eps, silu, dgamma, dbeta, dx,
                  accumulate: bool = False, csum_img=None, csum_tot=None, addend=None) -> torch.Tensor:
    """dx (+)= d/dx GroupNorm(+SiLU); `addend`: dx = d/dx + addend (another tensor of the same shape)."""
    red = torch.empty(2 * x.shape[0] * groups, dtype=torch.float32, device=x.device)
    if addend is not None:
        assert not accumulate
        check(load().fdx_groupnorm_bwd_add(ctypes.byref(act(x, "x")), ctypes.byref(act(dy, "dy")),
                                           ctypes.c_int(groups), ptr(stats), ptr(gamma), ptr(beta),
                                           ctypes.c_float(eps), ctypes.c_int(1 if silu else 0), ptr(red),
                                           ptr(dgamma), ptr(dbeta), ctypes.byref(act(dx, "dx")),
                                           ctypes.byref(act(addend, "addend")), ptr(csum_img), ptr(csum_tot),
                                           stream_ptr()), "groupnorm_bwd_add")
        return dx
    check(load().fdx_groupnorm_bwd(ctypes.byref(act(x, "x")), ctypes.byref(act(dy, "dy")),
                                   ctypes.c_int(groups), ptr(stats), ptr(gamma), ptr(beta),
                                   ctypes.c_float(eps), ctypes.c_int(1 if silu else 0), ptr(red),
                                   ptr(dgamma), ptr(dbeta), ctypes.byref(act(dx, "dx")),
                                   ctypes.c_int(1 if accumulate else 0), ptr(csum_img), ptr(csum_tot),
                                   stream_ptr()),
          "groupnorm_bwd")
    return dx


GN_FUSE_SLOTS = 8
GN_FUSE_MIN_PIXELS = 128    # fdx_conv3x3_dgrad_gn needs one image per 128-pixel tile


def groupnorm_coeffs(stats, gamma, beta, hw: int, eps: float) -> torch.Tensor:
    """ab[n][0][c] = rstd*gamma_c, ab[n][1][c] = beta_c - mean*rstd*gamma_c (f32)."""
    n, groups = stats.shape[0], stats.shape[1]
    c = gamma.numel()
    ab = torch.empty((n, 2, c), dtype=torch.float32, device=stats.device)
    check(load().fdx_groupnorm_coeffs(ptr(stats), ptr(gamma), ptr(beta), ctypes.c_int(n), ctypes.c_int(hw),
                                      ctypes.c_int(c), ctypes.c_int(groups), ctypes.c_float(eps), ptr(ab),
                                      stream_ptr()), "groupnorm_coeffs")
    return ab


def conv3x3_dgrad_gn(dy: torch.Tensor, w_hwio: torch.Tensor, dz: torch.Tensor, x: torch.Tensor,
                     ab: torch.Tensor, slots: int = GN_FUSE_SLOTS) -> torch.Tensor:
    """Stride-1 data gradient with the first pass of GroupNorm(+SiLU) backward fused into its epilogue:
    writes dz = dgrad * silu'(a x + b) and returns the per-slot sums workspace for groupnorm_bwd_dz."""
    n, c = dz.shape[0], dz.shape[-1]
    ws = torch.empty((slots, n, 2, c), dtype=torch.float32, device=dz.device)
    check(load().fdx_conv3x3_dgrad_gn(ctypes.byref(act(dy, "dy")), ptr(w_hwio), ctypes.byref(act(dz, "dz")),
                                      ctypes.byref(act(x, "x")), ptr(ab), ptr(ws), ctypes.c_int(slots),
                                      stream_ptr()), "conv3x3_dgrad_gn")
    return ws


def groupnorm_bwd_dz(x, dz, groups, stats, gamma, eps, ws_slots, dgamma, dbeta, dx,
                     accumulate: bool = False, csum_img=None, csum_tot=None, addend=None) -> torch.Tensor:
    if addend is not None:
        assert not accumulate, "groupnorm_bwd_dz: addend and accumulate are exclusive"
        check(load().fdx_groupnorm_bwd_dz_add(ctypes.byref(act(x, "x")), ctypes.byref(act(dz, "dz")),
                                              ctypes.c_int(groups), ptr(stats), ptr(gamma), ctypes.c_float(eps),
                                              ptr(ws_slots), ctypes.c_int(ws_slots.shape[0]), ptr(None), ptr(dgamma),
                                              ptr(dbeta), ctypes.byref(act(dx, "dx")),
                                              ctypes.byref(act(addend, "addend")), ptr(csum_img), ptr(csum_tot),
                                              stream_ptr()), "groupnorm_bwd_dz_add")
        return dx
    check(load().fdx_groupnorm_bwd_dz(ctypes.byref(act(x, "x")), ctypes.byref(act(dz, "dz")),
                                      ctypes.c_int(groups), ptr(stats), ptr(gamma), ctypes.c_float(eps),
                                      ptr(ws_slots), ctypes.c_int(ws_slots.shape[0]), ptr(None), ptr(dgamma),
                                      ptr(dbeta), ctypes.byref(act(dx, "dx")),
                                      ctypes.c_int(1 if accumulate else 0), ptr(csum_img), ptr(csum_tot),
                                      stream_ptr()), "groupnorm_bwd_dz")
    return dx


def _gn_fuse_default(x: torch.Tensor, dy: torch.Tensor) -> bool:
    """The fused first pass is the default where the data gradient runs on the transposed engine (eight epilogue
    warps hide the silu' arithmetic; DESIGN 3.2): Cin = 64 ... 512 not a multiple of 256, 16-aligned images."""
    cin, h, w = x.shape[-1], x.shape[1], x.shape[2]
    return (cin % 64 == 0 and cin % 256 != 0 and cin <= 512 and dy.shape[-1] % 64 == 0 and h % 16 == 0 and
            w % 16 == 0 and h * w >= GN_FUSE_MIN_PIXELS)


def conv_dgrad_groupnorm_bwd(dy, w_hwio, x, groups, stats, gamma, beta, eps, dgamma, dbeta, dx,
                             accumulate: bool = False, csum_img=None, csum_tot=None,
                             fused: Optional[bool] = None, addend=None) -> torch.Tensor:
    """d/dx of conv3x3(silu(groupnorm(x))) given dy = d/d(conv output): the data gradient with the first pass
    of the GroupNorm backward in its epilogue (dz = dy * silu'(z), sum dz, sum dz*x) where that convolution runs
    on the transposed engine, then ONE pass over x and dz; elsewhere data gradient + the two-pass GroupNorm
    backward.  FDX_GN_FUSE=0: never fused; FDX_GN_FUSE=1: fused wherever an image has >= 128 pixels (also on the
    pixels-as-M engine, where four epilogue warps make it slower - profiles/layers_r01_gn_fusion.txt)."""
    da = torch.empty(tuple(x.shape), dtype=torch.bfloat16, device=x.device)
    if fused is None:
        env = os.environ.get("FDX_GN_FUSE")
        if env is None or env == "":
            fused = _gn_fuse_default(x, dy)
        else:
            fused = env != "0" and x.shape[1] * x.shape[2] >= GN_FUSE_MIN_PIXELS
    if fused and x.shape[1] * x.shape[2] >= GN_FUSE_MIN_PIXELS:
        ab = groupnorm_coeffs(stats, gamma, beta, x.shape[1] * x.shape[2], eps)
        ws = conv3x3_dgrad_gn(dy, w_hwio, da, x, ab)
        return groupnorm_bwd_dz(x, da, groups, stats, gamma, eps, ws, dgamma, dbeta, dx, accumulate,
                                csum_img=csum_img, csum_tot=csum_tot, addend=addend)
    conv3x3_dgrad(dy, w_hwio, da)
    return groupnorm_bwd(x, da, groups, stats, gamma, beta, eps, True, dgamma, dbeta, dx, accumulate,
                         csum_img=csum_img, csum_tot=csum_tot, addend=addend)


def rmsnorm_fwd(x, scale, eps: float, out=None) -> torch.Tensor:
    if out is None:
        out = torch.empty(tuple(x.shape), dtype=torch.bfloat16, device=x.device)
    check(load().fdx_rmsnorm_fwd(ctypes.byref(act(x, "x")), ptr(scale), ctypes.c_float(eps),
                                 ctypes.byref(act(out, "out")), stream_ptr()), "rmsnorm_fwd")
    return out


def rmsnorm_bwd(x, dy, scale, eps, dx, dscale, accumulate: bool = False) -> torch.Tensor:
    check(load().fdx_rmsnorm_bwd(ctypes.byref(act(x, "x")), ctypes.byref(act(dy, "dy")), ptr(scale),
                                 ctypes.c_float(eps), ctypes.byref(act(dx, "dx")),
                                 ctypes.c_int(1 if accumulate else 0), ptr(dscale), stream_ptr()),
          "rmsnorm_bwd")
    return dx


# --------------------------------------------------------------------------- streaming
TARGET_X0, TARGET_EPS, TARGET_V = 0, 1, 2


def diffuse_forward(x0: torch.Tensor, eps: torch.Tensor, alpha, sigma, c_in, normalize: bool,
                    target_kind: int):
    """-> (x_t f32, target f32, model_in bf16); x0 may be uint8 or f32, shape (B, ...)."""
    B = x0.shape[0]
    E = x0.numel() // B
    assert x0.is_contiguous() and eps.is_contiguous() and eps.dtype == torch.float32
    assert x0.dtype in (torch.uint8, torch.float32)
    x_t = torch.empty(tuple(x0.shape), dtype=torch.float32, device=x0.device)
    target = torch.empty_like(x_t)
    model_in = torch.empty(tuple(x0.shape), dtype=torch.bfloat16, device=x0.device)
    check(load().fdx_diffuse_forward(ptr(x0), ctypes.c_int(1 if x0.dtype == torch.uint8 else 0),
                                     ptr(eps), ptr(_f32c(alpha)), ptr(_f32c(sigma)), ptr(_f32c(c_in)),
                                     ctypes.c_int(B), ctypes.c_longlong(E),
                                     ctypes.c_int(1 if normalize else 0), ctypes.c_int(target_kind),
                                     ptr(x_t), ptr(target), ptr(model_in), stream_ptr()),
          "diffuse_forward")
    return x_t, target, model_in


def _f32c(t: torch.Tensor) -> torch.Tensor:
    t = t.reshape(-1)
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.to(torch.float32).contiguous()
    return t


def loss_fwd_bwd(F: torch.Tensor, x_t, target, c_out, c_skip, weight, want_grad: bool = True):
    """-> (loss scalar tensor f32[1], dF f32 or None)."""
    B = F.shape[0]
    E = F.numel() // B
    loss = torch.empty(1, dtype=torch.float32, device=F.device)
    dF = torch.empty_like(F) if want_grad else None
    check(load().fdx_loss_fwd_bwd(ptr(F), ptr(x_t), ptr(target), ptr(_f32c(c_out)), ptr(_f32c(c_skip)),
                                  ptr(_f32c(weight)), ctypes.c_int(B), ctypes.c_longlong(E), ptr(loss),
                                  ptr(dF), stream_ptr()), "loss_fwd_bwd")
    return loss, dF


def affine_combine(inputs, coef1: torch.Tensor, coef2: Optional[torch.Tensor] = None,
                   want_out1: bool = True, bf16_scale: Optional[torch.Tensor] = None,
                   want_bf16: bool = False, clip=None):
    """out1 = sum_i coef1[i,b]*in_i; out2 = sum_i coef2[i,b]*in_i; bf16 = bf16(out1*scale[b])."""
    n_in = len(inputs)
    x = inputs[0]
    B = x.shape[0]
    E = x.numel() // B
    for t in inputs:
        assert t.dtype == torch.float32 and t.is_contiguous() and t.shape == x.shape
    coef1 = coef1.to(torch.float32).contiguous()
    assert coef1.shape == (n_in, B), (coef1.shape, n_in, B)
    if coef2 is not None:
        coef2 = coef2.to(torch.float32).contiguous()
    arr = (ctypes.c_void_p * n_in)(*[t.data_ptr() for t in inputs])
    out1 = torch.empty_like(x) if want_out1 else None
    out2 = torch.empty_like(x) if coef2 is not None else None
    outb = torch.empty(tuple(x.shape), dtype=torch.bfloat16, device=x.device) if want_bf16 else None
    lo, hi = (clip if clip is not None else (0.0, 0.0))
    check(load().fdx_affine_combine(ctypes.c_int(n_in), arr, ptr(coef1), ptr(coef2),
                                    ptr(_f32c(bf16_scale)) if bf16_scale is not None else ptr(None),
                                    ctypes.c_int(B), ctypes.c_longlong(E), ptr(out1), ptr(out2),
                                    ptr(outb), ctypes.c_int(1 if clip is not None else 0),
                                    ctypes.c_float(lo), ctypes.c_float(hi), stream_ptr()),
          "affine_combine")
    return out1, out2, outb


def adamw_ema_step(p, g, m, v, ema, shadow, lr, b1, b2, eps, weight_decay, step, ema_decay,
                   grad_scale: float = 1.0, gnorm_sq=None, clip_norm: float = 0.0, dyn=None):
    check(load().fdx_adamw_ema_step(ptr(p), ptr(g), ptr(m), ptr(v), ptr(ema), ptr(shadow),
                                    ctypes.c_longlong(p.numel()), ctypes.c_float(lr),
                                    ctypes.c_float(b1), ctypes.c_float(b2), ctypes.c_float(eps),
                                    ctypes.c_float(weight_decay), ctypes.c_int(step),
                                    ctypes.c_float(ema_decay), ctypes.c_float(grad_scale),
                                    ptr(gnorm_sq), ctypes.c_float(clip_norm), ptr(dyn), stream_ptr()),
          "adamw_ema_step")


def optimizer_step(kind: int, p, g, m, v, ema, shadow, lr, b1, b2, eps, weight_decay, step, ema_decay=0.999,
                   grad_scale: float = 1.0, gstats=None, clip_norm: float = 0.0, dyn=None, dynscale=None,
                   seg_offsets=None, seg_norms=None, u_ws=None):
    """fdx_optimizer_step: adam / adamw / lamb update (+ optional EMA, bf16 shadow refresh, global-norm clip,
    DynamicScale unscale-and-skip) over the flat buffers.  `ema=None` = TrainState.apply_gradients alone."""
    d = _lib.fdx_opt_desc()
    d.kind = kind
    d.p, d.g, d.m, d.v = ptr(p), ptr(g), ptr(m), ptr(v)
    d.ema, d.shadow_bf16, d.n = ptr(ema), ptr(shadow), p.numel()
    d.lr, d.b1, d.b2, d.eps, d.weight_decay = lr, b1, b2, eps, weight_decay
    d.step, d.ema_decay, d.grad_scale = step, ema_decay, grad_scale
    d.gstats, d.clip_norm, d.dyn_lr_bc, d.dynscale = ptr(gstats), clip_norm, ptr(dyn), ptr(dynscale)
    if seg_offsets is not None:
        assert seg_offsets.dtype == torch.int64
        d.seg_offsets, d.nseg = ptr(seg_offsets), seg_offsets.numel()
        d.seg_norms, d.u_ws = ptr(seg_norms), ptr(u_ws)
    check(load().fdx_optimizer_step(ctypes.byref(d), stream_ptr()), "optimizer_step")


def ema_update(ema: torch.Tensor, p: torch.Tensor, decay: float):
    """ema = decay * ema + (1 - decay) * p over the flat buffers (TrainState.apply_ema)."""
    check(load().fdx_ema_update(ptr(ema), ptr(p), ctypes.c_longlong(p.numel()), ctypes.c_float(decay),
                                stream_ptr()), "ema_update")


def grad_stats(g: torch.Tensor) -> torch.Tensor:
    """-> f32[2] = (sum g^2, number of non-finite elements)."""
    out = torch.empty(2, dtype=torch.float32, device=g.device)
    check(load().fdx_grad_stats(ptr(g), ctypes.c_longlong(g.numel()), ptr(out), stream_ptr()), "grad_stats")
    return out


def sumsq(g: torch.Tensor) -> torch.Tensor:
    return grad_stats(g)


def dynscale_update(state3: torch.Tensor, gstats: torch.Tensor, growth_factor=2.0, backoff_factor=0.5,
                    growth_interval=2000, minimum_scale=1.1754943508222875e-38):
    check(load().fdx_dynscale_update(ptr(state3), ptr(gstats), ctypes.c_float(growth_factor),
                                     ctypes.c_float(backoff_factor), ctypes.c_int(growth_interval),
                                     ctypes.c_float(minimum_scale), stream_ptr()), "dynscale_update")


# --------------------------------------------------------------------------- data-parallel exchange
class Comm:
    """fdx_comm handle: NCCL communicator bound inside libfdx (one per process).  `unique_id()` on rank 0,
    broadcast the 128 bytes by any side channel, then `Comm(rank, world, id)` on every rank."""

    @staticmethod
    def unique_id() -> bytes:
        buf = ctypes.create_string_buffer(128)
        check(load().fdx_comm_unique_id(buf), "comm_unique_id")
        return buf.raw

    def __init__(self, rank: int, world: int, uid: bytes):
        assert len(uid) == 128
        self._h = ctypes.c_void_p()
        check(load().fdx_comm_init(ctypes.byref(self._h), ctypes.c_int(rank), ctypes.c_int(world),
                                   ctypes.create_string_buffer(uid, 128)), "comm_init")
        self.rank, self.world = rank, world

    def allreduce_avg_(self, buf: torch.Tensor, stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
        """In-place mean over ranks of a contiguous f32 CUDA tensor (a bucket of the flat gradient buffer)."""
        assert buf.dtype == torch.float32 and buf.is_contiguous()
        st = ctypes.c_void_p((stream or torch.cuda.current_stream()).cuda_stream)
        check(load().fdx_comm_allreduce_avg(self._h, ptr(buf), ctypes.c_longlong(buf.numel()), st),
              "comm_allreduce_avg")
        return buf

    def destroy(self):
        if self._h:
            check(load().fdx_comm_destroy(self._h), "comm_destroy")
            self._h = ctypes.c_void_p()


def nccl_version() -> int:
    return int(load().fdx_comm_nccl_version())


def cast_f32_bf16(src: torch.Tensor, dst: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert src.dtype == torch.float32 and src.is_contiguous()
    if dst is None:
        dst = torch.empty(tuple(src.shape), dtype=torch.bfloat16, device=src.device)
    check(load().fdx_cast_f32_bf16(ptr(src), ptr(dst), ctypes.c_longlong(src.numel()), stream_ptr()),
          "cast_f32_bf16")
    return dst


def upsample2x(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    n, h, w, c = x.shape
    if out is None:
        out = torch.empty((n, 2 * h, 2 * w, c), dtype=torch.bfloat16, device=x.device)
    check(load().fdx_upsample2x(ctypes.byref(act(x, "x")), ctypes.byref(act(out, "out")), stream_ptr()),
          "upsample2x")
    return out


def upsample2x_bwd(dy: torch.Tensor, dx: torch.Tensor, accumulate: bool = False) -> torch.Tensor:
    check(load().fdx_upsample2x_bwd(ctypes.byref(act(dy, "dy")), ctypes.byref(act(dx, "dx")),
                                    ctypes.c_int(1 if accumulate else 0), stream_ptr()),
          "upsample2x_bwd")
    return dx


def act_add(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    check(load().fdx_act_add(ctypes.byref(act(a, "a")), ctypes.byref(act(b, "b")),
                             ctypes.byref(act(out, "out")), stream_ptr()), "act_add")
    return out


def colsum(x: torch.Tensor, per_image: bool, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        shape = (x.shape[0], x.shape[-1]) if per_image else (x.shape[-1],)
        out = torch.empty(shape, dtype=torch.float32, device=x.device)
    check(load().fdx_colsum(ctypes.byref(act(x, "x")), ptr(out), ctypes.c_int(1 if per_image else 0),
                            stream_ptr()), "colsum")
    return out


# --------------------------------------------------------------------------- upsample + conv (sub-pixel)
def upconv3x3_pack(w_hwio: torch.Tensor) -> torch.Tensor:
    """bf16 [16][Cin][Cout] parity/tap-summed weights of nearest-2x + conv3x3 from the f32 HWIO kernel."""
    assert w_hwio.dtype == torch.float32 and w_hwio.is_contiguous() and w_hwio.shape[:2] == (3, 3)
    cin, cout = w_hwio.shape[2], w_hwio.shape[3]
    weff = torch.empty((16, cin, cout), dtype=torch.bfloat16, device=w_hwio.device)
    check(load().fdx_upconv3x3_pack(ptr(w_hwio), ctypes.c_int(cin), ctypes.c_int(cout), ptr(weff), stream_ptr()),
          "upconv3x3_pack")
    return weff


def upconv3x3_fwd(x: torch.Tensor, weff: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor,
                  colstats=None) -> torch.Tensor:
    """out[B,2h,2w,Cout] = conv3x3_SAME(nearest2x(x)) + bias, without the upsampled tensor."""
    if colstats is not None:
        d = colstats[0].desc(colstats[1])
        check(load().fdx_upconv3x3_fwd_stats(ctypes.byref(act(x, "x")), ptr(weff), ptr(bias),
                                             ctypes.byref(act(out, "out")), ctypes.byref(d), stream_ptr()),
              "upconv3x3_fwd_stats")
        return out
    check(load().fdx_upconv3x3_fwd(ctypes.byref(act(x, "x")), ptr(weff), ptr(bias), ctypes.byref(act(out, "out")),
                                   stream_ptr()), "upconv3x3_fwd")
    return out


def upconv3x3_dgrad(dy: torch.Tensor, weff: torch.Tensor, dx: torch.Tensor, accumulate: bool = False) -> torch.Tensor:
    check(load().fdx_upconv3x3_dgrad(ctypes.byref(act(dy, "dy")), ptr(weff), ctypes.byref(act(dx, "dx")),
                                     ctypes.c_int(1 if accumulate else 0), stream_ptr()), "upconv3x3_dgrad")
    return dx


def upconv3x3_wgrad(x: torch.Tensor, dy: torch.Tensor, dw_hwio: torch.Tensor) -> torch.Tensor:
    """Accumulates d(loss)/dw of the 3x3 kernel (f32 HWIO) into dw_hwio."""
    assert dw_hwio.dtype == torch.float32 and dw_hwio.is_contiguous()
    ws = torch.empty((16, x.shape[-1], dy.shape[-1]), dtype=torch.float32, device=x.device)
    check(load().fdx_upconv3x3_wgrad(ctypes.byref(act(x, "x")), ctypes.byref(act(dy, "dy")), ptr(ws), ptr(dw_hwio),
                                     stream_ptr()), "upconv3x3_wgrad")
    return dw_hwio


# --------------------------------------------------------------------------- 3-channel convs
def conv_in_fwd(x_bf16: torch.Tensor, w: torch.Tensor, bias, out: torch.Tensor,
                w_bf16: Optional[torch.Tensor] = None) -> torch.Tensor:
    """conv_in 3->Cout as im2col (K = 27 padded to 32) + one tcgen05 GEMM with the bias fused."""
    n, h, w_, c = x_bf16.shape
    assert c == 3 and x_bf16.dtype == torch.bfloat16 and x_bf16.is_contiguous()
    cout = out.shape[-1]
    col = im2col3(x_bf16, +1, False)
    wb = w_bf16 if w_bf16 is not None else cast_f32_bf16(w)
    gemm(GEMM_KMN, col, wb, out, n * h * w_, cout, 27, 32, cout, out.stride(2), bias=bias)
    return out


def conv_in_fwd_direct(x_bf16: torch.Tensor, w: torch.Tensor, bias, out: torch.Tensor) -> torch.Tensor:
    """Workspace-free CUDA-core variant (fdx_conv_in_fwd)."""
    n, h, w_, c = x_bf16.shape
    assert c == 3 and x_bf16.dtype == torch.bfloat16 and x_bf16.is_contiguous()
    assert w.dtype == torch.float32 and w.is_contiguous()
    check(load().fdx_conv_in_fwd(ptr(x_bf16), ctypes.c_int(n), ctypes.c_int(h), ctypes.c_int(w_),
                                 ptr(w), ptr(bias), ctypes.byref(act(out, "out")), stream_ptr()),
          "conv_in_fwd")
    return out


def im2col3(src: torch.Tensor, sgn: int, ones_col: bool) -> torch.Tensor:
    n, h, w, c = src.shape
    assert c == 3 and src.is_contiguous() and src.dtype in (torch.float32, torch.bfloat16)
    col = torch.empty((n * h * w, 32), dtype=torch.bfloat16, device=src.device)
    check(load().fdx_im2col3x3_c3(ptr(src), ctypes.c_int(1 if src.dtype == torch.float32 else 0),
                                  ctypes.c_int(sgn), ctypes.c_int(n), ctypes.c_int(h), ctypes.c_int(w),
                                  ctypes.c_int(1 if ones_col else 0), ptr(col), stream_ptr()), "im2col3x3_c3")
    return col


def conv_in_wgrad(x_bf16, dy, dw, dbias):
    """dW[t][cs][co] (+ bias row) = im2col(x)^T @ dY on the tensor cores; accumulates into dw / dbias."""
    n, h, w, cout = dy.shape
    P = n * h * w
    col = im2col3(x_bf16, +1, True)
    tmp = torch.zeros((32, cout), dtype=torch.float32, device=dy.device)
    gemm(GEMM_MNMN, col, dy, tmp, 32, cout, P, 32, dy.stride(2), cout, atomic=True, reduce_batch=True)
    dw.view(27, cout).add_(tmp[:27])
    if dbias is not None:
        dbias.add_(tmp[27])


def conv_in_wgrad_direct(x_bf16, dy, dw, dbias):
    """Workspace-free CUDA-core variant (fdx_conv_in_wgrad)."""
    check(load().fdx_conv_in_wgrad(ptr(x_bf16), ctypes.byref(act(dy, "dy")), ptr(dw), ptr(dbias),
                                   stream_ptr()), "conv_in_wgrad")


def conv_out_fwd(x: torch.Tensor, w: torch.Tensor, bias) -> torch.Tensor:
    """conv_out Cin->3: one tcgen05 GEMM (pixels x Cin)(Cin x 27, padded to 32) with f32 output, then the
    col2im scatter that adds the nine taps' partial sums and the bias."""
    n, h, w_, cin = x.shape
    wr = torch.zeros((cin, 32), dtype=torch.float32, device=x.device)
    wr[:, :27] = w.reshape(9, cin, 3).permute(1, 0, 2).reshape(cin, 27)       # [ci][(t,k)]
    col = torch.empty((n * h * w_, 32), dtype=torch.float32, device=x.device)
    gemm(GEMM_KMN, x, cast_f32_bf16(wr), col, n * h * w_, 32, cin, x.stride(2), 32, 32)
    y = torch.empty((n, h, w_, 3), dtype=torch.float32, device=x.device)
    check(load().fdx_col2im3x3_c3(ptr(col), ptr(bias), ctypes.c_int(n), ctypes.c_int(h), ctypes.c_int(w_),
                                  ptr(y), stream_ptr()), "col2im3x3_c3")
    return y


def conv_out_fwd_direct(x: torch.Tensor, w: torch.Tensor, bias) -> torch.Tensor:
    """Workspace-free CUDA-core variant (fdx_conv_out_fwd)."""
    n, h, w_, c = x.shape
    y = torch.empty((n, h, w_, 3), dtype=torch.float32, device=x.device)
    check(load().fdx_conv_out_fwd(ctypes.byref(act(x, "x")), ptr(w), ptr(bias), ptr(y), stream_ptr()),
          "conv_out_fwd")
    return y


def conv_out_dgrad(dF: torch.Tensor, w: torch.Tensor, dx: torch.Tensor, col: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dx[p][ci] = sum_{t,k} dF[p - d(t)][k] w[t][ci][k]: im2col(dF) (shared with the weight gradient)
    times the (27 x Cin) re-arranged kernel on the tensor cores."""
    n, h, w_, cin = dx.shape
    if col is None:
        col = im2col3(dF, -1, False)
    wt = w.reshape(9, cin, 3).permute(0, 2, 1).reshape(27, cin).contiguous()      # [(t,k)][ci], 1.7 K elements
    gemm(GEMM_KMN, col, cast_f32_bf16(_pad4(wt)), dx, n * h * w_, cin, 27, 32, cin, dx.stride(2))
    return dx


def _pad4(t: torch.Tensor) -> torch.Tensor:
    return t if t.numel() % 4 == 0 else torch.nn.functional.pad(t.reshape(-1), (0, 4 - t.numel() % 4)).reshape(-1)


def conv_out_dgrad_direct(dF: torch.Tensor, w: torch.Tensor, dx: torch.Tensor) -> torch.Tensor:
    check(load().fdx_conv_out_dgrad(ptr(dF), ptr(w), ctypes.byref(act(dx, "dx")), stream_ptr()),
          "conv_out_dgrad")
    return dx


def conv_out_wgrad(x, dF, dw, dbias, col: Optional[torch.Tensor] = None):
    """dW[t][ci][k] = x^T @ im2col(dF) on the tensor cores; accumulates into dw / dbias."""
    n, h, w, cin = x.shape
    P = n * h * w
    if col is None:
        col = im2col3(dF, -1, False)
    tmp = torch.zeros((cin, 32), dtype=torch.float32, device=x.device)
    gemm(GEMM_MNMN, x, col, tmp, cin, 32, P, x.stride(2), 32, 32, atomic=True, reduce_batch=True)
    dw.add_(tmp[:, :27].view(cin, 9, 3).permute(1, 0, 2).reshape(3, 3, cin, 3))
    if dbias is not None:
        cs = colsum(col.view(n, h, w, 32), per_image=False)
        dbias.add_(cs[12:15])        # centre tap (t = 4) columns = sum over pixels of dF


def conv_out_wgrad_direct(x, dF, dw, dbias):
    """Workspace-free CUDA-core variant (fdx_conv_out_wgrad)."""
    check(load().fdx_conv_out_wgrad(ctypes.byref(act(x, "x")), ptr(dF), ptr(dw), ptr(dbias),
                                    stream_ptr()), "conv_out_wgrad")


# --------------------------------------------------------------------------- GEGLU
def geglu_fwd(u: torch.Tensor) -> torch.Tensor:
    """u [rows, 2*inner] bf16 -> hidden_linear * gelu_tanh(hidden_gelu) [rows, inner]."""
    rows, two = u.shape
    assert u.dtype == torch.bfloat16 and u.is_contiguous() and two % 16 == 0
    g = torch.empty((rows, two // 2), dtype=torch.bfloat16, device=u.device)
    check(load().fdx_geglu_fwd(ptr(u), ctypes.c_longlong(rows), ctypes.c_int(two // 2), ptr(g), stream_ptr()),
          "geglu_fwd")
    return g


def geglu_bwd(u: torch.Tensor, dg: torch.Tensor) -> torch.Tensor:
    rows, two = u.shape
    assert dg.shape == (rows, two // 2) and dg.is_contiguous() and dg.dtype == torch.bfloat16
    du = torch.empty_like(u)
    check(load().fdx_geglu_bwd(ptr(u), ptr(dg), ctypes.c_longlong(rows), ctypes.c_int(two // 2), ptr(du),
                               stream_ptr()), "geglu_bwd")
    return du


def colsum_rows(x2d: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[c] = sum over rows of x2d[:, c] (bias gradients of dense layers); columns in slabs of <= 2048."""
    rows, n = x2d.shape
    assert x2d.stride(1) == 1 and out.numel() == n
    for c0 in range(0, n, 2048):
        c1 = min(n, c0 + 2048)
        colsum(x2d[:, c0:c1].unsqueeze(0).unsqueeze(0), False, out=out[c0:c1])
    return out


# --------------------------------------------------------------------------- fused attention
def _attn_desc(q, k, v, o, lse, heads: int, dh: int, scale: float):
    """q / o: [B, L, heads*dh], k / v: [B, Lk, heads*dh] (bf16, last dim contiguous)."""
    B, L, HD = q.shape
    Lk = k.shape[1]
    assert HD == heads * dh and k.shape[2] == HD and v.shape == k.shape and o.shape == q.shape
    for t in (q, k, v, o):
        assert t.dtype == torch.bfloat16 and t.stride(2) == 1
    a = _lib.fdx_attn_desc()
    a.B, a.heads, a.L, a.Lk, a.dh, a.scale = B, heads, L, Lk, dh, scale
    a.q, a.q_ld, a.q_bs = ptr(q), q.stride(1), q.stride(0)
    a.k, a.k_ld, a.k_bs = ptr(k), k.stride(1), k.stride(0)
    a.v, a.v_ld, a.v_bs = ptr(v), v.stride(1), v.stride(0)
    a.o, a.o_ld, a.o_bs = ptr(o), o.stride(1), o.stride(0)
    a.lse = ptr(lse)
    return a


def attention_fwd(q, k, v, heads: int, dh: int, scale: float, out=None):
    """o = softmax(q k^T * scale) v per (image, head) - fdx_attention_fwd.  -> (o bf16 [B, L, heads*dh],
    lse f32 [B, heads, L]).  No (B, h, L, Lk) tensor exists in HBM."""
    B, L, HD = q.shape
    o = out if out is not None else torch.empty((B, L, HD), dtype=torch.bfloat16, device=q.device)
    lse = torch.empty((B, heads, L), dtype=torch.float32, device=q.device)
    a = _attn_desc(q, k, v, o, lse, heads, dh, scale)
    check(load().fdx_attention_fwd(ctypes.byref(a), stream_ptr()), "attention_fwd")
    return o, lse


def attention_bwd(q, k, v, o, lse, d_o, heads: int, dh: int, scale: float):
    """-> (dq [B, L, HD], dk, dv [B, Lk, HD]) bf16 - fdx_attention_bwd (S / P recomputed on chip)."""
    assert d_o.shape == q.shape and d_o.dtype == torch.bfloat16 and d_o.stride(2) == 1
    dq = torch.empty_like(q, memory_format=torch.contiguous_format)
    dk = torch.empty(tuple(k.shape), dtype=torch.bfloat16, device=k.device)
    dv = torch.empty(tuple(v.shape), dtype=torch.bfloat16, device=v.device)
    ws = torch.empty_like(lse)
    a = _attn_desc(q, k, v, o, lse, heads, dh, scale)
    a.d_o, a.do_ld, a.do_bs = ptr(d_o), d_o.stride(1), d_o.stride(0)
    a.dvec_ws = ptr(ws)
    a.dq, a.dq_ld, a.dq_bs = ptr(dq), dq.stride(1), dq.stride(0)
    a.dk, a.dk_ld, a.dk_bs = ptr(dk), dk.stride(1), dk.stride(0)
    a.dv, a.dv_ld, a.dv_bs = ptr(dv), dv.stride(1), dv.stride(0)
    check(load().fdx_attention_bwd(ctypes.byref(a), stream_ptr()), "attention_bwd")
    return dq, dk, dv


# --------------------------------------------------------------------------- temb / softmax
def time_embed_fwd(t, freqs, W1, b1, W2, b2):
    B, D = t.shape[0], W1.shape[0]
    dev = t.device
    four = torch.empty((B, D), dtype=torch.float32, device=dev)
    h1 = torch.empty_like(four)
    h2 = torch.empty_like(four)
    emb = torch.empty_like(four)
    emb16 = torch.empty((B, D), dtype=torch.bfloat16, device=dev)
    check(load().fdx_time_embed_fwd(ptr(_f32c(t)), ptr(freqs), ptr(W1), ptr(b1), ptr(W2), ptr(b2),
                                    ctypes.c_int(B), ctypes.c_int(D), ptr(four), ptr(h1), ptr(h2),
                                    ptr(emb), ptr(emb16), stream_ptr()), "time_embed_fwd")
    return emb, emb16, (four, h1, h2)


def time_embed_bwd(demb, saved, W2, dW1, db1, dW2, db2):
    four, h1, h2 = saved
    B, D = demb.shape
    ws1 = torch.empty_like(demb)
    ws2 = torch.empty_like(demb)
    check(load().fdx_time_embed_bwd(ptr(demb), ptr(four), ptr(h1), ptr(h2), ptr(W2), ctypes.c_int(B),
                                    ctypes.c_int(D), ptr(ws1), ptr(ws2), ptr(dW1), ptr(db1), ptr(dW2),
                                    ptr(db2), stream_ptr()), "time_embed_bwd")


def softmax_fwd(S: torch.Tensor, valid: Optional[int] = None) -> torch.Tensor:
    """Row softmax over the first `valid` of the last dim's columns (rest are padding -> 0)."""
    Lp = S.shape[-1]
    L = Lp if valid is None else valid
    P = torch.empty(tuple(S.shape), dtype=torch.bfloat16, device=S.device)
    check(load().fdx_softmax_fwd(ptr(S), ctypes.c_longlong(S.numel() // Lp), ctypes.c_int(L), ctypes.c_int(Lp),
                                 ptr(P), stream_ptr()), "softmax_fwd")
    return P


def softmax_bwd(P: torch.Tensor, dP: torch.Tensor, scale: float, valid: Optional[int] = None) -> torch.Tensor:
    Lp = P.shape[-1]
    L = Lp if valid is None else valid
    dS = torch.empty(tuple(P.shape), dtype=torch.bfloat16, device=P.device)
    check(load().fdx_softmax_bwd(ptr(P), ptr(dP), ctypes.c_longlong(P.numel() // Lp), ctypes.c_int(L),
                                 ctypes.c_int(Lp), ctypes.c_float(scale), ptr(dS), stream_ptr()), "softmax_bwd")
    return dS
