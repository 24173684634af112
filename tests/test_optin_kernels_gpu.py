"""The opt-in / alternative kernel arrangements (DESIGN.md $6 environment switches) under `-m gpu`:
each is compared with the default arrangement AND with a plain fp32 torch convolution on the same inputs.
  FDX_PAIR=1        CTA-pair (cta_group::2) tcgen05 kernels           fdx_tc.cu PAIR path
  FDX_CONV3=1       halo-sharing forward kernel                        fdx_conv3.cu
  FDX_NO_TCT=1      pixels-as-M engine instead of the transposed one   fdx_tc.cu vs fdx_tct.cu
  FDX_NO_WGRAD9T=1  tap-pair arrangement of the nine-tap weight gradient
  FDX_WGRAD9_V1=1   round-1 nine-tap weight-gradient kernel instead of the kx-in-N one
  FDX_GN_FUSE=1     GroupNorm-backward first pass fused into the dgrad epilogue
"""
import os

import pytest
import torch
import torch.nn.functional as Fnn

from flaxdiff_b200 import ops

pytestmark = pytest.mark.gpu
dev = torch.device("cuda")


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-20)).item()


class env:
    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        for k, v in self.kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _conv_ref(x, w, b=None, res=None):
    y = Fnn.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(3, 2, 0, 1), b, padding=1).permute(0, 2, 3, 1)
    return y if res is None else y + res.float()


SHAPES = [(2, 32, 32, 128, 256), (2, 32, 32, 256, 128), (4, 16, 16, 64, 64), (1, 64, 64, 64, 128), (2, 16, 16, 320, 192)]


@pytest.mark.parametrize("B,H,W,cin,cout", SHAPES + [(2, 48, 32, 64, 192), (1, 16, 16, 128, 320), (3, 32, 16, 384, 64)])
def test_transposed_engine_halo_sharing_vs_per_tap_loads(B, H, W, cin, cout):
    """fdx_tct_kernel<.., HALO=true> (one 16 x 18 pixel box per (kx, K chunk), ky taps as row-offset views)
    against the round-1 per-tap loads (FDX_TCT_HALO=0): bit-identical outputs are NOT expected (the taps are
    accumulated in a different order), both must match fp32 torch."""
    torch.manual_seed(0)
    x = torch.randn(B, H, W, cin, device=dev).bfloat16()
    w = (torch.randn(3, 3, cin, cout, device=dev) / (3 * cin ** 0.5)).bfloat16()
    bias = torch.randn(cout, device=dev)
    res = torch.randn(B, H, W, cout, device=dev).bfloat16()
    dy = torch.randn(B, H, W, cout, device=dev).bfloat16()
    want = _conv_ref(x, w, bias, res)
    xr = x.float().clone().requires_grad_(True)
    _conv_ref(xr, w).backward(dy.float())
    outs = []
    for halo in ("0", None):
        with env(FDX_TCT_HALO=halo):
            y = ops.conv3x3_fwd(x, w, bias, res=res)
            dx = torch.empty_like(x)
            ops.conv3x3_dgrad(dy, w, dx)
            torch.cuda.synchronize()
        assert rel(y, want) < 5e-3 and rel(dx, xr.grad) < 5e-3, halo
        outs.append((y, dx))
    assert rel(outs[1][0], outs[0][0]) < 2e-3 and rel(outs[1][1], outs[0][1]) < 2e-3


@pytest.mark.parametrize("flag", ["FDX_PAIR", "FDX_CONV3", "FDX_NO_TCT"])
@pytest.mark.parametrize("B,H,W,cin,cout", SHAPES)
def test_forward_and_dgrad_variants(flag, B, H, W, cin, cout):
    torch.manual_seed(0)
    x = torch.randn(B, H, W, cin, device=dev).bfloat16()
    w = (torch.randn(3, 3, cin, cout, device=dev) / (3 * cin ** 0.5)).bfloat16()
    bias = torch.randn(cout, device=dev)
    res = torch.randn(B, H, W, cout, device=dev).bfloat16()
    dy = torch.randn(B, H, W, cout, device=dev).bfloat16()
    want = _conv_ref(x, w, bias, res)
    xr = x.float().clone().requires_grad_(True)
    _conv_ref(xr, w).backward(dy.float())
    outs = []
    for on in (False, True):
        with env(**{flag: "1" if on else None}):
            y = ops.conv3x3_fwd(x, w, bias, res=res)
            dx = torch.empty_like(x)
            ops.conv3x3_dgrad(dy, w, dx)
            torch.cuda.synchronize()
        assert rel(y, want) < 5e-3 and rel(dx, xr.grad) < 5e-3, (flag, on)
        outs.append((y, dx))
    assert rel(outs[1][0], outs[0][0]) < 2e-3 and rel(outs[1][1], outs[0][1]) < 2e-3


@pytest.mark.parametrize("flag", ["FDX_NO_WGRAD9T", "FDX_WGRAD9_V1"])
@pytest.mark.parametrize("B,H,W,cin,cout", SHAPES)
def test_weight_gradient_variants(flag, B, H, W, cin, cout):
    torch.manual_seed(0)
    x = torch.randn(B, H, W, cin, device=dev).bfloat16()
    dy = torch.randn(B, H, W, cout, device=dev).bfloat16()
    wr = torch.zeros(3, 3, cin, cout, requires_grad=True, device=dev)
    _conv_ref(x, wr).backward(dy.float())
    for on in (False, True):
        extra = {"FDX_WGRAD9_V1": "1"} if (flag == "FDX_NO_WGRAD9T" and on) else {}
        with env(**{flag: "1" if on else None, **extra}):
            dw = torch.zeros(3, 3, cin, cout, device=dev)
            ops.conv3x3_wgrad(x, dy, dw)
            torch.cuda.synchronize()
        assert rel(dw, wr.grad) < 2e-3, (flag, on, rel(dw, wr.grad))


@pytest.mark.parametrize("B,H,W,cin,cout", [(2, 32, 32, 128, 256), (2, 16, 16, 64, 64), (1, 64, 64, 192, 64)])
def test_groupnorm_backward_fused_into_dgrad(B, H, W, cin, cout):
    """FDX_GN_FUSE=1 (fdx_conv3x3_dgrad_gn + fdx_groupnorm_bwd_dz) against the default two-pass path."""
    torch.manual_seed(0)
    G, eps = 8, 1e-4
    x = torch.randn(B, H, W, cin, device=dev).bfloat16()
    w = (torch.randn(3, 3, cin, cout, device=dev) / (3 * cin ** 0.5)).bfloat16()
    dy = torch.randn(B, H, W, cout, device=dev).bfloat16()
    gamma = 1 + 0.1 * torch.randn(cin, device=dev)
    beta = 0.1 * torch.randn(cin, device=dev)
    st = ops.groupnorm_stats(x, G)
    outs = []
    for fused in (False, True):
        dg, db = torch.zeros(cin, device=dev), torch.zeros(cin, device=dev)
        dx = torch.empty_like(x)
        ops.conv_dgrad_groupnorm_bwd(dy, w, x, G, st, gamma, beta, eps, dg, db, dx, fused=fused)
        torch.cuda.synchronize()
        outs.append((dx, dg, db))
    assert rel(outs[1][0], outs[0][0]) < 2e-2
    assert rel(outs[1][1], outs[0][1]) < 2e-2 and rel(outs[1][2], outs[0][2]) < 2e-2
    # and against autograd through GroupNorm -> SiLU -> conv in fp32
    xr = x.float().clone().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    xn = Fnn.group_norm(xr.permute(0, 3, 1, 2), G, gr, br, eps)
    _conv_ref(Fnn.silu(xn).permute(0, 2, 3, 1), w).backward(dy.float())
    assert rel(outs[0][0], xr.grad) < 2e-2 and rel(outs[0][1], gr.grad) < 2e-2 and rel(outs[0][2], br.grad) < 2e-2

