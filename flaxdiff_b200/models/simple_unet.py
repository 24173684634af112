"""`Unet` - the reference's UNet denoiser (flaxdiff/models/simple_unet.py:11-222) rebuilt as
an explicit forward / backward program over libfdx kernels.

API kept from the reference (flax.linen module surface):
    model = Unet(output_channels=3, emb_features=256, feature_depths=(64,128,256,512),
                 attention_configs=(None, None, None, {"heads": 8}), num_res_blocks=2,
                 num_middle_res_blocks=1, norm_groups=8, dtype=torch.bfloat16)
    params = model.init(key, x=ones(1,H,W,3), temb=ones(1), textcontext=None)   # {'params': tree}
    y = model.apply(params, x, temb, textcontext)                                  # (B,H,W,3)
Parameter names / layouts are flax's (HWIO conv kernels, (in,out) dense kernels, names as in
pretrained/*/_METADATA): `ConvLayer_0/conv/kernel`, `down_0_residual_0/norm1/scale`, ...

Execution design (B200-first, not a translation of the flax module tree):
  * activations are NHWC bf16; every skip concatenation (simple_unet.py:145,196) is a
    channel *slot* of a pre-allocated buffer, so producers write it in place and the
    concat is free; TMA reads the strided views directly;
  * each ResidualBlock (models/common.py:284-338) is: GN stats -> GN apply+SiLU ->
    conv3x3 [tcgen05] with bias + timestep row-vector fused in the epilogue -> GN stats ->
    apply+SiLU -> conv3x3 with bias + residual fused; the 1x1 residual conv is a GEMM;
  * backward is an explicit tape (no autograd engine): dgrad / wgrad on the same tcgen05
    engine, GroupNorm backward in two streaming passes, gradients accumulated at forks by
    the consumer kernels' accumulate flags;
  * reference quirks kept: res-blocks of a down level keep the incoming width, Upsample
    widths feature_depths[-i] (i=0 -> [0]), attention residual added to the normalised
    tensor (SURVEY.md Appendix A.1-3); `textcontext=None` selects self-attention (A.4).
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional, Sequence

import torch

from .. import ops, utils
from .._lib import GEMM_KK, GEMM_KMN, GEMM_MNMN, FdxError
from .params import FlatParams, ParamLayout, from_tree

BF16 = torch.bfloat16
F32 = torch.float32
RES_EPS = 1e-4      # ResidualBlock.norm_epsilon, models/common.py:271
OUT_EPS = 1e-6      # flax GroupNorm default epsilon for Unet.conv_out_norm (simple_unet.py:26)
ATTN_EPS = 1e-4     # TransformerBlock.norm_epsilon, models/attention.py:319


def _attn_width(d: int) -> int:
    """Stored head width for the fused attention kernels: 32 or 64 (narrower heads are zero-padded).
    FDX_ATTN_PAD64=1 stores every head 64 wide (one head per 128-byte swizzle row)."""
    if os.environ.get("FDX_ATTN_PAD64"):
        return 64
    return 32 if d <= 32 else 64


# 1x1 residual convolutions (ResidualBlock.residual_conv): conv-geometry launches by default - since the transposed
# engine got eight epilogue warps they beat the flat GEMM launch on the HBM-bound shapes
# (profiles/layers_r02_res1x1.txt); FDX_RES1X1_GEMM=1 restores the flat launch.
_RES1X1_GEMM = bool(os.environ.get("FDX_RES1X1_GEMM"))

class _SideStream:
    """Weight-gradient kernels have no consumer before the optimizer step, so the backward pass issues them
    on a second stream: the HBM-bound GroupNorm-backward kernels of the main (data-gradient) chain then
    share the SMs with the tensor-core-bound weight-gradient kernels instead of running after them.
    Tensors handed to `run` are kept alive until `join` (the caching allocator must not recycle them while
    the side stream still reads them).  Works inside CUDA-graph capture (event fork / wait_stream join)."""

    def __init__(self, enabled: bool):
        self.stream = torch.cuda.Stream() if enabled else None
        self.keep: List[torch.Tensor] = []

    def run(self, fn, *tensors):
        if self.stream is None:
            fn()
            return
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self.stream.wait_event(ev)
        with torch.cuda.stream(self.stream):
            fn()
        self.keep.extend(tensors)

    def join(self):
        if self.stream is not None:
            torch.cuda.current_stream().wait_stream(self.stream)
        self.keep.clear()


class Node:
    """An activation view plus (lazily) its gradient view.  `cs` / `coff` / `cs_ok`: the buffer's
    per-image channel-sum workspace (ops.ColStats, shared by a concat buffer and its slots), this view's
    channel offset in it, and whether every channel of this view has been summed by its producer."""
    __slots__ = ("t", "g", "gw", "parent", "cs", "coff", "cs_ok", "kids")

    def __init__(self, t: torch.Tensor, parent: Optional["Node"] = None, coff: int = 0):
        self.t = t
        self.g: Optional[torch.Tensor] = None
        self.gw = False          # gradient buffer holds valid data
        self.parent = parent
        self.cs = None
        self.coff = coff
        self.cs_ok = False
        self.kids: List["Node"] = []
        if parent is not None:
            parent.kids.append(self)

    def colstats(self):
        """(workspace, channel offset) for a producer's epilogue, or None when the images are too small
        for the fused sums (the consumer then runs the statistics kernel)."""
        if self.t.shape[1] * self.t.shape[2] < ops.COLSTATS_MIN_PIXELS:
            return None
        root = self.parent if self.parent is not None else self
        if root.cs is None:
            root.cs = ops.ColStats(root.t.shape[0], root.t.shape[-1], root.t.device)
        self.cs_ok = True
        return (root.cs, self.coff)

    def stats(self, groups: int) -> torch.Tensor:
        """GroupNorm statistics of this tensor: from the producers' epilogue sums when all of them
        contributed, else one pass of fdx_groupnorm_stats."""
        done = all(k.cs_ok for k in self.kids) if self.kids else self.cs_ok
        root = self.parent if self.parent is not None else self
        if done and root.cs is not None:
            return ops.groupnorm_stats_from_cols(root.cs, groups, self.coff, self.t.shape[-1])
        return ops.groupnorm_stats(self.t, groups)

    def norm_apply(self, groups: int, gamma, beta, eps: float, silu: bool):
        """(GroupNorm(+SiLU) of this tensor, its statistics): ONE launch when the producers' epilogues left the
        column sums (fdx_groupnorm_apply_cols), else statistics (from columns or by their own pass) + apply."""
        done = all(k.cs_ok for k in self.kids) if self.kids else self.cs_ok
        root = self.parent if self.parent is not None else self
        if done and root.cs is not None and groups <= 64:
            return ops.groupnorm_apply_cols(self.t, groups, root.cs, self.coff, gamma, beta, eps, silu)
        st = self.stats(groups)
        return ops.groupnorm_apply(self.t, groups, st, gamma, beta, eps, silu), st

    def grad_buf(self) -> torch.Tensor:
        if self.g is None:
            self.g = torch.empty(tuple(self.t.shape), dtype=BF16, device=self.t.device)
        return self.g


class Unet:
    def __init__(self, output_channels: int = 3, emb_features: int = 64 * 4,
                 feature_depths: Sequence[int] = (64, 128, 256, 512),
                 attention_configs: Sequence[Optional[dict]] = ({"heads": 8},) * 4,
                 num_res_blocks: int = 2, num_middle_res_blocks: int = 1, activation="swish",
                 norm_groups: int = 8, dtype=None, precision=None, named_norms: bool = False,
                 context_dim: Optional[int] = None):
        self.output_channels = output_channels
        self.emb_features = emb_features
        self.feature_depths = tuple(feature_depths)
        self.attention_configs = tuple(attention_configs)
        self.num_res_blocks = num_res_blocks
        self.num_middle_res_blocks = num_middle_res_blocks
        self.activation = activation
        self.norm_groups = norm_groups
        self.dtype = dtype
        self.precision = precision
        self.named_norms = named_norms
        # width of `textcontext` (e.g. 768 for CLIP): fixes the to_k / to_v kernel shapes exactly as flax
        # infers them at `init` time.  None = self-attention (`textcontext=None`, SURVEY.md Appendix A.4).
        self.context_dim = context_dim
        if norm_groups <= 0:
            raise FdxError("Unet: norm_groups=0 (RMSNorm blocks) is not on the supported hot path")
        # the kernels implement exactly one activation and one compute type: anything else must fail loudly
        act_name = activation if isinstance(activation, str) else getattr(activation, "__name__", repr(activation))
        if act_name not in ("swish", "silu"):
            raise FdxError(f"Unet: activation {act_name!r} is not supported (the fused kernels implement swish / silu)")
        if dtype is not None and dtype != torch.bfloat16:
            raise FdxError(f"Unet: dtype={dtype} is not supported: the engine computes in bf16 with f32 accumulation "
                           "(pass dtype=None or torch.bfloat16)")
        if output_channels != 3:
            raise FdxError("Unet: output_channels must be 3 (pixel-space configs of BASELINE.json)")
        if len(self.attention_configs) != len(self.feature_depths):
            raise FdxError("Unet: attention_configs must have one entry per level")
        for c in self.attention_configs:
            if c is None:
                continue
            if c.get("flash_attention", False):
                raise FdxError("Unet: flash_attention=True (EfficientAttention / jax pallas) has no counterpart here; "
                               "the fused attention kernel is always used")
            if not c.get("norm_inputs", True):
                raise FdxError("Unet: norm_inputs=False is not supported")
            if not c.get("only_pure_attention", True) and not c.get("explicitly_add_residual", True):
                raise FdxError("Unet: explicitly_add_residual=False is not supported")
        self._n1 = "GroupNorm_0" if named_norms else "norm1"
        self._n2 = "GroupNorm_1" if named_norms else "norm2"
        self._nout = "GroupNorm_0" if named_norms else "conv_out_norm"
        self._layouts: Dict[Optional[int], ParamLayout] = {}
        self._freqs: Dict[str, torch.Tensor] = {}

    # ------------------------------------------------------------------ structure
    def _plan(self):
        """Static structure: list of blocks with channel counts (simple_unet.py:33-222)."""
        fd = self.feature_depths
        L = len(fd)
        blocks = []
        c = fd[0]
        blocks.append(("conv_in", "ConvLayer_0", 3, c))
        skips = [c]
        for i, (dim_out, acfg) in enumerate(zip(fd, self.attention_configs)):
            dim_in = c
            for j in range(self.num_res_blocks):
                blocks.append(("res", f"down_{i}_residual_{j}", c, dim_in))
                c = dim_in
                if acfg is not None and j == self.num_res_blocks - 1:
                    blocks.append(("attn", f"down_{i}_attention_{j}", c, acfg))
                blocks.append(("push", None, c, None))
                skips.append(c)
            if i != L - 1:
                blocks.append(("down", f"down_{i}_downsample", c, dim_out))
                c = dim_out
        mid = fd[-1]
        macfg = self.attention_configs[-1]
        for j in range(self.num_middle_res_blocks):
            blocks.append(("res", f"middle_res1_{j}", c, mid))
            c = mid
            if macfg is not None and j == self.num_middle_res_blocks - 1:
                blocks.append(("attn", f"middle_attention_{j}", c, macfg))
            blocks.append(("res", f"middle_res2_{j}", c, mid))
        for i, (dim_out, acfg) in enumerate(zip(reversed(fd), reversed(self.attention_configs))):
            for j in range(self.num_res_blocks):
                cs = skips.pop()
                blocks.append(("cat", None, c, cs))
                blocks.append(("res", f"up_{i}_residual_{j}", c + cs, dim_out))
                c = dim_out
                if acfg is not None and j == self.num_res_blocks - 1:
                    blocks.append(("attn", f"up_{i}_attention_{j}", c, acfg))
            if i != L - 1:
                up_c = fd[-i] if i > 0 else fd[0]   # feature_depths[-i]; -0 == 0 (quirk, A.1)
                blocks.append(("up", f"up_{i}_upsample", c, up_c))
                c = up_c
        blocks.append(("conv", "ConvLayer_1", c, fd[0]))
        c = fd[0]
        cs = skips.pop()
        blocks.append(("cat", None, c, cs))
        blocks.append(("res", "final_residual", c + cs, fd[0]))
        c = fd[0]
        blocks.append(("out", "ConvLayer_2", c, self.output_channels))
        assert not skips
        return blocks

    def param_specs(self):
        E = self.emb_features
        specs = [("TimeProjection_0/DenseGeneral_0/kernel", (E, E)), ("TimeProjection_0/DenseGeneral_0/bias", (E,)),
                 ("TimeProjection_0/DenseGeneral_1/kernel", (E, E)), ("TimeProjection_0/DenseGeneral_1/bias", (E,))]
        for kind, name, cin, cout in self._plan():
            if kind in ("conv_in", "conv", "out"):
                specs += [(f"{name}/conv/kernel", (3, 3, cin, cout)), (f"{name}/conv/bias", (cout,))]
            elif kind == "res":
                specs += [(f"{name}/{self._n1}/scale", (cin,)), (f"{name}/{self._n1}/bias", (cin,)),
                          (f"{name}/conv1/conv/kernel", (3, 3, cin, cout)), (f"{name}/conv1/conv/bias", (cout,)),
                          (f"{name}/temb_projection/kernel", (E, cout)), (f"{name}/temb_projection/bias", (cout,)),
                          (f"{name}/{self._n2}/scale", (cout,)), (f"{name}/{self._n2}/bias", (cout,)),
                          (f"{name}/conv2/conv/kernel", (3, 3, cout, cout)), (f"{name}/conv2/conv/bias", (cout,))]
                if cin != cout:
                    specs += [(f"{name}/residual_conv/conv/kernel", (1, 1, cin, cout)),
                              (f"{name}/residual_conv/conv/bias", (cout,))]
            elif kind in ("down", "up"):
                specs += [(f"{name}/ConvLayer_0/conv/kernel", (3, 3, cin, cout)),
                          (f"{name}/ConvLayer_0/conv/bias", (cout,))]
            elif kind == "attn":
                # TransformerBlock (models/attention.py:305-380); names as flax generates them
                acfg = cout
                h = acfg["heads"]
                d = cin // h
                cctx = self.context_dim if self.context_dim else cin
                pure = acfg.get("only_pure_attention", True)
                proj = acfg.get("use_projection", False)
                specs += [(f"{name}/RMSNorm_0/scale", (cin,))]
                if proj:
                    specs += [(f"{name}/project_in/kernel", (cin, cin))]

                def mha(base, kdim):
                    return [(f"{base}/to_q/kernel", (cin, h, d)), (f"{base}/to_k/kernel", (kdim, h, d)),
                            (f"{base}/to_v/kernel", (kdim, h, d)), (f"{base}/to_out_0/kernel", (h, d, cin))]
                if pure:
                    specs += mha(f"{name}/Attention/Attention2", cctx)
                else:
                    if acfg.get("use_self_and_cross", True):
                        specs += mha(f"{name}/Attention/Attention1", cin)
                    specs += mha(f"{name}/Attention/Attention2", cctx)
                    specs += [(f"{name}/Attention/ff/net_0/proj/kernel", (cin, 8 * cin)),
                              (f"{name}/Attention/ff/net_0/proj/bias", (8 * cin,)),
                              (f"{name}/Attention/ff/net_2/kernel", (4 * cin, cin)),
                              (f"{name}/Attention/ff/net_2/bias", (cin,))]
                    if acfg.get("use_self_and_cross", True):
                        specs += [(f"{name}/Attention/norm1/scale", (cin,))]
                    specs += [(f"{name}/Attention/norm2/scale", (cin,)), (f"{name}/Attention/norm3/scale", (cin,))]
                if proj:
                    specs += [(f"{name}/project_out/kernel", (cin, cin))]
        specs += [(f"{self._nout}/scale", (self.feature_depths[0],)), (f"{self._nout}/bias", (self.feature_depths[0],))]
        return specs

    def layout(self) -> ParamLayout:
        if self.context_dim not in self._layouts:
            self._layouts[self.context_dim] = ParamLayout(self.param_specs())
        return self._layouts[self.context_dim]

    # ------------------------------------------------------------------ init
    def init(self, key, x=None, temb=None, textcontext=None, device=None) -> FlatParams:
        """flax `model.init(key, **ones)` (trainer/diffusion_trainer.py:107-108): lecun-normal
        kernels (flax default kernel_init), zero biases, unit norm scales."""
        if device is None:
            device = x.device if isinstance(x, torch.Tensor) else torch.device("cuda")
        if isinstance(textcontext, torch.Tensor):
            self.context_dim = int(textcontext.shape[-1])      # flax infers kernel shapes from the inputs
        lay = self.layout()
        flat = torch.zeros(lay.total, dtype=F32, device=device)
        fp = FlatParams(lay, flat)
        if isinstance(key, int):
            key = utils.PRNGKey(key)
        gen = torch.Generator(device=device)
        gen.manual_seed(utils.key_to_seed(tuple(key)))
        for name, t in fp.named.items():
            leaf = name.rsplit('/', 1)[1]
            if leaf == "scale":
                t.fill_(1.0)
            elif leaf == "kernel":
                if t.dim() == 4:
                    fan_in = t.shape[0] * t.shape[1] * t.shape[2]
                elif t.dim() == 3 and name.endswith("to_out_0/kernel"):
                    fan_in = t.shape[0] * t.shape[1]
                else:
                    fan_in = t.shape[0]
                std = math.sqrt(1.0 / fan_in) / 0.87962566103423978
                torch.nn.init.trunc_normal_(t, mean=0.0, std=std, a=-2 * std, b=2 * std, generator=gen)
        return fp

    def _fourier_freqs(self, device) -> torch.Tensor:
        """FourierEmbedding.freqs = jax.random.normal(PRNGKey(42), (features//2,)) * 16
        (models/common.py:101-102): a constant, not a parameter."""
        k = str(device)
        if k not in self._freqs:
            f = utils.normal(utils.PRNGKey(42), self.emb_features // 2) * 16.0
            self._freqs[k] = torch.from_numpy(f.astype("float32")).to(device)
        return self._freqs[k]

    # ------------------------------------------------------------------ public apply
    def _as_flat(self, params, device) -> FlatParams:
        if isinstance(params, FlatParams):
            return params
        return from_tree(self.layout(), params, device)

    def apply(self, params, x: torch.Tensor, temb: torch.Tensor, textcontext=None) -> torch.Tensor:
        """`model.apply(params, x, temb, textcontext)` (general_diffusion_trainer.py:292)."""
        if not x.is_cuda:
            raise FdxError("Unet.apply: CUDA tensors required (no CPU path in flaxdiff_b200)")
        fp = self._as_flat(params, x.device)
        xin = (x if x.dtype == BF16 else x.to(BF16)).contiguous()
        if x.dtype != BF16:                      # f32 -> bf16 through the libfdx cast (the flax module casts too)
            pad = (-x.numel()) % 4
            flat = x.to(F32).contiguous().reshape(-1)
            if pad == 0:
                xin = ops.cast_f32_bf16(flat).view(x.shape)
        out, _ = self.forward(fp, xin, temb, textcontext, save=False)
        return out

    # ------------------------------------------------------------------ forward program
    def forward(self, fp: FlatParams, x_bf16: torch.Tensor, temb: torch.Tensor, textcontext=None,
                save: bool = True):
        """Returns (F f32 [B,H,W,3], tape or None)."""
        has_attn = any(c is not None for c in self.attention_configs)
        ctx16 = None
        if textcontext is not None and has_attn:
            if self.context_dim is None or int(textcontext.shape[-1]) != self.context_dim:
                raise FdxError(f"Unet: textcontext width {tuple(textcontext.shape)} does not match the "
                               f"parameters (context_dim={self.context_dim}); build / init the model with it")
            tc = textcontext
            if tc.shape[0] == 1 and x_bf16.shape[0] > 1:
                tc = tc.expand(x_bf16.shape[0], -1, -1)
            tc = tc.contiguous()
            ctx16 = tc if tc.dtype == BF16 else ops.cast_f32_bf16(tc.to(F32))
        elif textcontext is None and has_attn and self.context_dim is not None:
            raise FdxError("Unet: parameters were built for cross-attention (context_dim set) but "
                           "textcontext is None")
        W = fp.named
        W16 = fp.shadow()
        B, H, Wd, _ = x_bf16.shape
        dev = x_bf16.device
        G = self.norm_groups
        plan = self._plan()
        tape: List[tuple] = []

        # timestep embedding (f32 MLP) -----------------------------------------
        tp = "TimeProjection_0/DenseGeneral_"
        temb = temb.reshape(-1).to(F32)
        if temb.numel() == 1 and B > 1:
            temb = temb.expand(B)
        emb, emb16, temb_saved = ops.time_embed_fwd(
            temb, self._fourier_freqs(dev), W[tp + "0/kernel"], W[tp + "0/bias"], W[tp + "1/kernel"],
            W[tp + "1/bias"])

        # Every ResidualBlock's timestep projection Dense(temb) (common.py:300-305) depends only on the embedding:
        # all of them are issued NOW on a side stream (23 tiny GEMMs that each occupy a handful of SMs for
        # 10-30 us), off the critical path; each block waits for its own row's event before its conv1.
        rows: Dict[str, tuple] = {}
        if not os.environ.get("FDX_NO_SIDE"):
            side = self.__dict__.setdefault("_temb_stream", {}).get(str(dev))
            if side is None:
                side = self._temb_stream[str(dev)] = torch.cuda.Stream(device=dev)
            ev0 = torch.cuda.Event()
            ev0.record(torch.cuda.current_stream())
            side.wait_event(ev0)
            with torch.cuda.stream(side):
                for kind, name, cin, cout in plan:
                    if kind == "res":
                        r = ops.linear_fwd(emb16, W16[f"{name}/temb_projection/kernel"],
                                           bias=W[f"{name}/temb_projection/bias"], out_dtype=F32)
                        ev = torch.cuda.Event()
                        ev.record(side)
                        rows[name] = (r, ev)
        self._rows = rows

        # concat slot buffers: walk the plan once to find (x channels, skip channels, resolution)
        # skip k is produced by the k-th ("conv_in" | "push"); consumed by "cat" in LIFO order.
        res_of_skip, ch_of_skip = [], []
        h, w = H, Wd
        for kind, name, cin, cout in plan:
            if kind == "conv_in":
                res_of_skip.append((h, w)); ch_of_skip.append(cout)
            elif kind == "push":
                res_of_skip.append((h, w)); ch_of_skip.append(cin)
            elif kind == "down":
                h, w = h // 2, w // 2
            elif kind == "up":
                h, w = h * 2, w * 2
        cat_cx = {}
        stack = list(range(len(ch_of_skip)))
        for kind, name, cin, cout in plan:
            if kind == "cat":
                k = stack.pop()
                cat_cx[k] = cin
        cat_nodes = {}
        for k, cx in cat_cx.items():
            hh, ww = res_of_skip[k]
            buf = torch.empty((B, hh, ww, cx + ch_of_skip[k]), dtype=BF16, device=dev)
            parent = Node(buf)
            cat_nodes[k] = (parent, Node(buf[..., :cx], parent, 0), Node(buf[..., cx:], parent, cx))

        def new_node(hh, ww, c):
            return Node(torch.empty((B, hh, ww, c), dtype=BF16, device=dev))

        # which op output must land in which slot: an op's output goes to the x-part of the cat
        # that follows it, or to the skip slot if a "push"/"conv_in" applies to it.
        skip_idx = 0
        pop_stack: List[int] = []
        h, w = H, Wd
        cur: Optional[Node] = None
        n_blocks = len(plan)

        def out_node(idx, hh, ww, c) -> Node:
            """Destination of the op at plan[idx]."""
            nxt = plan[idx + 1][0] if idx + 1 < n_blocks else None
            if nxt == "cat":
                k = pop_stack[-1]
                return cat_nodes[k][1]
            if nxt == "push":
                return cat_nodes[skip_idx][2]
            return new_node(hh, ww, c)

        for idx, (kind, name, cin, cout) in enumerate(plan):
            if kind == "conv_in":
                dst = cat_nodes[0][2]
                ops.conv_in_fwd(x_bf16, W[name + "/conv/kernel"], W[name + "/conv/bias"], dst.t,
                                w_bf16=W16[name + "/conv/kernel"])
                tape.append(("conv_in", name, x_bf16, dst))
                pop_stack.append(0)
                skip_idx = 1
                cur = dst
            elif kind == "push":
                pop_stack.append(skip_idx)
                skip_idx += 1
            elif kind == "cat":
                k = pop_stack.pop()
                cur = cat_nodes[k][0]
            elif kind == "res":
                dst = out_node(idx, h, w, cout)
                rec = self._res_fwd(name, cur, dst, emb16, W, W16, G, RES_EPS)
                tape.append(rec)
                cur = dst
            elif kind == "attn":
                dst = out_node(idx, h, w, cin)
                if cout.get("only_pure_attention", True) and not cout.get("use_projection", False):
                    rec = self._attn_fwd(name, cur, dst, cout["heads"], W, W16, ctx16)
                else:
                    rec = self._tblock_fwd(name, cur, dst, cout, W, W16, ctx16)
                tape.append(rec)
                cur = dst
            elif kind == "down":
                h, w = h // 2, w // 2
                dst = out_node(idx, h, w, cout)
                ops.conv3x3_fwd(cur.t, W16[name + "/ConvLayer_0/conv/kernel"],
                                W[name + "/ConvLayer_0/conv/bias"], out=dst.t, stride=2, colstats=dst.colstats())
                tape.append(("down", name, cur, dst))
                cur = dst
            elif kind == "up":
                # nearest-2x + conv3x3 as four 2x2 parity convolutions of the low-resolution tensor
                # (common.py:210-226); the upsampled activation is never materialised
                h, w = h * 2, w * 2
                dst = out_node(idx, h, w, cout)
                weff = ops.upconv3x3_pack(W[name + "/ConvLayer_0/conv/kernel"])
                cs = dst.colstats() if cur.t.shape[1] * cur.t.shape[2] >= ops.COLSTATS_MIN_PIXELS else None
                ops.upconv3x3_fwd(cur.t, weff, W[name + "/ConvLayer_0/conv/bias"], dst.t, colstats=cs)
                tape.append(("up", name, cur, dst, weff if save else None))
                cur = dst
            elif kind == "conv":
                dst = out_node(idx, h, w, cout)
                ops.conv3x3_fwd(cur.t, W16[name + "/conv/kernel"], W[name + "/conv/bias"], out=dst.t,
                                colstats=dst.colstats())
                tape.append(("conv", name, cur, dst))
                cur = dst
            elif kind == "out":
                a, st = cur.norm_apply(G, W[self._nout + "/scale"], W[self._nout + "/bias"], OUT_EPS, True)
                Fo = ops.conv_out_fwd(a, W[name + "/conv/kernel"], W[name + "/conv/bias"])
                tape.append(("out", name, cur, st, a))
                cur = None
        if not save:
            return Fo, None
        return Fo, {"tape": tape, "emb16": emb16, "temb_saved": temb_saved, "B": B}

    # ------------------------------------------------------------------ blocks: forward
    def _res_fwd(self, name, xin: Node, dst: Node, emb16, W, W16, G, eps):
        x = xin.t
        cin, cout = x.shape[-1], dst.t.shape[-1]
        a1, st1 = xin.norm_apply(G, W[f"{name}/{self._n1}/scale"], W[f"{name}/{self._n1}/bias"], eps, True)
        pre = self._rows.pop(name, None)
        if pre is not None:                       # computed on the side stream at the start of the forward
            row, ev = pre
            torch.cuda.current_stream().wait_event(ev)
            row.record_stream(torch.cuda.current_stream())
        else:
            row = ops.linear_fwd(emb16, W16[f"{name}/temb_projection/kernel"],
                                 bias=W[f"{name}/temb_projection/bias"], out_dtype=F32)
        hnode = Node(torch.empty((x.shape[0], x.shape[1], x.shape[2], cout), dtype=BF16, device=x.device))
        hmid = ops.conv3x3_fwd(a1, W16[f"{name}/conv1/conv/kernel"], W[f"{name}/conv1/conv/bias"], rowvec=row,
                               out=hnode.t, colstats=hnode.colstats())
        a2, st2 = hnode.norm_apply(G, W[f"{name}/{self._n2}/scale"], W[f"{name}/{self._n2}/bias"], eps, True)
        if cin != cout:
            Bn, hh, ww, _ = x.shape
            r = torch.empty((Bn, hh, ww, cout), dtype=BF16, device=x.device)
            if _RES1X1_GEMM:      # round-1 launch: one flat GEMM over all pixels (pixels-as-M engine)
                ops.gemm(GEMM_KMN, x, W16[f"{name}/residual_conv/conv/kernel"], r, Bn * hh * ww, cout, cin,
                         x.stride(2), cout, cout, bias=W[f"{name}/residual_conv/conv/bias"])
            else:                 # conv geometry: eligible for the transposed engine (8 epilogue warps)
                ops.conv1x1_fwd(x, W16[f"{name}/residual_conv/conv/kernel"], W[f"{name}/residual_conv/conv/bias"], out=r)
        else:
            r = x
        ops.conv3x3_fwd(a2, W16[f"{name}/conv2/conv/kernel"], W[f"{name}/conv2/conv/bias"], res=r, out=dst.t,
                        colstats=dst.colstats())
        return ("res", name, xin, dst, st1, a1, hmid, st2, a2)

    @staticmethod
    def _pad_heads(w: torch.Tensor, axis: int, d: int, dp: int) -> torch.Tensor:
        """Zero-pad the head dimension d -> dp (tensor-core tiles need >= 32 columns per head)."""
        if dp == d:
            return w
        pads = [0, 0] * (w.dim() - 1 - axis) + [0, dp - d]
        return torch.nn.functional.pad(w, pads)

    def _attn_fwd(self, name, xin: Node, dst: Node, heads, W, W16, ctx16=None):
        """TransformerBlock(only_pure_attention) (models/attention.py:321-380): xn = RMSNorm(x);
        out = xn + to_out(softmax(q k^T / sqrt(d)) v), keys / values from `textcontext` (cross-attention,
        77 x 768) or from xn itself.  q / k / v / out projections are tcgen05 GEMMs; the attention core is ONE
        fused kernel (fdx_attention_fwd: logits and probabilities stay in TMEM / shared memory).  Heads
        narrower than 32 are zero-padded to 32 (the kernel stores heads 32 or 64 wide).
        FDX_ATTN_UNFUSED=1 selects the round-1 path (separate QK^T / softmax / PV launches)."""
        if os.environ.get("FDX_ATTN_UNFUSED"):
            return self._attn_fwd_unfused(name, xin, dst, heads, W, W16, ctx16)
        x = xin.t
        Bn, hh, ww, C = x.shape
        L = hh * ww
        d = C // heads
        dp = _attn_width(d)
        if d > 64:
            raise FdxError(f"attention: head width {d} > 64 is not supported")
        HD = heads * dp
        base = f"{name}/Attention/Attention2"
        dev = x.device
        xn = ops.rmsnorm_fwd(x, W[f"{name}/RMSNorm_0/scale"], ATTN_EPS)
        x2 = xn.view(Bn * L, C)
        if ctx16 is None:
            ctx, Lk, Cc = xn.view(Bn, L, C), L, C
        else:
            ctx, Lk, Cc = ctx16, ctx16.shape[1], ctx16.shape[2]
        wq = self._pad_heads(W16[f"{base}/to_q/kernel"], 2, d, dp).reshape(C, HD)
        wk = self._pad_heads(W16[f"{base}/to_k/kernel"], 2, d, dp).reshape(Cc, HD)
        wv = self._pad_heads(W16[f"{base}/to_v/kernel"], 2, d, dp).reshape(Cc, HD)
        wo = self._pad_heads(W16[f"{base}/to_out_0/kernel"], 1, d, dp).reshape(HD, C)
        q = ops.linear_fwd(x2, wq).view(Bn, L, HD)
        k = torch.empty((Bn, Lk, HD), dtype=BF16, device=dev)
        v = torch.empty((Bn, Lk, HD), dtype=BF16, device=dev)
        ops.linear_fwd(ctx.reshape(Bn * Lk, Cc), wk, out=k.view(Bn * Lk, HD))
        ops.linear_fwd(ctx.reshape(Bn * Lk, Cc), wv, out=v.view(Bn * Lk, HD))
        o, lse = ops.attention_fwd(q, k, v, heads, dp, d ** -0.5)
        out2 = dst.t
        ops.gemm(GEMM_KMN, o, wo, out2, Bn * L, C, HD, HD, C, out2.stride(2), res=xn, r_ld=C)
        return ("attn", name, xin, dst, heads, xn, q, k, v, lse, o, ctx if ctx16 is not None else None,
                (wq, wk, wv, wo), Lk)

    def _attn_fwd_unfused(self, name, xin: Node, dst: Node, heads, W, W16, ctx16=None):
        """Round-1 attention path (FDX_ATTN_UNFUSED=1): xn = RMSNorm(x);
        out = xn + to_out(softmax(q k^T / sqrt(d)) v); keys/values come from `textcontext`
        (cross-attention, e.g. 77 x 768) or from xn itself (self-attention).  Heads narrower than 32
        and key counts that are not multiples of 32 are zero-padded for the tensor-core tiles."""
        x = xin.t
        Bn, hh, ww, C = x.shape
        L = hh * ww
        d = C // heads
        dp = max(32, d)
        HD = heads * dp
        base = f"{name}/Attention/Attention2"
        dev = x.device
        xn = ops.rmsnorm_fwd(x, W[f"{name}/RMSNorm_0/scale"], ATTN_EPS)
        x2 = xn.view(Bn * L, C)
        if ctx16 is None:
            ctx, Lk, Cc = xn.view(Bn, L, C), L, C
        else:
            ctx, Lk, Cc = ctx16, ctx16.shape[1], ctx16.shape[2]
        Lkp = (Lk + 31) // 32 * 32
        wq = self._pad_heads(W16[f"{base}/to_q/kernel"], 2, d, dp).reshape(C, HD)
        wk = self._pad_heads(W16[f"{base}/to_k/kernel"], 2, d, dp).reshape(Cc, HD)
        wv = self._pad_heads(W16[f"{base}/to_v/kernel"], 2, d, dp).reshape(Cc, HD)
        wo = self._pad_heads(W16[f"{base}/to_out_0/kernel"], 1, d, dp).reshape(HD, C)
        q = ops.linear_fwd(x2, wq)                                        # [B*L, h*dp]
        alloc = torch.zeros if Lkp != Lk else torch.empty
        k = alloc((Bn, Lkp, HD), dtype=BF16, device=dev)
        v = alloc((Bn, Lkp, HD), dtype=BF16, device=dev)
        for w_, o_ in ((wk, k), (wv, v)):
            ops.gemm(GEMM_KMN, ctx, w_, o_, Lk, HD, Cc, Cc, HD, HD, batch2=Bn,
                     a_s=(0, Lk * Cc), d_s=(0, Lkp * HD))
        S = torch.empty((Bn, heads, L, Lkp), dtype=F32, device=dev)
        ops.gemm(GEMM_KK, q, k, S, L, Lkp, dp, HD, HD, Lkp, batch1=heads, batch2=Bn,
                 a_s=(dp, L * HD), b_s=(dp, Lkp * HD), d_s=(L * Lkp, heads * L * Lkp), alpha=d ** -0.5)
        P = ops.softmax_fwd(S, valid=Lk)
        del S
        o = torch.empty((Bn * L, HD), dtype=BF16, device=dev)
        ops.gemm(GEMM_KMN, P, v, o, L, dp, Lkp, Lkp, HD, HD, batch1=heads, batch2=Bn,
                 a_s=(L * Lkp, heads * L * Lkp), b_s=(dp, Lkp * HD), d_s=(dp, L * HD))
        out2 = dst.t
        ops.gemm(GEMM_KMN, o, wo, out2, Bn * L, C, HD, HD, C, out2.stride(2), res=xn, r_ld=C)
        return ("attn_unfused", name, xin, dst, heads, xn, q, k, v, P, o, ctx if ctx16 is not None else None,
                (wq, wk, wv, wo), Lk)


    # ------------------------------------------------------------------ full transformer block (f3)
    def _mha_fwd(self, base, xq: torch.Tensor, ctx: torch.Tensor, heads: int, W16, res: torch.Tensor,
                 out: torch.Tensor):
        """NormalAttention (models/attention.py:117-177) on 2-D token matrices: out = res + to_out(attn(
        to_q(xq), to_k(ctx), to_v(ctx))).  xq [B, L, C], ctx [B, Lk, Cc] bf16; res / out [B*L, C]."""
        Bn, L, C = xq.shape
        Lk, Cc = ctx.shape[1], ctx.shape[2]
        d = C // heads
        dp = _attn_width(d)
        if d > 64:
            raise FdxError(f"attention: head width {d} > 64 is not supported")
        HD = heads * dp
        wq = self._pad_heads(W16[f"{base}/to_q/kernel"], 2, d, dp).reshape(C, HD)
        wk = self._pad_heads(W16[f"{base}/to_k/kernel"], 2, d, dp).reshape(Cc, HD)
        wv = self._pad_heads(W16[f"{base}/to_v/kernel"], 2, d, dp).reshape(Cc, HD)
        wo = self._pad_heads(W16[f"{base}/to_out_0/kernel"], 1, d, dp).reshape(HD, C)
        q = ops.linear_fwd(xq.reshape(Bn * L, C), wq).view(Bn, L, HD)
        k = ops.linear_fwd(ctx.reshape(Bn * Lk, Cc), wk).view(Bn, Lk, HD)
        v = ops.linear_fwd(ctx.reshape(Bn * Lk, Cc), wv).view(Bn, Lk, HD)
        o, lse = ops.attention_fwd(q, k, v, heads, dp, d ** -0.5)
        ops.gemm(GEMM_KMN, o, wo, out, Bn * L, C, HD, HD, C, out.stride(0), res=res, r_ld=res.stride(0))
        return (base, xq, ctx, heads, q, k, v, o, lse, (wq, wk, wv, wo))

    def _mha_bwd(self, saved, dout: torch.Tensor, Gd):
        """-> (d xq [B*L, C], d ctx [B*Lk, Cc]) bf16 given dout = d(out) [B*L, C] (the residual path is the
        caller's); accumulates the four projection-kernel gradients."""
        base, xq, ctx, heads, q, k, v, o, lse, (wq, wk, wv, wo) = saved
        Bn, L, C = xq.shape
        Lk, Cc = ctx.shape[1], ctx.shape[2]
        d = C // heads
        dp = _attn_width(d)
        HD = heads * dp
        M, Mk = Bn * L, Bn * Lk
        dev = xq.device

        def wgrad(pname, src2, dy2, rows, kin, shape_view, sl):
            g = Gd[pname]
            if dp == d:
                ops.gemm(GEMM_MNMN, src2, dy2, g.view(-1, dy2.shape[1]) if shape_view is None else g.view(shape_view),
                         kin, dy2.shape[1], rows, src2.stride(0), dy2.stride(0), dy2.shape[1], atomic=True,
                         reduce_batch=True)
            else:
                tmp = torch.zeros((kin, dy2.shape[1]), dtype=F32, device=dev)
                ops.gemm(GEMM_MNMN, src2, dy2, tmp, kin, dy2.shape[1], rows, src2.stride(0), dy2.stride(0),
                         dy2.shape[1], atomic=True, reduce_batch=True)
                g.add_(tmp.view(sl[0])[sl[1]])

        o2 = o.view(M, HD)
        g_o = Gd[f"{base}/to_out_0/kernel"]
        if dp == d:
            ops.gemm(GEMM_MNMN, o2, dout, g_o.view(HD, C), HD, C, M, HD, dout.stride(0), C, atomic=True,
                     reduce_batch=True)
        else:
            tmp = torch.zeros((HD, C), dtype=F32, device=dev)
            ops.gemm(GEMM_MNMN, o2, dout, tmp, HD, C, M, HD, dout.stride(0), C, atomic=True, reduce_batch=True)
            g_o.add_(tmp.view(heads, dp, C)[:, :d, :])
        do = torch.empty((Bn, L, HD), dtype=BF16, device=dev)
        ops.gemm(GEMM_KK, dout, wo, do, M, HD, C, dout.stride(0), C, HD)
        dq, dk, dv = ops.attention_bwd(q, k, v, o, lse, do, heads, dp, d ** -0.5)
        dq2, dk2, dv2 = dq.view(M, HD), dk.view(Mk, HD), dv.view(Mk, HD)
        xq2, ctx2 = xq.reshape(M, C), ctx.reshape(Mk, Cc)
        pad_view = ((C, heads, dp), (slice(None), slice(None), slice(0, d)))
        wgrad(f"{base}/to_q/kernel", xq2, dq2, M, C, (C, HD), pad_view)
        pad_view_c = ((Cc, heads, dp), (slice(None), slice(None), slice(0, d)))
        wgrad(f"{base}/to_k/kernel", ctx2, dk2, Mk, Cc, (Cc, HD), pad_view_c)
        wgrad(f"{base}/to_v/kernel", ctx2, dv2, Mk, Cc, (Cc, HD), pad_view_c)
        dxq = torch.empty((M, C), dtype=BF16, device=dev)
        ops.gemm(GEMM_KK, dq2, wq, dxq, M, C, HD, HD, HD, C)
        dctx = torch.empty((Mk, Cc), dtype=BF16, device=dev)
        ops.gemm(GEMM_KK, dk2, wk, dctx, Mk, Cc, HD, HD, HD, Cc)
        ops.gemm(GEMM_KK, dv2, wv, dctx, Mk, Cc, HD, HD, HD, Cc, res=dctx, r_ld=Cc)
        return dxq, dctx

    @staticmethod
    def _add2d(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor):
        """out = a + b on [rows, C] bf16 matrices (libfdx fdx_act_add)."""
        v = lambda t: t.unsqueeze(0).unsqueeze(0)
        ops.act_add(v(a), v(b), v(out))

    def _tblock_fwd(self, name, xin: Node, dst: Node, acfg: dict, W, W16, ctx16=None):
        """TransformerBlock with only_pure_attention=False and / or use_projection=True
        (models/attention.py:289-303, 321-380):
            xn = RMSNorm_0(x); px = project_in(xn)
            h = px + Attention1(norm1(px))                       [use_self_and_cross]
            h = h + Attention2(norm2(h), textcontext or px)
            h = h + net_2(GEGLU(net_0.proj(norm3(h))))
            out = xn + project_out(h)
        or, with only_pure_attention, out = xn + project_out(Attention2(project_in(xn), context))."""
        x = xin.t
        Bn, hh, ww, C = x.shape
        L, M = hh * ww, Bn * hh * ww
        heads = acfg["heads"]
        pure = acfg.get("only_pure_attention", True)
        proj = acfg.get("use_projection", False)
        both = acfg.get("use_self_and_cross", True)
        pre = f"{name}/Attention"
        dev = x.device
        xn = ops.rmsnorm_fwd(x, W[f"{name}/RMSNorm_0/scale"], ATTN_EPS)
        xn2 = xn.view(M, C)
        px = ops.linear_fwd(xn2, W16[f"{name}/project_in/kernel"]) if proj else xn2
        ctx = px.view(Bn, L, C) if ctx16 is None else ctx16
        out2 = dst.t.view(M, C) if dst.t.is_contiguous() else None
        sv = {"xn": xn, "px": px, "ctx_is_px": ctx16 is None, "ctx": ctx}
        zeros = None

        def rms(t2, pname):
            return ops.rmsnorm_fwd(t2.view(Bn, hh, ww, C), W[pname], ATTN_EPS).view(M, C)

        if pure:
            zeros = torch.zeros((M, C), dtype=BF16, device=dev)
            h = torch.empty((M, C), dtype=BF16, device=dev)
            sv["a2"] = self._mha_fwd(f"{pre}/Attention2", px.view(Bn, L, C), ctx, heads, W16, zeros, h)
        else:
            h = px
            if both:
                n1 = rms(h, f"{pre}/norm1/scale")
                h1 = torch.empty((M, C), dtype=BF16, device=dev)
                sv["h0"], sv["a1"] = h, self._mha_fwd(f"{pre}/Attention1", n1.view(Bn, L, C), n1.view(Bn, L, C),
                                                      heads, W16, h, h1)
                h = h1
            n2 = rms(h, f"{pre}/norm2/scale")
            h2 = torch.empty((M, C), dtype=BF16, device=dev)
            sv["h1"], sv["a2"] = h, self._mha_fwd(f"{pre}/Attention2", n2.view(Bn, L, C), ctx, heads, W16, h, h2)
            n3 = rms(h2, f"{pre}/norm3/scale")
            u = ops.linear_fwd(n3, W16[f"{pre}/ff/net_0/proj/kernel"], bias=W[f"{pre}/ff/net_0/proj/bias"])
            g = ops.geglu_fwd(u)
            h3 = ops.linear_fwd(g, W16[f"{pre}/ff/net_2/kernel"], bias=W[f"{pre}/ff/net_2/bias"], res=h2)
            sv.update(h2=h2, n3=n3, u=u, g=g)
            h = h3
        sv["h_last"] = h
        # out = xn + project_out(h)   (written straight into the destination slot)
        if proj:
            ops.gemm(GEMM_KMN, h, W16[f"{name}/project_out/kernel"], dst.t, M, C, C, C, C, dst.t.stride(2),
                     res=xn, r_ld=C)
        else:
            ops.act_add(xn, h.view(Bn, hh, ww, C), dst.t)
        return ("tblock", name, xin, dst, acfg, sv)

    def _tblock_bwd(self, rec, W, W16, Gd, want, grad_of):
        _, name, xin, dst, acfg, sv = rec
        x = xin.t
        Bn, hh, ww, C = x.shape
        L, M = hh * ww, Bn * hh * ww
        pure = acfg.get("only_pure_attention", True)
        proj = acfg.get("use_projection", False)
        both = acfg.get("use_self_and_cross", True)
        pre = f"{name}/Attention"
        dev = x.device
        dout = grad_of(dst)                                   # [B,h,w,C], possibly a slot view
        dout2 = dout.reshape(M, C) if dout.is_contiguous() else dout.contiguous().view(M, C)
        xn, px = sv["xn"], sv["px"]

        def lin_wgrad(pname, src2, dy2):
            kin, n = src2.shape[1], dy2.shape[1]
            ops.gemm(GEMM_MNMN, src2, dy2, Gd[pname], kin, n, src2.shape[0], src2.stride(0), dy2.stride(0), n,
                     atomic=True, reduce_batch=True)

        def lin_dgrad(dy2, w_kn, out=None, res=None):
            kin, n = w_kn.shape
            out = out if out is not None else torch.empty((dy2.shape[0], kin), dtype=BF16, device=dev)
            ops.gemm(GEMM_KK, dy2, w_kn, out, dy2.shape[0], kin, n, dy2.stride(0), n, kin,
                     res=res, r_ld=(res.stride(0) if res is not None else 0))
            return out

        def rms_bwd_into(x2, dy2, pname, dx2):
            """dx2 += d/dx RMSNorm(x2) given dy2 (accumulates in place)."""
            v4 = lambda t: t.view(Bn, hh, ww, C)
            ops.rmsnorm_bwd(v4(x2), v4(dy2), W[pname], ATTN_EPS, v4(dx2), Gd[pname], True)

        # out = xn + project_out(h)
        if proj:
            lin_wgrad(f"{name}/project_out/kernel", sv["h_last"], dout2)
            dh = lin_dgrad(dout2, W16[f"{name}/project_out/kernel"])
        else:
            dh = dout2.clone()
        dctx_px = None
        if pure:
            dpx, dctx = self._mha_bwd(sv["a2"], dh, Gd)
            if sv["ctx_is_px"]:
                dctx_px = dctx
        else:
            # h3 = h2 + net_2(g)
            g, u, n3, h2 = sv["g"], sv["u"], sv["n3"], sv["h2"]
            lin_wgrad(f"{pre}/ff/net_2/kernel", g, dh)
            ops.colsum_rows(dh, Gd[f"{pre}/ff/net_2/bias"])
            dg = lin_dgrad(dh, W16[f"{pre}/ff/net_2/kernel"])
            du = ops.geglu_bwd(u, dg)
            lin_wgrad(f"{pre}/ff/net_0/proj/kernel", n3, du)
            ops.colsum_rows(du, Gd[f"{pre}/ff/net_0/proj/bias"])
            dn3 = lin_dgrad(du, W16[f"{pre}/ff/net_0/proj/kernel"])
            rms_bwd_into(h2, dn3, f"{pre}/norm3/scale", dh)            # dh = d h2
            # h2 = h1 + Attention2(norm2(h1), ctx)
            dn2, dctx = self._mha_bwd(sv["a2"], dh, Gd)
            if sv["ctx_is_px"]:
                dctx_px = dctx
            rms_bwd_into(sv["h1"], dn2, f"{pre}/norm2/scale", dh)      # dh = d h1
            if both:
                # h1 = h0 + Attention1(norm1(h0)) with keys / values from the same normed tensor
                dn1, dkv1 = self._mha_bwd(sv["a1"], dh, Gd)
                self._add2d(dn1, dkv1, dn1)
                rms_bwd_into(sv["h0"], dn1, f"{pre}/norm1/scale", dh)  # dh = d h0 = d px
            dpx = dh
        if dctx_px is not None:                                        # context = px (textcontext is None)
            self._add2d(dpx, dctx_px, dpx)
        # px = project_in(xn);  d xn = dout (residual) + d px . W_in^T
        dxn = torch.empty((M, C), dtype=BF16, device=dev)
        if proj:
            lin_wgrad(f"{name}/project_in/kernel", xn.view(M, C), dpx)
            lin_dgrad(dpx, W16[f"{name}/project_in/kernel"], out=dxn, res=dout2)
        else:
            self._add2d(dpx, dout2, dxn)
        dx, acc = want(xin)
        ops.rmsnorm_bwd(x, dxn.view(Bn, hh, ww, C), W[f"{name}/RMSNorm_0/scale"], ATTN_EPS, dx,
                        Gd[f"{name}/RMSNorm_0/scale"], acc)

    # ------------------------------------------------------------------ backward program
    def backward(self, fp: FlatParams, saved: dict, dF: torch.Tensor, grads: FlatParams, on_ready=None):
        """Accumulates d(loss)/d(params) into `grads` (f32, caller zeroes it) given dF = dL/dF.
        `on_ready(lo, streams)`: called after each block's backward has been issued; every parameter
        gradient at flat offset >= lo is final once the work already queued on `streams` has run (the layout
        follows the forward order, the backward walks it from the end) - the data-parallel trainer launches
        its gradient all-reduce buckets from this hook (trainer.GradExchange)."""
        W, W16, Gd = fp.named, fp.shadow(), grads.named
        lows = self._block_offsets(fp.layout) if on_ready is not None else None
        G = self.norm_groups
        emb16 = saved["emb16"]
        B = saved["B"]
        dev = dF.device
        demb = torch.zeros((B, self.emb_features), dtype=F32, device=dev)
        side = _SideStream(not os.environ.get("FDX_NO_SIDE"))

        def want(node: Node):
            """(grad buffer, accumulate?) for a consumer adding into node's gradient."""
            if node.g is None:
                if node.parent is not None:
                    par = node.parent
                    if par.g is None:
                        par.g = torch.empty(tuple(par.t.shape), dtype=BF16, device=dev)
                    off = node.t.storage_offset() - par.t.storage_offset()
                    node.g = par.g[..., off:off + node.t.shape[-1]]
                else:
                    node.grad_buf()
            acc = node.gw
            node.gw = True
            return node.g, acc

        def grad_of(node: Node) -> torch.Tensor:
            if node.g is None or not node.gw:
                raise FdxError("backward: gradient of an activation was never produced")
            return node.g

        def mark_children_written(parent: Node, children):
            for ch in children:
                if ch.g is None:
                    off = ch.t.storage_offset() - parent.t.storage_offset()
                    ch.g = parent.g[..., off:off + ch.t.shape[-1]]
                ch.gw = True

        # parents -> children map for concat buffers
        children: Dict[int, List[Node]] = {}
        for rec in saved["tape"]:
            for obj in rec:
                if isinstance(obj, Node) and obj.parent is not None:
                    lst = children.setdefault(id(obj.parent), [])
                    if all(o is not obj for o in lst):
                        lst.append(obj)

        for rec in reversed(saved["tape"]):
            kind, name = rec[0], rec[1]
            if kind == "out":
                _, _, xin, st, a = rec
                da = torch.empty_like(a)
                col = ops.im2col3(dF, -1, False)          # shared by the data and weight gradients
                ops.conv_out_dgrad(dF, W[name + "/conv/kernel"], da, col=col)
                side.run(lambda: ops.conv_out_wgrad(a, dF, Gd[name + "/conv/kernel"], Gd[name + "/conv/bias"], col=col),
                         col)
                dx, acc = want(xin)
                ops.groupnorm_bwd(xin.t, da, G, st, W[self._nout + "/scale"], W[self._nout + "/bias"], OUT_EPS,
                                  True, Gd[self._nout + "/scale"], Gd[self._nout + "/bias"], dx, acc)
            elif kind == "res":
                self._res_bwd(rec, W, W16, Gd, G, emb16, demb, want, grad_of, side)
                xin = rec[2]
                if id(xin) in children:
                    mark_children_written(xin, children[id(xin)])
            elif kind == "attn":
                self._attn_bwd(rec, W, W16, Gd, want, grad_of)
            elif kind == "attn_unfused":
                self._attn_bwd_unfused(rec, W, W16, Gd, want, grad_of)
            elif kind == "tblock":
                self._tblock_bwd(rec, W, W16, Gd, want, grad_of)
            elif kind == "conv":
                _, _, xin, dst = rec
                dy = grad_of(dst)
                side.run(lambda: (ops.conv3x3_wgrad(xin.t, dy, Gd[name + "/conv/kernel"]),
                                  ops.colsum(dy, False, out=Gd[name + "/conv/bias"])))
                dx, acc = want(xin)
                ops.conv3x3_dgrad(dy, W16[name + "/conv/kernel"], dx, accumulate=acc)
            elif kind == "down":
                _, _, xin, dst = rec
                dy = grad_of(dst)
                kn = name + "/ConvLayer_0/conv/"
                side.run(lambda: (ops.conv3x3_wgrad(xin.t, dy, Gd[kn + "kernel"], stride=2),
                                  ops.colsum(dy, False, out=Gd[kn + "bias"])))
                dx, acc = want(xin)
                ops.conv3x3_dgrad(dy, W16[kn + "kernel"], dx, stride=2, accumulate=acc)
            elif kind == "up":
                _, _, xin, dst, weff = rec
                dy = grad_of(dst)
                kn = name + "/ConvLayer_0/conv/"
                if weff is None:
                    weff = ops.upconv3x3_pack(W[kn + "kernel"])
                side.run(lambda: (ops.upconv3x3_wgrad(xin.t, dy, Gd[kn + "kernel"]),
                                  ops.colsum(dy, False, out=Gd[kn + "bias"])))
                dx, acc = want(xin)
                ops.upconv3x3_dgrad(dy, weff, dx, accumulate=acc)
            elif kind == "conv_in":
                _, _, x_bf16, dst = rec
                dy = grad_of(dst)
                side.run(lambda: ops.conv_in_wgrad(x_bf16, dy, Gd[name + "/conv/kernel"], Gd[name + "/conv/bias"]))
            if on_ready is not None:
                on_ready(lows[name], [torch.cuda.current_stream(), side.stream])
        side.join()
        # timestep-embedding MLP
        tp = "TimeProjection_0/DenseGeneral_"
        ops.time_embed_bwd(demb, saved["temb_saved"], W[tp + "1/kernel"], Gd[tp + "0/kernel"], Gd[tp + "0/bias"],
                           Gd[tp + "1/kernel"], Gd[tp + "1/bias"])

    def _block_offsets(self, layout: ParamLayout) -> Dict[str, int]:
        """First flat offset of each block's parameters (block = first path component of the names)."""
        key = id(layout)
        cache = self.__dict__.setdefault("_lows", {})
        if key not in cache:
            lows: Dict[str, int] = {}
            for pname, (off, _) in layout.table.items():
                head = pname.split('/', 1)[0]
                lows[head] = min(lows.get(head, off), off)
            cache[key] = lows
        return cache[key]

    def _res_bwd(self, rec, W, W16, Gd, G, emb16, demb, want, grad_of, side):
        _, name, xin, dst, st1, a1, hmid, st2, a2 = rec
        x = xin.t
        cin, cout = x.shape[-1], dst.t.shape[-1]
        dout = grad_of(dst)
        Bn, hh, ww, _ = x.shape
        E = emb16.shape[1]
        # conv2
        kres = f"{name}/residual_conv/conv/"
        M = Bn * hh * ww

        def conv2_param_grads():
            ops.conv3x3_wgrad(a2, dout, Gd[f"{name}/conv2/conv/kernel"])
            ops.colsum(dout, False, out=Gd[f"{name}/conv2/conv/bias"])
            if cin != cout:      # the 1x1 residual conv sees the same dout
                ops.gemm(GEMM_MNMN, x, dout, Gd[kres + "kernel"], cin, cout, M, x.stride(2), dout.stride(2), cout,
                         atomic=True, reduce_batch=True)
                Gd[kres + "bias"].copy_(Gd[f"{name}/conv2/conv/bias"])
        side.run(conv2_param_grads)
        # conv2 data gradient -> norm2 + silu backward (first pass fused into the dgrad epilogue).
        # The same pass also emits the per-image / total column sums of dh: the timestep
        # row-vector gradient and the conv1 (= temb_projection) bias gradient
        dh = torch.empty_like(hmid)
        drow = torch.empty((Bn, cout), dtype=F32, device=x.device)
        ops.conv_dgrad_groupnorm_bwd(dout, W16[f"{name}/conv2/conv/kernel"], hmid, G, st2,
                                     W[f"{name}/{self._n2}/scale"], W[f"{name}/{self._n2}/bias"], RES_EPS,
                                     Gd[f"{name}/{self._n2}/scale"], Gd[f"{name}/{self._n2}/bias"], dh, False,
                                     csum_img=drow, csum_tot=Gd[f"{name}/conv1/conv/bias"])

        def conv1_param_grads():
            # timestep projection (its bias gradient = conv1's), then the conv1 weight gradient
            Gd[f"{name}/temb_projection/bias"].copy_(Gd[f"{name}/conv1/conv/bias"])
            drow16 = ops.cast_f32_bf16(drow)
            ops.gemm(GEMM_MNMN, emb16, drow16, Gd[f"{name}/temb_projection/kernel"], E, cout, Bn, E, cout, cout,
                     atomic=True, reduce_batch=True)
            ops.gemm(GEMM_KK, drow16, W16[f"{name}/temb_projection/kernel"], demb, Bn, E, cout, cout, cout, E,
                     atomic=True)
            side.keep.append(drow16)
            ops.conv3x3_wgrad(a1, dh, Gd[f"{name}/conv1/conv/kernel"])
        side.run(conv1_param_grads, dh, drow)
        # conv1 data gradient -> norm1 + silu backward -> dx, joined with the skip gradient (out = h + residual,
        # common.py:334-336) WITHOUT a separate read-modify-write pass over dx:
        #   1x1 residual conv : its data gradient is written (or accumulated) into dx FIRST - a plain store when dx is
        #                       fresh - and the GroupNorm backward adds on top (reads dx at HBM speed instead of
        #                       the GEMM epilogue re-reading it);
        #   identity residual : the GroupNorm backward takes dout as its addend (no act_add launch).
        dx, acc = want(xin)
        gn1 = (dh, W16[f"{name}/conv1/conv/kernel"], x, G, st1, W[f"{name}/{self._n1}/scale"],
               W[f"{name}/{self._n1}/bias"], RES_EPS, Gd[f"{name}/{self._n1}/scale"], Gd[f"{name}/{self._n1}/bias"], dx)
        if cin != cout:
            if _RES1X1_GEMM:
                ops.gemm(GEMM_KK, dout, W16[kres + "kernel"].view(cin, cout), dx, M, cin, cout, dout.stride(2), cout,
                         dx.stride(2), res=dx if acc else None, r_ld=dx.stride(2) if acc else 0)
            else:
                ops.conv1x1_dgrad(dout, W16[kres + "kernel"], dx, accumulate=acc)
            ops.conv_dgrad_groupnorm_bwd(*gn1, True)
        elif acc:
            ops.conv_dgrad_groupnorm_bwd(*gn1, True)
            ops.act_add(dx, dout, dx)
        else:
            ops.conv_dgrad_groupnorm_bwd(*gn1, False, addend=dout)
        del dh

    def _attn_bwd(self, rec, W, W16, Gd, want, grad_of):
        """Backward of _attn_fwd: projection GEMMs around fdx_attention_bwd (dQ / dK / dV with the logits
        recomputed on chip from the saved log-sum-exp)."""
        _, name, xin, dst, heads, xn, q, k, v, lse, o, ctx, (wq, wk, wv, wo), Lk = rec
        x = xin.t
        Bn, hh, ww, C = x.shape
        L = hh * ww
        d = C // heads
        dp = _attn_width(d)
        HD = heads * dp
        cross = ctx is not None
        kv_src = ctx if cross else xn.view(Bn, L, C)
        Cc = kv_src.shape[2]
        base = f"{name}/Attention/Attention2"
        dout = grad_of(dst)
        M = Bn * L
        dev = x.device

        def grad_target(pname, shape_p):
            g = Gd[pname]
            if dp == d:
                return g.view(shape_p), None
            return torch.zeros(shape_p, dtype=F32, device=dev), g

        def finish(tmp, g, axis_view, sl):
            if g is not None:
                g.add_(tmp.view(axis_view)[sl])

        o2 = o.view(M, HD)
        t_o, g_o = grad_target(f"{base}/to_out_0/kernel", (HD, C))
        ops.gemm(GEMM_MNMN, o2, dout, t_o, HD, C, M, HD, dout.stride(2), C, atomic=True, reduce_batch=True)
        finish(t_o, g_o, (heads, dp, C), (slice(None), slice(0, d), slice(None)))
        do = torch.empty((Bn, L, HD), dtype=BF16, device=dev)
        ops.gemm(GEMM_KK, dout, wo, do, M, HD, C, dout.stride(2), C, HD)
        dq, dk, dv = ops.attention_bwd(q, k, v, o, lse, do, heads, dp, d ** -0.5)
        dq2, dk2, dv2 = dq.view(M, HD), dk.view(Bn * Lk, HD), dv.view(Bn * Lk, HD)
        x2 = xn.view(M, C)
        t_q, g_q = grad_target(f"{base}/to_q/kernel", (C, HD))
        ops.gemm(GEMM_MNMN, x2, dq2, t_q, C, HD, M, C, HD, HD, atomic=True, reduce_batch=True)
        finish(t_q, g_q, (C, heads, dp), (slice(None), slice(None), slice(0, d)))
        src2 = kv_src.reshape(Bn * Lk, Cc)
        for nm, dy_ in (("to_k", dk2), ("to_v", dv2)):
            t_w, g_w = grad_target(f"{base}/{nm}/kernel", (Cc, HD))
            ops.gemm(GEMM_MNMN, src2, dy_, t_w, Cc, HD, Bn * Lk, Cc, HD, HD, atomic=True, reduce_batch=True)
            finish(t_w, g_w, (Cc, heads, dp), (slice(None), slice(None), slice(0, d)))
        # d(xn) = dout (residual) + dq Wq^T (+ dk Wk^T + dv Wv^T for self-attention)
        dxn = torch.empty((Bn, hh, ww, C), dtype=BF16, device=dev)
        dxn2 = dxn.view(M, C)
        ops.gemm(GEMM_KK, dq2, wq, dxn2, M, C, HD, HD, HD, C, res=dout, r_ld=dout.stride(2))
        if not cross:
            for dy_, w_ in ((dk2, wk), (dv2, wv)):
                ops.gemm(GEMM_KK, dy_, w_, dxn2, M, C, HD, HD, HD, C, res=dxn2, r_ld=C)
        dx, acc = want(xin)
        ops.rmsnorm_bwd(x, dxn, W[f"{name}/RMSNorm_0/scale"], ATTN_EPS, dx, Gd[f"{name}/RMSNorm_0/scale"], acc)

    def _attn_bwd_unfused(self, rec, W, W16, Gd, want, grad_of):
        _, name, xin, dst, heads, xn, q, k, v, P, o, ctx, (wq, wk, wv, wo), Lk = rec
        x = xin.t
        Bn, hh, ww, C = x.shape
        L = hh * ww
        d = C // heads
        dp = max(32, d)
        HD = heads * dp
        Lkp = k.shape[1]
        cross = ctx is not None
        kv_src = ctx if cross else xn.view(Bn, L, C)
        Cc = kv_src.shape[2]
        base = f"{name}/Attention/Attention2"
        dout = grad_of(dst)                      # [B,h,w,C] view
        M = Bn * L
        dev = x.device
        alpha = d ** -0.5

        def grad_target(pname, shape_p):
            """(buffer to accumulate into, finisher): padded heads go through a scratch buffer."""
            g = Gd[pname]
            if dp == d:
                return g.view(shape_p), None
            return torch.zeros(shape_p, dtype=F32, device=dev), g

        def finish(tmp, g, axis_view, sl):
            if g is not None:
                g.add_(tmp.view(axis_view)[sl])

        # out = xn + o @ Wo
        t_o, g_o = grad_target(f"{base}/to_out_0/kernel", (HD, C))
        ops.gemm(GEMM_MNMN, o, dout, t_o, HD, C, M, HD, dout.stride(2), C, atomic=True, reduce_batch=True)
        finish(t_o, g_o, (heads, dp, C), (slice(None), slice(0, d), slice(None)))
        do = torch.empty((M, HD), dtype=BF16, device=dev)
        ops.gemm(GEMM_KK, dout, wo, do, M, HD, C, dout.stride(2), C, HD)
        # o = P v
        dv = torch.empty((Bn, Lkp, HD), dtype=BF16, device=dev)
        ops.gemm(GEMM_MNMN, P, do, dv, Lkp, dp, L, Lkp, HD, HD, batch1=heads, batch2=Bn,
                 a_s=(L * Lkp, heads * L * Lkp), b_s=(dp, L * HD), d_s=(dp, Lkp * HD))
        dP = torch.empty((Bn, heads, L, Lkp), dtype=F32, device=dev)
        ops.gemm(GEMM_KK, do, v, dP, L, Lkp, dp, HD, HD, Lkp, batch1=heads, batch2=Bn,
                 a_s=(dp, L * HD), b_s=(dp, Lkp * HD), d_s=(L * Lkp, heads * L * Lkp))
        dS = ops.softmax_bwd(P, dP, alpha, valid=Lk)
        del dP
        dq = torch.empty((M, HD), dtype=BF16, device=dev)
        ops.gemm(GEMM_KMN, dS, k, dq, L, dp, Lkp, Lkp, HD, HD, batch1=heads, batch2=Bn,
                 a_s=(L * Lkp, heads * L * Lkp), b_s=(dp, Lkp * HD), d_s=(dp, L * HD))
        dk = torch.empty((Bn, Lkp, HD), dtype=BF16, device=dev)
        ops.gemm(GEMM_MNMN, dS, q, dk, Lkp, dp, L, Lkp, HD, HD, batch1=heads, batch2=Bn,
                 a_s=(L * Lkp, heads * L * Lkp), b_s=(dp, L * HD), d_s=(dp, Lkp * HD))
        del dS
        # projection weight gradients: y = src @ W  ->  dW = src^T dy (reduced over tokens and images)
        x2 = xn.view(M, C)
        t_q, g_q = grad_target(f"{base}/to_q/kernel", (C, HD))
        ops.gemm(GEMM_MNMN, x2, dq, t_q, C, HD, M, C, HD, HD, atomic=True, reduce_batch=True)
        finish(t_q, g_q, (C, heads, dp), (slice(None), slice(None), slice(0, d)))
        for nm, dy_ in (("to_k", dk), ("to_v", dv)):
            t_w, g_w = grad_target(f"{base}/{nm}/kernel", (Cc, HD))
            ops.gemm(GEMM_MNMN, kv_src, dy_, t_w, Cc, HD, Lk, Cc, HD, HD, batch2=Bn,
                     a_s=(0, Lk * Cc), b_s=(0, Lkp * HD), atomic=True, reduce_batch=True)
            finish(t_w, g_w, (Cc, heads, dp), (slice(None), slice(None), slice(0, d)))
        # d(xn) = dout (residual) + dq Wq^T (+ dk Wk^T + dv Wv^T for self-attention)
        dxn = torch.empty((Bn, hh, ww, C), dtype=BF16, device=dev)
        dxn2 = dxn.view(M, C)
        ops.gemm(GEMM_KK, dq, wq, dxn2, M, C, HD, HD, HD, C, res=dout, r_ld=dout.stride(2))
        if not cross:
            for dy_, w_ in ((dk, wk), (dv, wv)):
                # rows of the padded [B, Lkp, HD] buffers map to tokens batch by batch
                ops.gemm(GEMM_KK, dy_, w_, dxn2, L, C, HD, HD, HD, C, batch2=Bn, a_s=(0, Lkp * HD),
                         d_s=(0, L * C), res=dxn2, r_ld=C, r_s=(0, L * C))
        dx, acc = want(xin)
        ops.rmsnorm_bwd(x, dxn, W[f"{name}/RMSNorm_0/scale"], ATTN_EPS, dx, Gd[f"{name}/RMSNorm_0/scale"], acc)
