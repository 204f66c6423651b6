"""ResnetBlock2D / Downsample2D / Upsample2D — the diffusers==0.14.0 blocks the reference imports un-vendored
(e4t/models/unet_2d_blocks.py:26), rebuilt on channels-last activations:
  GroupNorm(32)+SiLU (fused kernel) -> 3x3 implicit-GEMM conv on tcgen05 with bias + time-embedding row add in the
  epilogue -> GroupNorm+SiLU -> 3x3 conv with bias + shortcut/residual add in the epilogue.
Same parameter names/shapes as diffusers (norm1, conv1, time_emb_proj, norm2, conv2, conv_shortcut; conv)."""
import torch
import torch.nn.functional as F
from torch import nn

from e4t_b200 import functional as FN
from e4t_b200 import ops


def f32(p):
    """fp32 view of a bias / norm parameter: the parameter itself when fp32, else a cached fp32 copy (a model cast with
    .to(dtype=bf16/fp16), e.g. the frozen VAE at pretrain_e4t.py:423)."""
    return p if p is None or p.dtype == torch.float32 else FN.prepared(p, "f32", lambda t: t.float().contiguous())


def conv_w9(conv):
    """(Cout,Cin,3,3) fp32 -> bf16 (9,Cout,Cin), tap = ky*3+kx."""
    return FN.prepared(conv.weight, "w9", lambda w: w.permute(2, 3, 0, 1).reshape(9, w.shape[0], w.shape[1])
                       .to(torch.bfloat16).contiguous())


def conv_w9_dgrad(conv):
    """Taps flipped and (Cout,Cin) transposed: dX = conv3x3(dY, W')."""
    return FN.prepared(conv.weight, "w9d", lambda w: w.flip(2, 3).permute(2, 3, 1, 0).reshape(9, w.shape[1], w.shape[0])
                       .to(torch.bfloat16).contiguous())


def conv3x3(conv, x, rowgroup=None, residual=None):
    return FN.Conv3x3Fn.apply(x, conv_w9(conv), conv_w9_dgrad(conv), f32(conv.bias), rowgroup, residual, conv.weight)


class Upsample2D(nn.Module):
    def __init__(self, channels, use_conv=False, use_conv_transpose=False, out_channels=None, name="conv"):
        super().__init__()
        if not use_conv or use_conv_transpose:
            raise NotImplementedError("SD-v1.x uses nearest x2 + 3x3 conv upsampling only")
        self.channels = channels
        self.out_channels = out_channels or channels
        self.name = name
        conv = nn.Conv2d(self.channels, self.out_channels, 3, padding=1)
        if name == "conv":
            self.conv = conv
        else:
            self.Conv2d_0 = conv

    def forward(self, hidden_states, output_size=None):
        if output_size is not None:
            raise NotImplementedError("output_size forwarding (non power-of-two latents) is not supported")
        conv = self.conv if self.name == "conv" else self.Conv2d_0
        return conv3x3(conv, FN.ResampleFn.apply(hidden_states, 0))


class Downsample2D(nn.Module):
    def __init__(self, channels, use_conv=False, out_channels=None, padding=1, name="conv"):
        super().__init__()
        if not use_conv or padding not in (0, 1):
            raise NotImplementedError("SD-v1.x uses 3x3 stride-2 conv downsampling with padding 1 (UNet) or 0 (VAE)")
        self.channels = channels
        self.out_channels = out_channels or channels
        self.padding = padding
        conv = nn.Conv2d(self.channels, self.out_channels, 3, stride=2, padding=padding)
        if name == "conv":
            self.Conv2d_0 = conv
            self.conv = conv
        else:
            self.conv = conv

    def forward(self, hidden_states):
        # stride-2 convolution computed directly at the output resolution (SURVEY.md §8 a-9)
        c = self.conv
        if self.padding == 0:
            # the VAE encoder's F.pad(x, (0,1,0,1)) + pad-0 conv (frozen VAE, forward only); the bottom/right zeros are
            # the kernel's out-of-bounds fill
            if torch.is_grad_enabled() and (c.weight.requires_grad or hidden_states.requires_grad):
                raise NotImplementedError("Downsample2D(padding=0) is forward-only (the VAE is frozen)")
            return ops.conv3x3_ex(FN._c(hidden_states), conv_w9(c), stride=2, pad=0, bias=f32(c.bias))
        return FN.Conv3x3S2Fn.apply(hidden_states, conv_w9(c), conv_w9_dgrad(c), c.bias, c.weight)


class ResnetBlock2D(nn.Module):
    def __init__(self, *, in_channels, out_channels=None, conv_shortcut=False, dropout=0.0, temb_channels=512,
                 groups=32, groups_out=None, pre_norm=True, eps=1e-6, non_linearity="swish",
                 time_embedding_norm="default", kernel=None, output_scale_factor=1.0, use_in_shortcut=None, up=False,
                 down=False, conv_shortcut_bias=True, conv_2d_out_channels=None):
        super().__init__()
        if not pre_norm or up or down or kernel is not None or time_embedding_norm != "default":
            raise NotImplementedError("only the SD-v1.x ResnetBlock2D configuration is supported")
        if non_linearity not in ("swish", "silu"):
            raise NotImplementedError(non_linearity)
        out_channels = in_channels if out_channels is None else out_channels
        self.in_channels, self.out_channels = in_channels, out_channels
        self.output_scale_factor = output_scale_factor
        groups_out = groups if groups_out is None else groups_out
        self.norm1 = nn.GroupNorm(num_groups=groups, num_channels=in_channels, eps=eps, affine=True)
        self.conv1 = nn.Conv2d(in_channels, out_channels, 3, stride=1, padding=1)
        self.time_emb_proj = nn.Linear(temb_channels, out_channels) if temb_channels is not None else None
        self.norm2 = nn.GroupNorm(num_groups=groups_out, num_channels=out_channels, eps=eps, affine=True)
        self.dropout = nn.Dropout(dropout)
        conv_2d_out_channels = conv_2d_out_channels or out_channels
        self.conv2 = nn.Conv2d(out_channels, conv_2d_out_channels, 3, stride=1, padding=1)
        self.use_in_shortcut = in_channels != conv_2d_out_channels if use_in_shortcut is None else use_in_shortcut
        self.conv_shortcut = None
        if self.use_in_shortcut:
            self.conv_shortcut = nn.Conv2d(in_channels, conv_2d_out_channels, 1, stride=1, padding=0,
                                           bias=conv_shortcut_bias)
        self._temb_row = None  # (id(temb), (B,Cout) fp32) set by UNet2DConditionModel for the batched projection

    def temb_row(self, temb):
        if temb is None or self.time_emb_proj is None:
            return None
        if self._temb_row is not None and self._temb_row[0] is temb:
            return self._temb_row[1]
        # stand-alone use (no UNet-level batched projection): differentiable when the projection is trainable
        with torch.set_grad_enabled(torch.is_grad_enabled() and self.time_emb_proj.weight.requires_grad):
            return F.linear(F.silu(temb.float()), self.time_emb_proj.weight, self.time_emb_proj.bias).contiguous()

    def forward(self, input_tensor, temb):
        if self.output_scale_factor != 1.0:
            raise NotImplementedError("output_scale_factor != 1")
        x = input_tensor
        n1, n2 = self.norm1, self.norm2
        h = FN.GroupNormFn.apply(x, f32(n1.weight), f32(n1.bias), n1.num_groups, n1.eps, True)
        h = conv3x3(self.conv1, h, rowgroup=self.temb_row(temb))
        h = FN.GroupNormFn.apply(h, f32(n2.weight), f32(n2.bias), n2.num_groups, n2.eps, True)
        if self.conv_shortcut is not None:
            B, H, W, C = x.shape
            w = FN.prepared(self.conv_shortcut.weight, "bf16_1x1",
                            lambda t: t.reshape(t.shape[0], t.shape[1]).to(torch.bfloat16).contiguous())
            x = FN.LinearFn.apply(x.view(B, H * W, C), w, f32(self.conv_shortcut.bias), None,
                                  self.conv_shortcut.weight).view(B, H, W, -1)
        return conv3x3(self.conv2, h, residual=x)
