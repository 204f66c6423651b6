"""Encoder / Decoder / DiagonalGaussianDistribution of diffusers 0.14 (models/vae.py) on the sm_100a kernels, forward
only (the VAE is frozen: pretrain_e4t.py:262, used under .detach() at :597-599).  Same module names, config surface and
state-dict keys as diffusers.  Images / latents cross the boundary as NCHW fp32; inside, activations are channels-last
bf16:
  encoder: conv_in (narrow 3 -> C kernel) -> DownEncoderBlock2D x n (pad-0 stride-2 downsample) -> UNetMidBlock2D
           (AttentionBlock) -> GroupNorm+SiLU -> conv_out with quant_conv folded in (narrow C -> 8 kernel)
  decoder: conv_in (4 -> C) -> UNetMidBlock2D -> UpDecoderBlock2D x n -> GroupNorm+SiLU -> conv_out (C -> 3)"""
import torch
from torch import nn

from e4t.models.resnet import f32
from e4t.models.unet_2d_blocks import UNetMidBlock2D, get_down_block, get_up_block
from e4t_b200 import functional as FN
from e4t_b200 import ops


def _w_f32(conv):
    return f32(conv.weight).contiguous()


class Encoder(nn.Module):
    def __init__(self, in_channels=3, out_channels=3, down_block_types=("DownEncoderBlock2D",), block_out_channels=(64,),
                 layers_per_block=2, norm_num_groups=32, act_fn="silu", double_z=True):
        super().__init__()
        self.layers_per_block = layers_per_block
        self.conv_in = nn.Conv2d(in_channels, block_out_channels[0], kernel_size=3, stride=1, padding=1)
        self.mid_block = None
        self.down_blocks = nn.ModuleList([])
        output_channel = block_out_channels[0]
        for i, down_block_type in enumerate(down_block_types):
            input_channel = output_channel
            output_channel = block_out_channels[i]
            is_final_block = i == len(block_out_channels) - 1
            self.down_blocks.append(get_down_block(
                down_block_type, num_layers=self.layers_per_block, in_channels=input_channel,
                out_channels=output_channel, add_downsample=not is_final_block, resnet_eps=1e-6, downsample_padding=0,
                resnet_act_fn=act_fn, resnet_groups=norm_num_groups, attn_num_head_channels=None, temb_channels=None))
        self.mid_block = UNetMidBlock2D(in_channels=block_out_channels[-1], resnet_eps=1e-6, resnet_act_fn=act_fn,
                                        output_scale_factor=1, resnet_time_scale_shift="default",
                                        attn_num_head_channels=None, resnet_groups=norm_num_groups, temb_channels=None)
        self.conv_norm_out = nn.GroupNorm(num_channels=block_out_channels[-1], num_groups=norm_num_groups, eps=1e-6)
        self.conv_act = nn.SiLU()
        conv_out_channels = 2 * out_channels if double_z else out_channels
        self.conv_out = nn.Conv2d(block_out_channels[-1], conv_out_channels, 3, padding=1)

    def features(self, x):
        """x NCHW fp32 -> the conv_out input: GroupNorm+SiLU'd channels-last bf16 (B, h, w, C)."""
        h = ops.conv_in_fwd(x.float().contiguous(), _w_f32(self.conv_in), f32(self.conv_in.bias))
        for blk in self.down_blocks:
            h = blk(h)
        h = self.mid_block(h)
        n = self.conv_norm_out
        return FN.GroupNormFn.apply(h, f32(n.weight), f32(n.bias), n.num_groups, n.eps, True)

    def forward(self, x):
        """x NCHW fp32 -> conv_out output NCHW fp32 (without quant_conv)."""
        return ops.conv_out_fwd(self.features(x), _w_f32(self.conv_out), f32(self.conv_out.bias))


class Decoder(nn.Module):
    def __init__(self, in_channels=3, out_channels=3, up_block_types=("UpDecoderBlock2D",), block_out_channels=(64,),
                 layers_per_block=2, norm_num_groups=32, act_fn="silu"):
        super().__init__()
        self.layers_per_block = layers_per_block
        self.conv_in = nn.Conv2d(in_channels, block_out_channels[-1], kernel_size=3, stride=1, padding=1)
        self.mid_block = None
        self.up_blocks = nn.ModuleList([])
        self.mid_block = UNetMidBlock2D(in_channels=block_out_channels[-1], resnet_eps=1e-6, resnet_act_fn=act_fn,
                                        output_scale_factor=1, resnet_time_scale_shift="default",
                                        attn_num_head_channels=None, resnet_groups=norm_num_groups, temb_channels=None)
        reversed_block_out_channels = list(reversed(block_out_channels))
        output_channel = reversed_block_out_channels[0]
        for i, up_block_type in enumerate(up_block_types):
            prev_output_channel = output_channel
            output_channel = reversed_block_out_channels[i]
            is_final_block = i == len(block_out_channels) - 1
            self.up_blocks.append(get_up_block(
                up_block_type, num_layers=self.layers_per_block + 1, in_channels=prev_output_channel,
                out_channels=output_channel, prev_output_channel=None, add_upsample=not is_final_block,
                resnet_eps=1e-6, resnet_act_fn=act_fn, resnet_groups=norm_num_groups, attn_num_head_channels=None,
                temb_channels=None))
        self.conv_norm_out = nn.GroupNorm(num_channels=block_out_channels[0], num_groups=norm_num_groups, eps=1e-6)
        self.conv_act = nn.SiLU()
        self.conv_out = nn.Conv2d(block_out_channels[0], out_channels, 3, padding=1)

    def forward(self, z):
        """z NCHW fp32 (already through post_quant_conv) -> image NCHW fp32."""
        h = ops.conv_in_fwd(z.float().contiguous(), _w_f32(self.conv_in), f32(self.conv_in.bias))
        h = self.mid_block(h)
        for blk in self.up_blocks:
            h = blk(h)
        n = self.conv_norm_out
        h = FN.GroupNormFn.apply(h, f32(n.weight), f32(n.bias), n.num_groups, n.eps, True)
        return ops.conv_out_fwd(h, _w_f32(self.conv_out), f32(self.conv_out.bias))


class DiagonalGaussianDistribution:
    """diffusers 0.14 DiagonalGaussianDistribution over NCHW fp32 moments (mean | logvar along dim 1)."""

    def __init__(self, parameters, deterministic=False):
        self.parameters = parameters
        self.mean, self.logvar = torch.chunk(parameters, 2, dim=1)
        self.logvar = torch.clamp(self.logvar, -30.0, 20.0)
        self.deterministic = deterministic
        self.std = torch.exp(0.5 * self.logvar)
        self.var = torch.exp(self.logvar)
        if self.deterministic:
            self.var = self.std = torch.zeros_like(self.mean)

    def sample(self, generator=None):
        # diffusers' randn_tensor: drawn on the generator's device, then moved, so a seeded generator gives the same ε
        dev = generator.device if generator is not None else self.parameters.device
        eps = torch.randn(self.mean.shape, generator=generator, device=dev, dtype=torch.float32)
        return self.mean + self.std * eps.to(self.parameters.device)

    def mode(self):
        return self.mean
