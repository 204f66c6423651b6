"""Restatement of the diffusers 0.14.0 models/vae.py containers (Encoder, Decoder) — **parity unpinned**: diffusers is
not installed, so these containers are restated from its published behaviour, as ResnetBlock2D is in resnet.py.  Their
blocks are the reference's own (e4t/models/unet_2d_blocks.py DownEncoderBlock2D / UNetMidBlock2D / UpDecoderBlock2D,
and through them the reference's AttentionBlock), imported unchanged.  Used only by oracle/gen_golden_vae.py."""
import torch
from torch import nn

from e4t.models.unet_2d_blocks import UNetMidBlock2D, get_down_block, get_up_block


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

    def forward(self, x):
        sample = self.conv_in(x)
        for down_block in self.down_blocks:
            sample = down_block(sample)
        sample = self.mid_block(sample)
        sample = self.conv_act(self.conv_norm_out(sample))
        return self.conv_out(sample)


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
        sample = self.conv_in(z)
        sample = self.mid_block(sample)
        for up_block in self.up_blocks:
            sample = up_block(sample)
        sample = self.conv_act(self.conv_norm_out(sample))
        return self.conv_out(sample)


class DiagonalGaussianDistribution:
    def __init__(self, parameters, deterministic=False):
        self.parameters = parameters
        self.mean, self.logvar = torch.chunk(parameters, 2, dim=1)
        self.logvar = torch.clamp(self.logvar, -30.0, 20.0)
        self.std = torch.exp(0.5 * self.logvar)
        self.var = torch.exp(self.logvar)

    def sample(self, generator=None):
        return self.mean + self.std * torch.randn(self.mean.shape, generator=generator, dtype=self.parameters.dtype)

    def mode(self):
        return self.mean
