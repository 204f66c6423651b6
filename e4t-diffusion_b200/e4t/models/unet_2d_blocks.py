"""UNet blocks used by SD-v1.x — mirror of e4t/models/unet_2d_blocks.py (vendored diffusers 0.14.0):
get_down_block/get_up_block (31-372), UNetMidBlock2DCrossAttn (454-551), CrossAttnDownBlock2D (727-855),
DownBlock2D (858-934), CrossAttnUpBlock2D (1697-1827), UpBlock2D (1830-1901), and the VAE's UNetMidBlock2D
(375-451), DownEncoderBlock2D (937-994), UpDecoderBlock2D (1904-1955).
Activations are channels-last (B,H,W,C) bf16; the skip concat is along the last dim."""
import torch
from torch import nn

from e4t.models.attention import AttentionBlock
from e4t.models.resnet import Downsample2D, ResnetBlock2D, Upsample2D
from e4t.models.transformer_2d import Transformer2DModel


def get_down_block(down_block_type, num_layers, in_channels, out_channels, temb_channels, add_downsample, resnet_eps,
                   resnet_act_fn, attn_num_head_channels, resnet_groups=None, cross_attention_dim=None,
                   downsample_padding=None, dual_cross_attention=False, use_linear_projection=False,
                   only_cross_attention=False, upcast_attention=False, resnet_time_scale_shift="default"):
    down_block_type = down_block_type[7:] if down_block_type.startswith("UNetRes") else down_block_type
    if down_block_type == "DownBlock2D":
        return DownBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                           temb_channels=temb_channels, add_downsample=add_downsample, resnet_eps=resnet_eps,
                           resnet_act_fn=resnet_act_fn, resnet_groups=resnet_groups,
                           downsample_padding=downsample_padding, resnet_time_scale_shift=resnet_time_scale_shift)
    if down_block_type == "CrossAttnDownBlock2D":
        if cross_attention_dim is None:
            raise ValueError("cross_attention_dim must be specified for CrossAttnDownBlock2D")
        return CrossAttnDownBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                    temb_channels=temb_channels, add_downsample=add_downsample, resnet_eps=resnet_eps,
                                    resnet_act_fn=resnet_act_fn, resnet_groups=resnet_groups,
                                    downsample_padding=downsample_padding, cross_attention_dim=cross_attention_dim,
                                    attn_num_head_channels=attn_num_head_channels,
                                    dual_cross_attention=dual_cross_attention,
                                    use_linear_projection=use_linear_projection,
                                    only_cross_attention=only_cross_attention, upcast_attention=upcast_attention,
                                    resnet_time_scale_shift=resnet_time_scale_shift)
    if down_block_type == "DownEncoderBlock2D":
        return DownEncoderBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                  add_downsample=add_downsample, resnet_eps=resnet_eps, resnet_act_fn=resnet_act_fn,
                                  resnet_groups=resnet_groups, downsample_padding=downsample_padding,
                                  resnet_time_scale_shift=resnet_time_scale_shift)
    raise ValueError(f"{down_block_type} is not part of the SD-v1.x E4T path (SURVEY.md §2 #5)")


def get_up_block(up_block_type, num_layers, in_channels, out_channels, prev_output_channel, temb_channels, add_upsample,
                 resnet_eps, resnet_act_fn, attn_num_head_channels, resnet_groups=None, cross_attention_dim=None,
                 dual_cross_attention=False, use_linear_projection=False, only_cross_attention=False,
                 upcast_attention=False, resnet_time_scale_shift="default"):
    up_block_type = up_block_type[7:] if up_block_type.startswith("UNetRes") else up_block_type
    if up_block_type == "UpBlock2D":
        return UpBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                         prev_output_channel=prev_output_channel, temb_channels=temb_channels,
                         add_upsample=add_upsample, resnet_eps=resnet_eps, resnet_act_fn=resnet_act_fn,
                         resnet_groups=resnet_groups, resnet_time_scale_shift=resnet_time_scale_shift)
    if up_block_type == "CrossAttnUpBlock2D":
        if cross_attention_dim is None:
            raise ValueError("cross_attention_dim must be specified for CrossAttnUpBlock2D")
        return CrossAttnUpBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                  prev_output_channel=prev_output_channel, temb_channels=temb_channels,
                                  add_upsample=add_upsample, resnet_eps=resnet_eps, resnet_act_fn=resnet_act_fn,
                                  resnet_groups=resnet_groups, cross_attention_dim=cross_attention_dim,
                                  attn_num_head_channels=attn_num_head_channels,
                                  dual_cross_attention=dual_cross_attention,
                                  use_linear_projection=use_linear_projection,
                                  only_cross_attention=only_cross_attention, upcast_attention=upcast_attention,
                                  resnet_time_scale_shift=resnet_time_scale_shift)
    if up_block_type == "UpDecoderBlock2D":
        return UpDecoderBlock2D(num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                                add_upsample=add_upsample, resnet_eps=resnet_eps, resnet_act_fn=resnet_act_fn,
                                resnet_groups=resnet_groups, resnet_time_scale_shift=resnet_time_scale_shift)
    raise ValueError(f"{up_block_type} is not part of the SD-v1.x E4T path (SURVEY.md §2 #5)")


def _resnet(in_c, out_c, temb_channels, eps, groups, dropout, act, tss, scale, pre_norm):
    return ResnetBlock2D(in_channels=in_c, out_channels=out_c, temb_channels=temb_channels, eps=eps, groups=groups,
                         dropout=dropout, time_embedding_norm=tss, non_linearity=act, output_scale_factor=scale,
                         pre_norm=pre_norm)


def _transformer(heads, out_c, cross_attention_dim, groups, use_linear_projection, only_cross_attention,
                 upcast_attention):
    return Transformer2DModel(heads, out_c // heads, in_channels=out_c, num_layers=1,
                              cross_attention_dim=cross_attention_dim, norm_num_groups=groups,
                              use_linear_projection=use_linear_projection, only_cross_attention=only_cross_attention,
                              upcast_attention=upcast_attention)


class UNetMidBlock2DCrossAttn(nn.Module):
    def __init__(self, in_channels, temb_channels, dropout=0.0, num_layers=1, resnet_eps=1e-6,
                 resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32, resnet_pre_norm=True,
                 attn_num_head_channels=1, output_scale_factor=1.0, cross_attention_dim=1280,
                 dual_cross_attention=False, use_linear_projection=False, upcast_attention=False):
        super().__init__()
        if dual_cross_attention:
            raise NotImplementedError("dual_cross_attention")
        self.has_cross_attention = True
        self.attn_num_head_channels = attn_num_head_channels
        resnet_groups = resnet_groups if resnet_groups is not None else min(in_channels // 4, 32)
        mk = lambda: _resnet(in_channels, in_channels, temb_channels, resnet_eps, resnet_groups, dropout,
                             resnet_act_fn, resnet_time_scale_shift, output_scale_factor, resnet_pre_norm)
        resnets = [mk()]
        attentions = []
        for _ in range(num_layers):
            attentions.append(_transformer(attn_num_head_channels, in_channels, cross_attention_dim, resnet_groups,
                                           use_linear_projection, False, upcast_attention))
            resnets.append(mk())
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, attention_mask=None,
                cross_attention_kwargs=None):
        hidden_states = self.resnets[0](hidden_states, temb)
        for attn, resnet in zip(self.attentions, self.resnets[1:]):
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states,
                                 cross_attention_kwargs=cross_attention_kwargs).sample
            hidden_states = resnet(hidden_states, temb)
        return hidden_states


class CrossAttnDownBlock2D(nn.Module):
    def __init__(self, in_channels, out_channels, temb_channels, dropout=0.0, num_layers=1, resnet_eps=1e-6,
                 resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32, resnet_pre_norm=True,
                 attn_num_head_channels=1, cross_attention_dim=1280, output_scale_factor=1.0, downsample_padding=1,
                 add_downsample=True, dual_cross_attention=False, use_linear_projection=False,
                 only_cross_attention=False, upcast_attention=False):
        super().__init__()
        if dual_cross_attention:
            raise NotImplementedError("dual_cross_attention")
        self.has_cross_attention = True
        self.attn_num_head_channels = attn_num_head_channels
        resnets, attentions = [], []
        for i in range(num_layers):
            in_c = in_channels if i == 0 else out_channels
            resnets.append(_resnet(in_c, out_channels, temb_channels, resnet_eps, resnet_groups, dropout, resnet_act_fn,
                                   resnet_time_scale_shift, output_scale_factor, resnet_pre_norm))
            attentions.append(_transformer(attn_num_head_channels, out_channels, cross_attention_dim, resnet_groups,
                                           use_linear_projection, only_cross_attention, upcast_attention))
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)
        self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                        padding=downsample_padding, name="op")]) if add_downsample else None
        self.gradient_checkpointing = False

    def forward(self, hidden_states, temb=None, encoder_hidden_states=None, attention_mask=None,
                cross_attention_kwargs=None):
        output_states = ()
        for resnet, attn in zip(self.resnets, self.attentions):
            hidden_states = resnet(hidden_states, temb)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states,
                                 cross_attention_kwargs=cross_attention_kwargs).sample
            output_states += (hidden_states,)
        if self.downsamplers is not None:
            for downsampler in self.downsamplers:
                hidden_states = downsampler(hidden_states)
            output_states += (hidden_states,)
        return hidden_states, output_states


class DownBlock2D(nn.Module):
    def __init__(self, in_channels, out_channels, temb_channels, dropout=0.0, num_layers=1, resnet_eps=1e-6,
                 resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32, resnet_pre_norm=True,
                 output_scale_factor=1.0, add_downsample=True, downsample_padding=1):
        super().__init__()
        resnets = []
        for i in range(num_layers):
            in_c = in_channels if i == 0 else out_channels
            resnets.append(_resnet(in_c, out_channels, temb_channels, resnet_eps, resnet_groups, dropout, resnet_act_fn,
                                   resnet_time_scale_shift, output_scale_factor, resnet_pre_norm))
        self.resnets = nn.ModuleList(resnets)
        self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                        padding=downsample_padding, name="op")]) if add_downsample else None
        self.gradient_checkpointing = False

    def forward(self, hidden_states, temb=None):
        output_states = ()
        for resnet in self.resnets:
            hidden_states = resnet(hidden_states, temb)
            output_states += (hidden_states,)
        if self.downsamplers is not None:
            for downsampler in self.downsamplers:
                hidden_states = downsampler(hidden_states)
            output_states += (hidden_states,)
        return hidden_states, output_states


class CrossAttnUpBlock2D(nn.Module):
    def __init__(self, in_channels, out_channels, prev_output_channel, temb_channels, dropout=0.0, num_layers=1,
                 resnet_eps=1e-6, resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32,
                 resnet_pre_norm=True, attn_num_head_channels=1, cross_attention_dim=1280, output_scale_factor=1.0,
                 add_upsample=True, dual_cross_attention=False, use_linear_projection=False,
                 only_cross_attention=False, upcast_attention=False):
        super().__init__()
        if dual_cross_attention:
            raise NotImplementedError("dual_cross_attention")
        self.has_cross_attention = True
        self.attn_num_head_channels = attn_num_head_channels
        resnets, attentions = [], []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(_resnet(resnet_in_channels + res_skip_channels, out_channels, temb_channels, resnet_eps,
                                   resnet_groups, dropout, resnet_act_fn, resnet_time_scale_shift, output_scale_factor,
                                   resnet_pre_norm))
            attentions.append(_transformer(attn_num_head_channels, out_channels, cross_attention_dim, resnet_groups,
                                           use_linear_projection, only_cross_attention, upcast_attention))
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)
        self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)]) \
            if add_upsample else None
        self.gradient_checkpointing = False

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, encoder_hidden_states=None,
                cross_attention_kwargs=None, upsample_size=None, attention_mask=None):
        for resnet, attn in zip(self.resnets, self.attentions):
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=-1)   # channel concat (NHWC)
            hidden_states = resnet(hidden_states, temb)
            hidden_states = attn(hidden_states, encoder_hidden_states=encoder_hidden_states,
                                 cross_attention_kwargs=cross_attention_kwargs).sample
        if self.upsamplers is not None:
            for upsampler in self.upsamplers:
                hidden_states = upsampler(hidden_states, upsample_size)
        return hidden_states


class UpBlock2D(nn.Module):
    def __init__(self, in_channels, prev_output_channel, out_channels, temb_channels, dropout=0.0, num_layers=1,
                 resnet_eps=1e-6, resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32,
                 resnet_pre_norm=True, output_scale_factor=1.0, add_upsample=True):
        super().__init__()
        resnets = []
        for i in range(num_layers):
            res_skip_channels = in_channels if (i == num_layers - 1) else out_channels
            resnet_in_channels = prev_output_channel if i == 0 else out_channels
            resnets.append(_resnet(resnet_in_channels + res_skip_channels, out_channels, temb_channels, resnet_eps,
                                   resnet_groups, dropout, resnet_act_fn, resnet_time_scale_shift, output_scale_factor,
                                   resnet_pre_norm))
        self.resnets = nn.ModuleList(resnets)
        self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)]) \
            if add_upsample else None
        self.gradient_checkpointing = False

    def forward(self, hidden_states, res_hidden_states_tuple, temb=None, upsample_size=None):
        for resnet in self.resnets:
            res_hidden_states = res_hidden_states_tuple[-1]
            res_hidden_states_tuple = res_hidden_states_tuple[:-1]
            hidden_states = torch.cat([hidden_states, res_hidden_states], dim=-1)
            hidden_states = resnet(hidden_states, temb)
        if self.upsamplers is not None:
            for upsampler in self.upsamplers:
                hidden_states = upsampler(hidden_states, upsample_size)
        return hidden_states


class UNetMidBlock2D(nn.Module):
    """The VAE mid-block: resnet, then (AttentionBlock, resnet) x num_layers; no time embedding in the VAE."""

    def __init__(self, in_channels, temb_channels, dropout=0.0, num_layers=1, resnet_eps=1e-6,
                 resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32, resnet_pre_norm=True,
                 add_attention=True, attn_num_head_channels=1, output_scale_factor=1.0):
        super().__init__()
        resnet_groups = resnet_groups if resnet_groups is not None else min(in_channels // 4, 32)
        self.add_attention = add_attention
        mk = lambda: _resnet(in_channels, in_channels, temb_channels, resnet_eps, resnet_groups, dropout,
                             resnet_act_fn, resnet_time_scale_shift, output_scale_factor, resnet_pre_norm)
        resnets = [mk()]
        attentions = []
        for _ in range(num_layers):
            attentions.append(AttentionBlock(in_channels, num_head_channels=attn_num_head_channels,
                                             rescale_output_factor=output_scale_factor, eps=resnet_eps,
                                             norm_num_groups=resnet_groups) if add_attention else None)
            resnets.append(mk())
        self.attentions = nn.ModuleList(attentions)
        self.resnets = nn.ModuleList(resnets)

    def forward(self, hidden_states, temb=None):
        hidden_states = self.resnets[0](hidden_states, temb)
        for attn, resnet in zip(self.attentions, self.resnets[1:]):
            if attn is not None:
                hidden_states = attn(hidden_states)
            hidden_states = resnet(hidden_states, temb)
        return hidden_states


class DownEncoderBlock2D(nn.Module):
    def __init__(self, in_channels, out_channels, dropout=0.0, num_layers=1, resnet_eps=1e-6,
                 resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32, resnet_pre_norm=True,
                 output_scale_factor=1.0, add_downsample=True, downsample_padding=1):
        super().__init__()
        self.resnets = nn.ModuleList([
            _resnet(in_channels if i == 0 else out_channels, out_channels, None, resnet_eps, resnet_groups, dropout,
                    resnet_act_fn, resnet_time_scale_shift, output_scale_factor, resnet_pre_norm)
            for i in range(num_layers)])
        self.downsamplers = nn.ModuleList([Downsample2D(out_channels, use_conv=True, out_channels=out_channels,
                                                        padding=downsample_padding, name="op")]) if add_downsample else None

    def forward(self, hidden_states):
        for resnet in self.resnets:
            hidden_states = resnet(hidden_states, temb=None)
        if self.downsamplers is not None:
            for downsampler in self.downsamplers:
                hidden_states = downsampler(hidden_states)
        return hidden_states


class UpDecoderBlock2D(nn.Module):
    def __init__(self, in_channels, out_channels, dropout=0.0, num_layers=1, resnet_eps=1e-6,
                 resnet_time_scale_shift="default", resnet_act_fn="swish", resnet_groups=32, resnet_pre_norm=True,
                 output_scale_factor=1.0, add_upsample=True):
        super().__init__()
        self.resnets = nn.ModuleList([
            _resnet(in_channels if i == 0 else out_channels, out_channels, None, resnet_eps, resnet_groups, dropout,
                    resnet_act_fn, resnet_time_scale_shift, output_scale_factor, resnet_pre_norm)
            for i in range(num_layers)])
        self.upsamplers = nn.ModuleList([Upsample2D(out_channels, use_conv=True, out_channels=out_channels)]) \
            if add_upsample else None

    def forward(self, hidden_states):
        for resnet in self.resnets:
            hidden_states = resnet(hidden_states, temb=None)
        if self.upsamplers is not None:
            for upsampler in self.upsamplers:
                hidden_states = upsampler(hidden_states)
        return hidden_states
