"""ORACLE for the SD-v1.x AutoencoderKL (diffusers 0.14 models/vae.py + autoencoder_kl.py) — TEST INFRASTRUCTURE ONLY.

Plain-torch fp32 functional restatement on state dicts with diffusers' key names; runs on CPU or on CUDA tensors (on
CUDA under bf16 autocast it is the stock-torch comparator of tools/vae_bench.py).  Pinned against the reference's own
DownEncoderBlock2D / UNetMidBlock2D / UpDecoderBlock2D / AttentionBlock by oracle/gen_golden_vae.py
(tests/golden/vae_*.pt); the Encoder/Decoder containers around them are restated (see oracle/shim/diffusers/models/vae.py).
"""
import torch
import torch.nn.functional as F

_VAE_BASE = dict(in_channels=3, out_channels=3, act_fn="silu", latent_channels=4, norm_num_groups=32,
                 scaling_factor=0.18215)
# tiny: four levels so that the latent scale factor is 8, as in SD-v1.x (composes with the tiny pipeline test)
TINY_VAE = dict(_VAE_BASE, down_block_types=("DownEncoderBlock2D",) * 4, up_block_types=("UpDecoderBlock2D",) * 4,
                block_out_channels=(64, 64, 128, 128), layers_per_block=1, sample_size=128)
# CompVis/stable-diffusion-v1-4 vae/config.json
SD14_VAE = dict(_VAE_BASE, down_block_types=("DownEncoderBlock2D",) * 4, up_block_types=("UpDecoderBlock2D",) * 4,
                block_out_channels=(128, 256, 512, 512), layers_per_block=2, sample_size=512)


def _conv(s, p, cout, cin, k):
    s[p + "weight"] = (cout, cin, k, k)
    s[p + "bias"] = (cout,)


def _norm(s, p, c):
    s[p + "weight"] = (c,)
    s[p + "bias"] = (c,)


def _res_shapes(s, p, cin, cout):
    _norm(s, p + "norm1.", cin)
    _conv(s, p + "conv1.", cout, cin, 3)
    _norm(s, p + "norm2.", cout)
    _conv(s, p + "conv2.", cout, cout, 3)
    if cin != cout:
        _conv(s, p + "conv_shortcut.", cout, cin, 1)


def _mid_shapes(s, p, c):
    _res_shapes(s, p + "resnets.0.", c, c)
    _norm(s, p + "attentions.0.group_norm.", c)
    for n in ("query", "key", "value", "proj_attn"):
        s[p + f"attentions.0.{n}.weight"] = (c, c)
        s[p + f"attentions.0.{n}.bias"] = (c,)
    _res_shapes(s, p + "resnets.1.", c, c)


def vae_param_shapes(cfg):
    """state-dict key -> shape of diffusers' AutoencoderKL(**cfg)."""
    s = {}
    boc, L, lat = cfg["block_out_channels"], cfg["layers_per_block"], cfg["latent_channels"]
    n = len(boc)
    _conv(s, "encoder.conv_in.", boc[0], cfg["in_channels"], 3)
    cout = boc[0]
    for i in range(n):
        cin, cout = cout, boc[i]
        for j in range(L):
            _res_shapes(s, f"encoder.down_blocks.{i}.resnets.{j}.", cin if j == 0 else cout, cout)
        if i < n - 1:
            _conv(s, f"encoder.down_blocks.{i}.downsamplers.0.conv.", cout, cout, 3)
    _mid_shapes(s, "encoder.mid_block.", boc[-1])
    _norm(s, "encoder.conv_norm_out.", boc[-1])
    _conv(s, "encoder.conv_out.", 2 * lat, boc[-1], 3)
    _conv(s, "decoder.conv_in.", boc[-1], lat, 3)
    _mid_shapes(s, "decoder.mid_block.", boc[-1])
    rev = list(reversed(boc))
    cout = rev[0]
    for i in range(n):
        cin, cout = cout, rev[i]
        for j in range(L + 1):
            _res_shapes(s, f"decoder.up_blocks.{i}.resnets.{j}.", cin if j == 0 else cout, cout)
        if i < n - 1:
            _conv(s, f"decoder.up_blocks.{i}.upsamplers.0.conv.", cout, cout, 3)
    _norm(s, "decoder.conv_norm_out.", boc[0])
    _conv(s, "decoder.conv_out.", cfg["out_channels"], boc[0], 3)
    _conv(s, "quant_conv.", 2 * lat, 2 * lat, 1)
    _conv(s, "post_quant_conv.", lat, lat, 1)
    return s


def _gn(sd, p, x, groups, silu):
    h = F.group_norm(x, groups, sd[p + "weight"], sd[p + "bias"], 1e-6)
    return F.silu(h) if silu else h


def _resnet(sd, p, x, groups):
    """diffusers ResnetBlock2D with temb_channels=None (eps 1e-6, swish)."""
    h = F.conv2d(_gn(sd, p + "norm1.", x, groups, True), sd[p + "conv1.weight"], sd[p + "conv1.bias"], padding=1)
    h = F.conv2d(_gn(sd, p + "norm2.", h, groups, True), sd[p + "conv2.weight"], sd[p + "conv2.bias"], padding=1)
    if p + "conv_shortcut.weight" in sd:
        x = F.conv2d(x, sd[p + "conv_shortcut.weight"], sd[p + "conv_shortcut.bias"])
    return x + h


def attention_block(sd, p, x, groups):
    """AttentionBlock.forward, one head (reference attention.py:125-178)."""
    B, C, H, W = x.shape
    h = _gn(sd, p + "group_norm.", x, groups, False).view(B, C, H * W).transpose(1, 2)
    q = F.linear(h, sd[p + "query.weight"], sd[p + "query.bias"])
    k = F.linear(h, sd[p + "key.weight"], sd[p + "key.bias"])
    v = F.linear(h, sd[p + "value.weight"], sd[p + "value.bias"])
    if q.is_cuda and torch.is_autocast_enabled():
        o = F.scaled_dot_product_attention(q, k, v)            # stock-torch comparator: SDPA
    else:
        o = torch.softmax((q @ k.transpose(-1, -2)) * C ** -0.5, dim=-1) @ v
    o = F.linear(o, sd[p + "proj_attn.weight"], sd[p + "proj_attn.bias"])
    return o.transpose(-1, -2).reshape(B, C, H, W) + x


def _mid(sd, p, x, groups):
    x = _resnet(sd, p + "resnets.0.", x, groups)
    x = attention_block(sd, p + "attentions.0.", x, groups)
    return _resnet(sd, p + "resnets.1.", x, groups)


def vae_encode(sd, cfg, x):
    """AutoencoderKL.encode(x).latent_dist -> (mean, logvar) (logvar clamped to [-30, 20]), NCHW."""
    G, L, n = cfg["norm_num_groups"], cfg["layers_per_block"], len(cfg["block_out_channels"])
    h = F.conv2d(x, sd["encoder.conv_in.weight"], sd["encoder.conv_in.bias"], padding=1)
    for i in range(n):
        for j in range(L):
            h = _resnet(sd, f"encoder.down_blocks.{i}.resnets.{j}.", h, G)
        if i < n - 1:
            p = f"encoder.down_blocks.{i}.downsamplers.0.conv."
            h = F.conv2d(F.pad(h, (0, 1, 0, 1)), sd[p + "weight"], sd[p + "bias"], stride=2)
    h = _mid(sd, "encoder.mid_block.", h, G)
    h = F.conv2d(_gn(sd, "encoder.conv_norm_out.", h, G, True), sd["encoder.conv_out.weight"],
                 sd["encoder.conv_out.bias"], padding=1)
    moments = F.conv2d(h, sd["quant_conv.weight"], sd["quant_conv.bias"])
    mean, logvar = torch.chunk(moments, 2, dim=1)
    return mean, torch.clamp(logvar, -30.0, 20.0)


def vae_decode(sd, cfg, z):
    """AutoencoderKL.decode(z).sample, NCHW."""
    G, L, n = cfg["norm_num_groups"], cfg["layers_per_block"], len(cfg["block_out_channels"])
    z = F.conv2d(z, sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])
    h = F.conv2d(z, sd["decoder.conv_in.weight"], sd["decoder.conv_in.bias"], padding=1)
    h = _mid(sd, "decoder.mid_block.", h, G)
    for i in range(n):
        for j in range(L + 1):
            h = _resnet(sd, f"decoder.up_blocks.{i}.resnets.{j}.", h, G)
        if i < n - 1:
            p = f"decoder.up_blocks.{i}.upsamplers.0.conv."
            h = F.conv2d(F.interpolate(h, scale_factor=2.0, mode="nearest"), sd[p + "weight"], sd[p + "bias"],
                         padding=1)
    return F.conv2d(_gn(sd, "decoder.conv_norm_out.", h, G, True), sd["decoder.conv_out.weight"],
                    sd["decoder.conv_out.bias"], padding=1)

