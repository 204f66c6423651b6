"""AutoencoderKL of diffusers 0.14 (models/autoencoder_kl.py) on the sm_100a kernels, forward only: the frozen VAE of
pretrain_e4t.py:237,597-599 / tuning_e4t.py:102,268-269 (encode) and of the E4T pipeline's decode_latents.  Constructor
kwargs, config (scaling_factor included) and state-dict keys are diffusers', so an SD-v1.x `vae/` folder loads with
`from_pretrained(path, subfolder="vae")`.  The model may be cast with `.to(device, dtype=bf16/fp16)`; the kernels read
bf16 weight copies and fp32 bias / norm copies.

quant_conv (1x1, 8 -> 8) is folded into the encoder's conv_out (exact: both are linear and quant_conv has no spatial
extent).  post_quant_conv is NOT folded into the decoder's conv_in: conv_in zero-pads the transformed latents, which a
folded bias would get wrong on the border pixels; it runs as its own pointwise kernel."""
from dataclasses import dataclass
from typing import Tuple

import torch
from torch import nn

from e4t._mixins import BaseOutput, ConfigMixin, ModelMixin, register_to_config
from e4t.models.resnet import f32
from e4t.models.vae import Decoder, DiagonalGaussianDistribution, Encoder
from e4t_b200 import functional as FN
from e4t_b200 import ops


@dataclass
class AutoencoderKLOutput(BaseOutput):
    latent_dist: DiagonalGaussianDistribution = None


@dataclass
class DecoderOutput(BaseOutput):
    sample: torch.FloatTensor = None


def _check_cuda(x):
    if not x.is_cuda:
        from e4t_b200._lib import E4TError
        raise E4TError("AutoencoderKL runs on the sm_100a kernels only (no CPU fallback): move the model and input to "
                       "a CUDA device")


class AutoencoderKL(ModelMixin, ConfigMixin):
    @register_to_config
    def __init__(self, in_channels: int = 3, out_channels: int = 3,
                 down_block_types: Tuple[str] = ("DownEncoderBlock2D",),
                 up_block_types: Tuple[str] = ("UpDecoderBlock2D",), block_out_channels: Tuple[int] = (64,),
                 layers_per_block: int = 1, act_fn: str = "silu", latent_channels: int = 4, norm_num_groups: int = 32,
                 sample_size: int = 32, scaling_factor: float = 0.18215):
        super().__init__()
        if act_fn not in ("silu", "swish"):
            raise NotImplementedError(f"AutoencoderKL: act_fn {act_fn!r} (SD-v1.x uses silu)")
        self.encoder = Encoder(in_channels=in_channels, out_channels=latent_channels, down_block_types=down_block_types,
                               block_out_channels=block_out_channels, layers_per_block=layers_per_block,
                               act_fn=act_fn, norm_num_groups=norm_num_groups, double_z=True)
        self.decoder = Decoder(in_channels=latent_channels, out_channels=out_channels, up_block_types=up_block_types,
                               block_out_channels=block_out_channels, layers_per_block=layers_per_block,
                               norm_num_groups=norm_num_groups, act_fn=act_fn)
        self.quant_conv = nn.Conv2d(2 * latent_channels, 2 * latent_channels, 1)
        self.post_quant_conv = nn.Conv2d(latent_channels, latent_channels, 1)
        self.use_slicing = False
        self.use_tiling = False

    def _encoder_out_folded(self):
        """conv_out followed by quant_conv as one 3x3 conv: W' = Q·W, b' = Q·b + b_q (fp32)."""
        co, q = self.encoder.conv_out, self.quant_conv
        key = ("quant_fold", co.bias._version, co.bias.data_ptr(), q.weight._version, q.weight.data_ptr(),
               q.bias._version, q.bias.data_ptr())

        def fold(w):
            Q = q.weight.detach().float().flatten(1)                                   # (8, 8)
            wf = torch.einsum("oj,jchw->ochw", Q, w.float()).contiguous()
            bf = (Q @ co.bias.detach().float() + q.bias.detach().float()).contiguous()
            return wf, bf

        return FN.prepared(co.weight, key, fold)

    def _post_quant(self):
        pq = self.post_quant_conv
        return f32(pq.weight).flatten(1).contiguous(), f32(pq.bias)

    @torch.no_grad()
    def encode(self, x: torch.FloatTensor, return_dict: bool = True):
        """x NCHW (B, in_channels, H, W), H and W multiples of 2 ** (len(block_out_channels) - 1)."""
        _check_cuda(x)
        w, b = self._encoder_out_folded()
        moments = ops.conv_out_fwd(self.encoder.features(x), w, b)
        posterior = DiagonalGaussianDistribution(moments)
        if not return_dict:
            return (posterior,)
        return AutoencoderKLOutput(latent_dist=posterior)

    @torch.no_grad()
    def decode(self, z: torch.FloatTensor, return_dict: bool = True):
        """z NCHW (B, latent_channels, h, w) -> image NCHW fp32."""
        _check_cuda(z)
        w, b = self._post_quant()
        dec = self.decoder(ops.pointwise_nchw(z.float().contiguous(), w, b))
        if not return_dict:
            return (dec,)
        return DecoderOutput(sample=dec)

    def forward(self, sample: torch.FloatTensor, sample_posterior: bool = False, return_dict: bool = True,
                generator=None):
        posterior = self.encode(sample).latent_dist
        z = posterior.sample(generator=generator) if sample_posterior else posterior.mode()
        dec = self.decode(z).sample
        if not return_dict:
            return (dec,)
        return DecoderOutput(sample=dec)

    def enable_slicing(self):
        raise NotImplementedError("AutoencoderKL: sliced encode/decode is not supported")

    def enable_tiling(self, use_tiling: bool = True):
        raise NotImplementedError("AutoencoderKL: tiled encode/decode is not supported")
