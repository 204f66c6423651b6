"""Restatement of the diffusers 0.14.0 AutoencoderKL container — **parity unpinned** (diffusers is not installed; see
vae.py).  Used only by oracle/gen_golden_vae.py."""
from torch import nn

from diffusers.models.vae import Decoder, DiagonalGaussianDistribution, Encoder


class AutoencoderKL(nn.Module):
    def __init__(self, in_channels=3, out_channels=3, down_block_types=("DownEncoderBlock2D",),
                 up_block_types=("UpDecoderBlock2D",), block_out_channels=(64,), layers_per_block=1, act_fn="silu",
                 latent_channels=4, norm_num_groups=32, sample_size=32, scaling_factor=0.18215):
        super().__init__()
        self.encoder = Encoder(in_channels=in_channels, out_channels=latent_channels, down_block_types=down_block_types,
                               block_out_channels=block_out_channels, layers_per_block=layers_per_block,
                               act_fn=act_fn, norm_num_groups=norm_num_groups, double_z=True)
        self.decoder = Decoder(in_channels=latent_channels, out_channels=out_channels, up_block_types=up_block_types,
                               block_out_channels=block_out_channels, layers_per_block=layers_per_block,
                               norm_num_groups=norm_num_groups, act_fn=act_fn)
        self.quant_conv = nn.Conv2d(2 * latent_channels, 2 * latent_channels, 1)
        self.post_quant_conv = nn.Conv2d(latent_channels, latent_channels, 1)

    def encode(self, x):
        return DiagonalGaussianDistribution(self.quant_conv(self.encoder(x)))

    def decode(self, z):
        return self.decoder(self.post_quant_conv(z))
