"""Generate tests/golden/vae_{tiny,sd14}.pt by running the REFERENCE's own VAE blocks (DownEncoderBlock2D,
UNetMidBlock2D, UpDecoderBlock2D and its AttentionBlock, imported unchanged from a checkout of the original project)
inside the restated diffusers 0.14 Encoder / Decoder / AutoencoderKL containers of oracle/shim, on seeded synthetic
weights and inputs:

    E4T_REFERENCE=<checkout> python oracle/gen_golden_vae.py

Each fixture holds the posterior mean / logvar of a seeded image, a row sample of the decode of a seeded latent, the
sha256 of the model's key:shape inventory, and the bf16-autocast error of oracle/vae_oracle.py against fp32 (the
tolerance scale of the CUDA parity tests).  Inputs are re-drawn from the stored seed by the tests.
"""
import hashlib
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if not os.path.isdir(os.environ.get("E4T_REFERENCE", "")):
    raise SystemExit("set E4T_REFERENCE to a checkout of the original e4t-diffusion project")
sys.path[:0] = [os.environ["E4T_REFERENCE"], os.path.join(HERE, "shim"), ROOT]

# the reference's unet_2d_blocks imports AttentionBlock from diffusers; resolve it to the reference's own class
import diffusers.models.attention as _shim_attention  # noqa: E402
from e4t.models.attention import AttentionBlock as _RefAttentionBlock  # noqa: E402

_shim_attention.AttentionBlock = _RefAttentionBlock

from diffusers.models.autoencoder_kl import AutoencoderKL  # noqa: E402  (restated container, reference blocks)
from oracle import e4t_oracle as O  # noqa: E402
from oracle import vae_oracle as V  # noqa: E402
from oracle.golden import sample_rows  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
torch.set_num_threads(os.cpu_count())


def inventory_sha(sd):
    return hashlib.sha256("\n".join(f"{k}:{tuple(sd[k].shape)}" for k in sorted(sd)).encode()).hexdigest()


def inputs(B, hw, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, hw, hw, generator=g) * 2 - 1
    z = torch.randn(B, 4, hw // 8, hw // 8, generator=g)
    return x, z


def case(cfg, B, hw, seed, row_stride):
    kw = {k: v for k, v in cfg.items()}
    m = AutoencoderKL(**kw).eval()
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    mine = V.vae_param_shapes(cfg)
    assert shapes == mine, (set(shapes) ^ set(mine), [k for k in shapes if k in mine and shapes[k] != mine[k]][:5])
    sd = O.synth_state_dict(mine, seed)
    m.load_state_dict(sd, strict=True)
    x, z = inputs(B, hw, seed + 17)
    with torch.no_grad():
        post = m.encode(x)
        dec = m.decode(z)
        with torch.autocast("cpu", dtype=torch.bfloat16):
            mean_a, logvar_a = V.vae_encode(sd, cfg, x)
            dec_a = V.vae_decode(sd, cfg, z)
    err = dict(mean=(mean_a.float() - post.mean).abs().max().item(),
               logvar=(logvar_a.float() - post.logvar).abs().max().item(),
               dec=(dec_a.float() - dec).abs().max().item())
    rec = dict(cfg=cfg, seed=seed, B=B, hw=hw, input_seed=seed + 17, mean=post.mean.clone(),
               logvar=post.logvar.clone(), dec=sample_rows(dec.reshape(-1, dec.shape[-1]), row_stride),
               dec_shape=tuple(dec.shape), sha256=inventory_sha(m.state_dict()), n_keys=len(shapes),
               bf16_err=err)
    print(f"  {cfg['block_out_channels']} hw={hw}: bf16-autocast err {err}")
    return rec


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.save(case(V.TINY_VAE, 2, 128, 5, 2), os.path.join(OUT, "vae_tiny.pt"))
    torch.save(case(V.SD14_VAE, 1, 256, 6, 4), os.path.join(OUT, "vae_sd14.pt"))
    for f in ("vae_tiny.pt", "vae_sd14.pt"):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
