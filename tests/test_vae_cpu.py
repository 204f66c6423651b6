"""AutoencoderKL without a GPU: the VAE oracle against the fixtures produced by the reference's own blocks, the mirror's
state-dict layout (SD-v1.4 config, save/load round trip, strict loading), and the refusal of CPU tensors."""
import json
import os

import pytest
import torch

from oracle import e4t_oracle as O
from oracle import vae_oracle as V

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# CompVis/stable-diffusion-v1-4 vae/config.json
SD14_VAE_CONFIG = {
    "_class_name": "AutoencoderKL",
    "_diffusers_version": "0.2.2",
    "act_fn": "silu",
    "block_out_channels": [128, 256, 512, 512],
    "down_block_types": ["DownEncoderBlock2D", "DownEncoderBlock2D", "DownEncoderBlock2D", "DownEncoderBlock2D"],
    "in_channels": 3,
    "latent_channels": 4,
    "layers_per_block": 2,
    "norm_num_groups": 32,
    "out_channels": 3,
    "sample_size": 512,
    "up_block_types": ["UpDecoderBlock2D", "UpDecoderBlock2D", "UpDecoderBlock2D", "UpDecoderBlock2D"],
}


def golden_inputs(rec):
    g = torch.Generator().manual_seed(rec["input_seed"])
    B, hw = rec["B"], rec["hw"]
    x = torch.rand(B, 3, hw, hw, generator=g) * 2 - 1
    z = torch.randn(B, 4, hw // 8, hw // 8, generator=g)
    return x, z


def _inventory_sha(sd):
    import hashlib
    return hashlib.sha256("\n".join(f"{k}:{tuple(sd[k].shape)}" for k in sorted(sd)).encode()).hexdigest()


@pytest.mark.parametrize("name", ["vae_tiny", "vae_sd14"])
def test_oracle_matches_golden(name):
    rec = torch.load(os.path.join(GOLD, name + ".pt"))
    cfg = rec["cfg"]
    sd = O.synth_state_dict(V.vae_param_shapes(cfg), rec["seed"])
    x, z = golden_inputs(rec)
    with torch.no_grad():
        mean, logvar = V.vae_encode(sd, cfg, x)
        dec = V.vae_decode(sd, cfg, z)
    assert (mean - rec["mean"]).abs().max().item() < 1e-4
    assert (logvar - rec["logvar"]).abs().max().item() < 1e-4
    assert tuple(dec.shape) == rec["dec_shape"]
    rows = dec.reshape(-1, dec.shape[-1])[::rec["dec"]["row_stride"]]
    assert (rows - rec["dec"]["rows"]).abs().max().item() < 1e-4


@pytest.mark.parametrize("name", ["vae_tiny", "vae_sd14"])
def test_mirror_key_inventory(name):
    from e4t.models.autoencoder_kl import AutoencoderKL
    rec = torch.load(os.path.join(GOLD, name + ".pt"))
    m = AutoencoderKL(**rec["cfg"])
    sd = m.state_dict()
    assert len(sd) == rec["n_keys"]
    assert _inventory_sha(sd) == rec["sha256"]
    assert {k: tuple(v.shape) for k, v in sd.items()} == V.vae_param_shapes(rec["cfg"])


def test_sd14_config_roundtrip_strict(tmp_path):
    from e4t.models.autoencoder_kl import AutoencoderKL
    cfg = {k: v for k, v in SD14_VAE_CONFIG.items() if not k.startswith("_")}
    m = AutoencoderKL(**cfg)
    assert m.config.scaling_factor == 0.18215 and list(m.config.block_out_channels) == [128, 256, 512, 512]
    sd = O.synth_state_dict(V.vae_param_shapes(V.SD14_VAE), 9)
    m.load_state_dict(sd, strict=True)
    # a published vae/ folder: config.json as released (with its "_" keys) + diffusion_pytorch_model.bin
    d = tmp_path / "sd14" / "vae"
    m.save_pretrained(str(d))
    with open(d / "config.json", "w") as f:
        json.dump(SD14_VAE_CONFIG, f)
    m2 = AutoencoderKL.from_pretrained(str(tmp_path / "sd14"), subfolder="vae")
    missing, unexpected = m2.load_state_dict(torch.load(d / "diffusion_pytorch_model.bin"), strict=True)
    assert not missing and not unexpected
    for k, v in m2.state_dict().items():
        assert torch.equal(v, sd[k]), k
    assert 2 ** (len(m2.config.block_out_channels) - 1) == 8


def test_cpu_tensor_raises():
    from e4t.models.autoencoder_kl import AutoencoderKL
    from e4t_b200._lib import E4TError
    m = AutoencoderKL(**V.TINY_VAE)
    with pytest.raises(E4TError):
        m.encode(torch.zeros(1, 3, 64, 64))
    with pytest.raises(E4TError):
        m.decode(torch.zeros(1, 4, 8, 8))


def test_attention_block_multi_head_not_supported():
    from e4t.models.attention import AttentionBlock
    with pytest.raises(NotImplementedError):
        AttentionBlock(64, num_head_channels=32)
    AttentionBlock(64, num_head_channels=None)
    AttentionBlock(64, num_head_channels=64)
