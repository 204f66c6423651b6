"""AutoencoderKL on the sm_100a kernels: wide-image and pad-0 convolutions, the single-head dh = 512 attention core, the
GroupNorm statistics at VAE sizes, module parity against the reference-produced fixtures, the pipeline's decode and the
pre-training step with on-device encode."""
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import e4t_oracle as O
from oracle import vae_oracle as V

pytestmark = pytest.mark.gpu
torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.allow_tf32 = False
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _rel(a, b):
    a = a.float(); b = b.float()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt().clamp_min(1e-12)).item()


def _mk(shape, g, scale=1.0):
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(torch.bfloat16)


def _w9(w):
    return w.permute(2, 3, 0, 1).reshape(9, w.shape[0], w.shape[1]).contiguous()


@pytest.mark.parametrize("W", [256, 512])
@pytest.mark.parametrize("Cin", [128, 256, 512])
def test_wide_conv(W, Cin):
    from e4t_b200 import ops
    Cout, H, B = 128, 8, 2
    g = torch.Generator(device="cuda").manual_seed(W + Cin)
    x = _mk((B, H, W, Cin), g)
    w = _mk((Cout, Cin, 3, 3), g, Cin ** -0.5 / 3)
    bias = torch.randn(Cout, generator=g, device="cuda")
    res = _mk((B, H, W, Cout), g)
    ref = F.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), bias, padding=1) + res.permute(0, 3, 1, 2).float()
    out = ops.conv3x3(x, _w9(w), bias=bias, residual=res, out_dtype=torch.float32)
    assert _rel(out.permute(0, 3, 1, 2), ref) < 2e-3
    out2 = ops.conv3x3_ex(x, _w9(w), stride=1, pad=1, bias=bias, residual=res)
    assert _rel(out2.permute(0, 3, 1, 2), ref) < 4e-3
    # stride 2 / pad 1 at the same input widths (output widths 128 and 256)
    ref2 = F.conv2d(x.permute(0, 3, 1, 2).float(), w.float(), bias, stride=2, padding=1)
    out3 = ops.conv3x3_ex(x, _w9(w), stride=2, pad=1, bias=bias)
    assert _rel(out3.permute(0, 3, 1, 2), ref2) < 4e-3


@pytest.mark.parametrize("Win", [512, 128])
def test_pad0_stride2_conv(Win):
    from e4t_b200 import ops
    B, Hin, Cin, Cout = 2, 16, 128, 128
    g = torch.Generator(device="cuda").manual_seed(Win)
    x = _mk((B, Hin, Win, Cin), g)
    w = _mk((Cout, Cin, 3, 3), g, Cin ** -0.5 / 3)
    bias = torch.randn(Cout, generator=g, device="cuda")
    ref = F.conv2d(F.pad(x.permute(0, 3, 1, 2).float(), (0, 1, 0, 1)), w.float(), bias, stride=2)
    out = ops.conv3x3_ex(x, _w9(w), stride=2, pad=0, bias=bias)
    assert out.shape == (B, Hin // 2, Win // 2, Cout)
    assert _rel(out.permute(0, 3, 1, 2), ref) < 4e-3


@pytest.mark.parametrize("N", [1024, 4096])
def test_attention_core_dh512(N):
    from e4t_b200 import ops
    B, C = 2, 512
    g = torch.Generator(device="cuda").manual_seed(N)
    qkv = _mk((B, N, 3 * C), g)
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    s = ops.gemm(q, k, out_dtype=torch.float32, alpha=C ** -0.5)
    p = ops.softmax_rows(s)
    o = ops.gemm(p, v, b_mn=True)
    ref = torch.softmax(q.float() @ k.float().transpose(1, 2) * C ** -0.5, dim=-1) @ v.float()
    assert _rel(o, ref) < 1e-2
    assert (p.float().sum(-1) - 1).abs().max().item() < 2e-2


def test_softmax_rows_long():
    from e4t_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    s = torch.randn(64, 16384, generator=g, device="cuda") * 4
    p = ops.softmax_rows(s)
    assert (p.float() - torch.softmax(s, -1)).abs().max().item() < 2e-3 * torch.softmax(s, -1).max().item() + 1e-6


def test_groupnorm_silu_vae_size():
    from e4t_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(1)
    C, G = 128, 32
    x = (torch.randn(1, 512, 512, C, generator=g, device="cuda") * 0.5 + 3.0).to(torch.bfloat16)
    gamma = 1 + 0.1 * torch.randn(C, generator=g, device="cuda")
    beta = 0.1 * torch.randn(C, generator=g, device="cuda")
    y, _ = ops.groupnorm_fwd(x, gamma, beta, G, 1e-6, True)
    ref = F.silu(F.group_norm(x.permute(0, 3, 1, 2).double(), G, gamma.double(), beta.double(), 1e-6))
    err = (y.permute(0, 3, 1, 2).double() - ref).abs().max().item()
    assert err < 3e-2, err
    assert _rel(y.permute(0, 3, 1, 2), ref) < 8e-3


def _vae(cfg, seed, dtype=torch.float32):
    from e4t.models.autoencoder_kl import AutoencoderKL
    sd = O.synth_state_dict(V.vae_param_shapes(cfg), seed)
    m = AutoencoderKL(**cfg)
    m.load_state_dict(sd, strict=True)
    return m.to("cuda", dtype=dtype), sd


def _golden_inputs(rec):
    g = torch.Generator().manual_seed(rec["input_seed"])
    B, hw = rec["B"], rec["hw"]
    x = torch.rand(B, 3, hw, hw, generator=g) * 2 - 1
    z = torch.randn(B, 4, hw // 8, hw // 8, generator=g)
    return x, z


@pytest.mark.parametrize("name", ["vae_tiny", "vae_sd14"])
def test_module_parity_vs_golden(name):
    rec = torch.load(os.path.join(GOLD, name + ".pt"))
    m, _ = _vae(rec["cfg"], rec["seed"])
    x, z = _golden_inputs(rec)
    d = m.encode(x.cuda()).latent_dist
    dec = m.decode(z.cuda()).sample
    torch.cuda.synchronize()
    tol = rec["bf16_err"]
    e_mean = (d.mean.cpu() - rec["mean"]).abs().max().item()
    e_logvar = (d.logvar.cpu() - rec["logvar"]).abs().max().item()
    rows = dec.cpu().reshape(-1, dec.shape[-1])[::rec["dec"]["row_stride"]]
    e_dec = (rows - rec["dec"]["rows"]).abs().max().item()
    print(f"[vae {name}] max err mean {e_mean:.3e} logvar {e_logvar:.3e} dec {e_dec:.3e} (bf16-autocast oracle {tol})")
    assert tuple(dec.shape) == rec["dec_shape"] and dec.dtype == torch.float32
    assert e_mean <= 2 * tol["mean"] and e_logvar <= 2 * tol["logvar"] and e_dec <= 2 * tol["dec"]
    assert torch.allclose(d.std, torch.exp(0.5 * d.logvar))


def test_bf16_cast_vae_matches_fp32():
    m32, _ = _vae(V.TINY_VAE, 11)
    m16, _ = _vae(V.TINY_VAE, 11, torch.bfloat16)
    g = torch.Generator().manual_seed(2)
    x = (torch.rand(2, 3, 128, 128, generator=g) * 2 - 1).cuda()
    z = torch.randn(2, 4, 16, 16, generator=g).cuda()
    a, b = m32.encode(x).latent_dist, m16.encode(x.to(torch.bfloat16)).latent_dist
    assert b.mean.dtype == torch.float32
    assert _rel(b.mean, a.mean) < 3e-2 and _rel(b.logvar, a.logvar) < 3e-2
    assert _rel(m16.decode(z).sample, m32.decode(z).sample) < 3e-2


def test_sample_uses_generator_like_diffusers():
    m, _ = _vae(V.TINY_VAE, 12)
    x = torch.zeros(1, 3, 64, 64, device="cuda")
    d = m.encode(x).latent_dist
    s = d.sample(generator=torch.Generator().manual_seed(5))
    eps = torch.randn(d.mean.shape, generator=torch.Generator().manual_seed(5), dtype=torch.float32).cuda()
    assert torch.equal(s, d.mean + d.std * eps)
    assert torch.equal(d.mode(), d.mean)


def test_no_vendor_kernels_in_encode_decode(tmp_path):
    from torch.profiler import ProfilerActivity, profile
    m, _ = _vae(V.TINY_VAE, 13)
    x = torch.rand(2, 3, 128, 128, device="cuda") * 2 - 1
    z = torch.randn(2, 4, 16, 16, device="cuda")
    m.decode(m.encode(x).latent_dist.mean)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.decode(z)
        m.encode(x)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    bad = [n for n in names if any(s in n.lower() for s in ("cudnn", "cublas", "cutlass", "gemm_", "sm90_", "sm100_",
                                                             "conv2d", "convolution", "implicit_gemm", "ampere",
                                                             "nvjet", "xmma", "flash", "fmha"))
           and "e4t_gemm_kernel" not in n]
    assert any("e4t_gemm_kernel" in n for n in names), names
    assert not bad, bad


def test_pipeline_decodes_with_tiny_vae():
    from test_pipeline_gpu import _Tok
    import types
    from e4t.encoder import E4TEncoder
    from e4t.models.modeling_clip import CLIPTextConfig, CLIPTextModel
    from e4t.models.unet_2d_condition import UNet2DConditionModel
    from e4t.pipeline_stable_diffusion_e4t import DDIMScheduler, StableDiffusionE4TPipeline
    ucfg, vcfg, tcfg = O.TINY_UNET, O.VIT_TINY, O.CLIP_TEXT_TINY
    fd = O.pooled_feature_dim(ucfg)
    unet = UNet2DConditionModel(**O.ref_unet_kwargs(ucfg))
    unet.load_state_dict(O.synth_state_dict(O.unet_param_shapes(ucfg), 41))
    enc = E4TEncoder(arch="ViT-tiny-test", word_embedding_dim=tcfg["width"], n_odd_layers=129, unet_feature_dim=fd)
    enc.load_state_dict(O.synth_state_dict(O.encoder_param_shapes(vcfg, fd, tcfg["width"], 129), 42))
    sd_t = O.synth_state_dict(O.text_param_shapes(tcfg), 43)
    text = CLIPTextModel(CLIPTextConfig(vocab_size=tcfg["vocab"] - 1, hidden_size=tcfg["width"],
                                        intermediate_size=tcfg["mlp"], num_hidden_layers=tcfg["layers"],
                                        num_attention_heads=tcfg["heads"]))
    sd_t["text_model.embeddings.token_embedding.weight"] = sd_t["text_model.embeddings.token_embedding.weight"][:-1]
    text.load_state_dict(sd_t)
    vae, sd_v = _vae(V.TINY_VAE, 44)
    cfg = types.SimpleNamespace(placeholder_token="*s", domain_class_token="a", domain_embed_scale=0.1)
    pipe = StableDiffusionE4TPipeline(vae, text.cuda(), _Tok(), unet.cuda(), enc.cuda(), DDIMScheduler(), e4t_config=cfg)
    assert pipe.vae_scale_factor == 8
    g = torch.Generator().manual_seed(3)
    image = torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
    latents = torch.randn(2, 4, 16, 16, generator=g)
    prompt = ["a photo of *s", "a photo of *s"]
    lat = pipe(prompt, num_inference_steps=2, latents=latents.clone(), image=image, output_type="latent").images
    out = pipe(prompt, num_inference_steps=2, latents=latents.clone(), image=image, output_type="np").images
    assert out.shape == (2, 128, 128, 3)
    assert out.min() >= 0.0 and out.max() <= 1.0
    with torch.no_grad():
        ref = V.vae_decode({k: v.cuda() for k, v in sd_v.items()}, V.TINY_VAE, lat.cuda().float() / 0.18215)
    ref = (ref / 2 + 0.5).clamp(0, 1).permute(0, 2, 3, 1).cpu().numpy()
    err = abs(out - ref).max()
    print(f"[pipeline+vae] decoded image max err vs oracle {err:.3e}")
    assert err < 0.05


def _step_models(seed=1):
    from e4t.encoder import E4TEncoder
    from e4t.models.modeling_clip import CLIPTextConfig, CLIPTextModel
    from e4t.models.unet_2d_condition import UNet2DConditionModel
    ucfg, vcfg, tcfg = O.TINY_UNET, O.VIT_TINY, O.CLIP_TEXT_TINY
    fd = O.pooled_feature_dim(ucfg)
    unet = UNet2DConditionModel(**O.ref_unet_kwargs(ucfg))
    unet.load_state_dict(O.synth_state_dict(O.unet_param_shapes(ucfg), seed))
    enc = E4TEncoder(arch="ViT-tiny-test", word_embedding_dim=tcfg["width"], n_odd_layers=129, unet_feature_dim=fd)
    enc.load_state_dict(O.synth_state_dict(O.encoder_param_shapes(vcfg, fd, tcfg["width"], 129), seed + 1))
    text = CLIPTextModel(CLIPTextConfig(vocab_size=tcfg["vocab"], hidden_size=tcfg["width"],
                                        intermediate_size=tcfg["mlp"], num_hidden_layers=tcfg["layers"],
                                        num_attention_heads=tcfg["heads"]))
    text.load_state_dict(O.synth_state_dict(O.text_param_shapes(tcfg), seed + 2))
    return unet.cuda(), enc.cuda(), text.cuda()


@pytest.mark.parametrize("graph", [False, True])
def test_pretrain_step_with_vae_encode(graph):
    """The step with on-device encode computes latents = (mean + std·ε)·scaling_factor from its own posterior (checked
    bitwise on the latents it hands to add_noise), and its loss matches a step fed those latents.  The loss comparison
    is to 1e-3 relative, not bitwise: GroupNorm statistics are summed with fp32 atomics in an order that varies from
    run to run, and through the bf16 activations of two UNet passes that moves the loss by up to ~3e-4 relative on this
    model (eager step 1, and after the warm-up step of a captured graph alike)."""
    from e4t_b200 import engine
    from e4t_b200.engine import PretrainStep
    vae, _ = _vae(V.TINY_VAE, 45)
    batch = {k: v.cuda() for k, v in O.synth_batch(2, seed=42, latent_hw=16, image_hw=128).items()}
    eps = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(7)).cuda()
    with_vae = dict(batch, latent_eps=eps)
    del with_vae["latents"]
    seen = {}
    encode, add_noise = vae.encode, engine.add_noise

    def encode_spy(x, *a, **k):
        out = encode(x, *a, **k)
        seen["d"] = out.latent_dist
        return out

    def add_noise_spy(latents, noise, timesteps, acp):
        if torch.cuda.is_current_stream_capturing():
            return add_noise(latents, noise, timesteps, acp)
        d = seen.pop("d", None)
        if d is not None:     # an encode ran for this step: the latents must be exactly its sample with the batch's ε
            seen["latents"] = latents.clone()
            seen["expected"] = (d.mean + d.std * eps) * vae.config.scaling_factor
        return add_noise(latents, noise, timesteps, acp)

    vae.encode, engine.add_noise = encode_spy, add_noise_spy
    try:
        losses = []
        for v in (vae, None):
            unet, enc, text = _step_models()
            step = PretrainStep(unet, enc, text, O.PLACEHOLDER_ID, class_token_id=320, lr=1e-3,
                                weight_dtype=torch.float32, vae=v)
            b = with_vae if v is not None else dict(batch, latents=seen["latents"])
            if graph:
                b = dict(b, placeholder_idxs=torch.as_tensor(step.placeholder_idxs(b["input_ids"]), device="cuda"))
                step.enable_cuda_graph(b, warmup=1)
            losses.append(step(b)["loss"].item())
            if v is not None:
                assert torch.equal(seen["latents"], seen["expected"])
                seen.pop("d", None)   # (graph: the capture's posterior; no add_noise call consumed it)
            del step
            torch.cuda.synchronize()
    finally:
        engine.add_noise = add_noise
    diff = abs(losses[0] - losses[1])
    print(f"[step+vae] graph={graph} loss with on-device encode {losses[0]:.7f}, with its latents given {losses[1]:.7f}")
    assert diff <= 1e-3 * abs(losses[1]), diff
