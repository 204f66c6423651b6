"""Drop-in proof: one E4T pre-training iteration written the way a training script drives the module API (VAE-style
latents, noise and timesteps, a random prompt template, the UNet's encoder half, the E4T encoder, the placeholder word
embedding replaced in place, the text encoder, the full UNet, MSE + embedding regulariser, backward, AdamW), run against
the mirror package with `unet` and `e4t_encoder` wrapped in real torch DistributedDataParallel as accelerate's `prepare`
does, and a torch.optim.AdamW over the E4T parameter selection (encoder head + every WeightOffsets parameter).

DDP raises "Expected to have finished reduction in the prior iteration" on the second step if any requires_grad
parameter did not receive a gradient — the training recipe leaves every base UNet weight trainable, so this test also
proves that the mirror produces all of those gradients."""
import os
import random

import pytest
import torch
import torch.nn.functional as F

from oracle import e4t_oracle as O

pytestmark = pytest.mark.gpu


def _train_iteration(unet, e4t_encoder, text_encoder, optimizer, class_embed, null_context, pixel_values, acp, rnd):
    """One optimiser step; returns (loss, prediction, input ids, placeholder positions)."""
    from e4t_b200.engine import add_noise
    B, dev = pixel_values.shape[0], pixel_values.device
    # stand-in for the frozen VAE (not on the hot path): 4 latent channels at 1/4 resolution, SD scaling factor
    latents = 0.18215 * F.avg_pool2d(torch.cat([pixel_values, pixel_values.mean(1, keepdim=True)], 1), 4)
    noise = torch.randn_like(latents)
    timesteps = torch.randint(0, 1000, (B,), device=dev)
    input_ids, idxs = O.synth_input_ids(rnd.choices(range(len(O.TEMPLATES)), k=B))
    input_ids = input_ids.to(dev)
    token_embeds = text_encoder.get_input_embeddings()(input_ids)
    noisy = add_noise(latents, noise, timesteps, acp)
    down = unet(noisy, timesteps, null_context.expand(B, -1, -1), return_encoder_outputs=True)["down_block_samples"]
    word = class_embed.expand(B, -1) + 0.1 * e4t_encoder(x=pixel_values, unet_down_block_samples=down)
    token_embeds[torch.arange(B, device=dev), torch.tensor(idxs, device=dev)] = word
    context = text_encoder(inputs_embeds=token_embeds)[0]
    pred = unet(noisy, timesteps, context).sample
    loss = F.mse_loss(pred.float(), noise.float()) + 0.01 * word.pow(2).sum()
    loss.backward()
    optimizer.step()
    optimizer.zero_grad()
    return loss, pred, input_ids, idxs


def test_training_loop_body_runs_under_ddp():
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    from e4t.encoder import E4TEncoder
    from e4t.models.modeling_clip import CLIPTextConfig, CLIPTextModel
    from e4t.models.unet_2d_condition import UNet2DConditionModel
    from e4t_b200.engine import ddpm_alphas_cumprod
    ucfg, vcfg, tcfg = O.TINY_UNET, O.VIT_TINY, O.CLIP_TEXT_TINY
    fd = O.pooled_feature_dim(ucfg)
    dev = torch.device("cuda", 0)
    unet = UNet2DConditionModel(**O.ref_unet_kwargs(ucfg))
    unet.load_state_dict(O.synth_state_dict(O.unet_param_shapes(ucfg), 31))
    e4t_encoder = E4TEncoder(arch="ViT-tiny-test", word_embedding_dim=tcfg["width"], n_odd_layers=129, unet_feature_dim=fd)
    e4t_encoder.load_state_dict(O.synth_state_dict(O.encoder_param_shapes(vcfg, fd, tcfg["width"], 129), 32))
    text_encoder = CLIPTextModel(CLIPTextConfig(vocab_size=tcfg["vocab"], hidden_size=tcfg["width"],
                                                intermediate_size=tcfg["mlp"], num_hidden_layers=tcfg["layers"],
                                                num_attention_heads=tcfg["heads"]))
    text_encoder.load_state_dict(O.synth_state_dict(O.text_param_shapes(tcfg), 33))
    text_encoder.requires_grad_(False)
    unet, e4t_encoder, text_encoder = unet.to(dev), e4t_encoder.to(dev), text_encoder.to(dev)
    unet.train(); e4t_encoder.train()
    # trainable: the encoder head and the WeightOffsets parameters, AdamW with the training recipe's settings
    optim_params = [p for p in e4t_encoder.parameters() if p.requires_grad]
    for n, p in unet.named_parameters():
        if "wo" in n:
            optim_params += [p]
    optimizer = torch.optim.AdamW(optim_params, lr=1e-3, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    n_trainable_unet = sum(p.requires_grad for p in unet.parameters())
    assert n_trainable_unet == len(list(unet.parameters()))        # the recipe never freezes the base UNet
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", rank=0, world_size=1)
    try:
        unet = DDP(unet, device_ids=[0])                                                  # accelerator.prepare
        e4t_encoder = DDP(e4t_encoder, device_ids=[0])
        acp = ddpm_alphas_cumprod(device=dev)
        with torch.no_grad():
            class_embed = text_encoder.get_input_embeddings()(torch.tensor([320], device=dev))
            null_context = text_encoder(torch.tensor([[O.BOS] + [O.EOS] * 76], device=dev))[0]
        rnd = random.Random(0)
        torch.manual_seed(0)
        w_before = {k: v.detach().clone() for k, v in unet.module.state_dict().items() if "wo" in k}
        losses = []
        for it in range(3):                                                               # the DDP error shows on step 2
            g = torch.Generator().manual_seed(50 + it)
            pixel_values = (torch.rand(2, 3, 64, 64, generator=g) * 2 - 1).to(dev)
            loss, pred, input_ids, idxs = _train_iteration(unet, e4t_encoder, text_encoder, optimizer, class_embed,
                                                           null_context, pixel_values, acp, rnd)
            losses.append(loss.item())
            assert pred.shape == (2, 4, 16, 16) and pred.dtype == torch.float32
            assert idxs == [r.index(O.PLACEHOLDER_ID) for r in input_ids.tolist()]
        assert all(torch.isfinite(torch.tensor(losses))), losses
        changed = sum(not torch.equal(w_before[k], v) for k, v in unet.module.state_dict().items() if "wo" in k)
        assert changed > 0.9 * len(w_before), (changed, len(w_before))
        print("[drop-in] training iteration x3 under DDP: losses", [round(l, 5) for l in losses])
    finally:
        if created:
            dist.destroy_process_group()
