"""Whole-step golden at the REAL configuration (BASELINE.json configs[0]/[1] model: SD-v1.4 UNet + E4T encoder with
CLIP ViT-H/14 + CLIP-L text, B=2, 512^2 pixels / 64^2 latents, fp32 CPU):

    E4T_REFERENCE=<checkout> python oracle/gen_golden_step.py [--steps 10]   # -> tests/golden/step_sd14_vith.pt
                                                                              #    (~10-15 min on 8 cores)

What runs where (pretrain_e4t.py:616-654):
  * both UNet passes (:624, :636)      -> the REFERENCE's own e4t/models/*.py imported from $E4T_REFERENCE (oracle/shim
                                          stands in for the absent diffusers package), autograd for every "wo" gradient
  * CLIP ViT-H/14 tower (encoder.py:154) -> transformers.CLIPVisionModel at the ViT-H/14 size: an INDEPENDENT
                                          implementation; the oracle's vit_forward is checked against it here at full
                                          size and the measured difference is stored in the fixture (`pin_vit`)
  * encoder head (encoder.py:141-168)  -> literal 129-iteration loop (oracle.encoder_forward semantics)
  * CLIP-L text with inputs_embeds (modeling_clip.py:10-82) -> oracle.text_forward, checked here at full CLIP-L size
                                          against transformers.CLIPTextModel(input_ids) (`pin_text`)
  * loss (:645-647), AdamW over {encoder head, "wo"} (:274-278, :652) -> torch, fp32

The fixture holds: the per-step losses of a `--steps`-step run (different seeded batch every step), and for step 0
`pred`, `domain_embed`, `placeholder_idxs`, the WeightOffsets gradients (small ones verbatim, corner+norm of the square
ones) and corner+norm of the encoder-head gradients: every scalar among them (INCLUDING the 96 `.v` scalars) and a
fixed fifth of the others (oracle/golden.py keeps the file below 1 MB).
Weights/inputs come from oracle.synth_state_dict / synth_batch seeds so the GPU test rebuilds them bit-identically.
"""
import argparse
import os
import sys
import time

import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if not os.path.isdir(os.environ.get("E4T_REFERENCE", "")):
    raise SystemExit("set E4T_REFERENCE to a checkout of the original e4t-diffusion project")
sys.path[:0] = [os.environ["E4T_REFERENCE"], os.path.join(HERE, "shim"), ROOT]

from oracle import e4t_oracle as O  # noqa: E402
from oracle.golden import sample_grads  # noqa: E402

from e4t.models.unet_2d_condition import UNet2DConditionModel  # noqa: E402  (the reference's)

OUT = os.path.join(ROOT, "tests", "golden")
SEED_U, SEED_E, SEED_T = 11, 12, 13
LR = 1e-4
CLASS_TOKEN_ID = 320


def rel(a, b):
    a = a.double(); b = b.double()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt().clamp_min(1e-30)).item()


def hf_vision(sd, v):
    """transformers.CLIPVisionModel loaded with the open_clip-named synthetic weights (same mapping as
    tests/test_oracle_cpu.py::test_vit_matches_transformers_clip_vision)."""
    from transformers import CLIPVisionConfig, CLIPVisionModel
    cfg = CLIPVisionConfig(hidden_size=v["width"], intermediate_size=v["mlp"], num_hidden_layers=v["layers"],
                           num_attention_heads=v["heads"], image_size=v["image"], patch_size=v["patch"],
                           hidden_act="gelu", layer_norm_eps=1e-5)
    with torch.device("meta"):
        hf = CLIPVisionModel(cfg)
    hf = hf.to_empty(device="cpu").eval()
    p = "clip_vision."
    m = {"vision_model.embeddings.class_embedding": sd[p + "class_embedding"],
         "vision_model.embeddings.patch_embedding.weight": sd[p + "conv1.weight"],
         "vision_model.embeddings.position_embedding.weight": sd[p + "positional_embedding"],
         "vision_model.pre_layrnorm.weight": sd[p + "ln_pre.weight"], "vision_model.pre_layrnorm.bias": sd[p + "ln_pre.bias"],
         "vision_model.post_layernorm.weight": sd[p + "ln_post.weight"],
         "vision_model.post_layernorm.bias": sd[p + "ln_post.bias"]}
    W = v["width"]
    for i in range(v["layers"]):
        b = p + f"transformer.resblocks.{i}."
        h = f"vision_model.encoder.layers.{i}."
        wi, bi = sd[b + "attn.in_proj_weight"], sd[b + "attn.in_proj_bias"]
        for j, n in enumerate(("q_proj", "k_proj", "v_proj")):
            m[h + f"self_attn.{n}.weight"] = wi[j * W:(j + 1) * W]
            m[h + f"self_attn.{n}.bias"] = bi[j * W:(j + 1) * W]
        m[h + "self_attn.out_proj.weight"] = sd[b + "attn.out_proj.weight"]
        m[h + "self_attn.out_proj.bias"] = sd[b + "attn.out_proj.bias"]
        for a, c in (("layer_norm1", "ln_1"), ("layer_norm2", "ln_2"), ("mlp.fc1", "mlp.c_fc"), ("mlp.fc2", "mlp.c_proj")):
            m[h + a + ".weight"] = sd[b + c + ".weight"]
            m[h + a + ".bias"] = sd[b + c + ".bias"]
    missing, unexpected = hf.load_state_dict(m, strict=False)
    assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
    if hasattr(hf.vision_model.embeddings, "position_ids"):
        n = hf.vision_model.embeddings.position_ids.shape[-1]
        hf.vision_model.embeddings.position_ids = torch.arange(n).unsqueeze(0)
    hf.requires_grad_(False)
    return hf


def hf_text(sd, t):
    from transformers import CLIPTextConfig, CLIPTextModel
    cfg = CLIPTextConfig(vocab_size=t["vocab"], hidden_size=t["width"], intermediate_size=t["mlp"],
                         num_hidden_layers=t["layers"], num_attention_heads=t["heads"],
                         max_position_embeddings=t["positions"], hidden_act="quick_gelu", layer_norm_eps=1e-5,
                         eos_token_id=O.EOS, bos_token_id=O.BOS, pad_token_id=O.EOS)
    hf = CLIPTextModel(cfg).eval()
    missing, unexpected = hf.load_state_dict(sd, strict=False)
    assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
    return hf


def summarise(grads):
    out = {}
    for k, g in grads.items():
        if g.numel() <= 4096:
            out[k] = g.clone()
        else:
            g2 = g.reshape(g.shape[0], -1)
            out[k + "#corner"] = g2[:16, :16].clone()
            out[k + "#norm"] = g.norm().clone()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=2)
    args = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    ucfg, vcfg, tcfg = O.SD14_UNET, O.VIT_H14, O.CLIP_TEXT_L
    B = args.batch
    t0 = time.time()
    unet = UNet2DConditionModel(**O.ref_unet_kwargs(ucfg))
    sd_u = O.synth_state_dict(O.unet_param_shapes(ucfg), SEED_U)
    unet.load_state_dict(sd_u, strict=True)
    # pretrain_e4t.py never freezes the base UNet but only "wo" params reach the optimiser (:274-278): freezing the
    # rest changes no result and spares 3.4 GB of unused gradients
    wo_params = {}
    for k, p in unet.named_parameters():
        p.requires_grad_("wo" in k)
        if "wo" in k:
            wo_params[k] = p
    sd_e = O.synth_state_dict(O.encoder_param_shapes(vcfg, 10880, tcfg["width"], 129), SEED_E)
    sd_t = O.synth_state_dict(O.text_param_shapes(tcfg), SEED_T)
    head = {k: v.requires_grad_(True) for k, v in sd_e.items() if not k.startswith("clip_vision.")}
    vis = hf_vision(sd_e, vcfg)
    print(f"models built in {time.time()-t0:.1f}s")

    # ---- pins at full size -------------------------------------------------------------------------------------
    pins = {}
    xb = O.synth_batch(B, seed=42)["pixel_values"]
    with torch.no_grad():
        xp = O.encoder_preprocess(xb, vcfg["image"])
        o = vis(pixel_values=xp)
        pooled_o, tokens_o = O.vit_forward(sd_e, vcfg, xp)
        pins["pin_vit"] = dict(pooled=rel(pooled_o, o.pooler_output), tokens=rel(tokens_o, o.last_hidden_state[:, 1:]))
        ids, _ = O.synth_input_ids([0, 5, 9])
        ht = hf_text(sd_t, tcfg)
        pins["pin_text"] = rel(O.text_forward(sd_t, tcfg, input_ids=ids), ht(input_ids=ids).last_hidden_state)
        del ht
    print("pins (oracle restatement vs transformers at FULL size):", pins)
    assert pins["pin_vit"]["pooled"] < 1e-4 and pins["pin_vit"]["tokens"] < 1e-4 and pins["pin_text"] < 1e-4

    emb_w = sd_t["text_model.embeddings.token_embedding.weight"]
    class_embed = emb_w[CLASS_TOKEN_ID].detach()
    with torch.no_grad():
        ehs_e4t = O.text_forward(sd_t, tcfg, input_ids=torch.tensor([[O.BOS] + [O.EOS] * 76]))

    def encoder_forward(pixel_values, maps):
        """E4TEncoder.forward (encoder.py:141-168) with the tower evaluated by transformers.CLIPVisionModel."""
        u = torch.cat([m.mean(dim=(2, 3)) for m in maps], dim=-1)
        u = F.linear(F.leaky_relu(F.linear(u, head["unet_feature_embedder.0.weight"], head["unet_feature_embedder.0.bias"])),
                     head["unet_feature_embedder.2.weight"], head["unet_feature_embedder.2.bias"])
        with torch.no_grad():
            o = vis(pixel_values=O.encoder_preprocess(pixel_values, vcfg["image"]))
        pooled, tokens = o.pooler_output, o.last_hidden_state[:, 1:]
        hs = torch.cat([pooled.unsqueeze(1), tokens[:, 1::2, :]], dim=1)
        outs = []
        for i in range(hs.shape[1]):
            h = F.linear(torch.cat([hs[:, i, :], u], dim=-1), head["feature_linear.weight"], head["feature_linear.bias"])
            outs.append(F.linear(h, head[f"first_linears.{i}.weight"], head[f"first_linears.{i}.bias"]))
        h = F.leaky_relu(torch.stack(outs).mean(dim=0))
        return F.linear(h, head["final_linear.weight"], head["final_linear.bias"])

    def step(batch):
        pixel_values, latents, noise = batch["pixel_values"], batch["latents"], batch["noise"]
        timesteps, input_ids = batch["timesteps"], batch["input_ids"]
        inputs_embeds = emb_w[input_ids].detach().clone()                                              # :616
        idxs = [row.index(O.PLACEHOLDER_ID) for row in input_ids.tolist()]                             # :617
        noisy = O.add_noise(latents, noise, timesteps)                                                 # :621
        enc = unet(noisy, timesteps, ehs_e4t.expand(B, -1, -1), return_encoder_outputs=True)           # :624
        domain_embed = encoder_forward(pixel_values, enc["down_block_samples"])                        # :626
        domain_embed = class_embed.clone().expand(B, -1) + 0.1 * domain_embed                          # :628
        for i, idx in enumerate(idxs):                                                                 # :630-631
            inputs_embeds[i, idx, :] = domain_embed[i]
        ehs = O.text_forward(sd_t, tcfg, inputs_embeds=inputs_embeds)                                  # :634
        pred = unet(noisy, timesteps, ehs).sample                                                      # :636
        loss_diff = F.mse_loss(pred.float(), noise.float(), reduction="mean")                          # :645
        loss_reg = 0.01 * domain_embed.pow(2).sum()                                                    # :646
        return dict(loss=loss_diff + loss_reg, loss_diff=loss_diff, loss_reg=loss_reg, pred=pred,
                    domain_embed=domain_embed, placeholder_idxs=idxs)

    train = list(wo_params.values()) + list(head.values())
    opt = torch.optim.AdamW(train, lr=LR, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    rec = dict(cfg=dict(unet=ucfg, vit=vcfg, text=tcfg), seeds=(SEED_U, SEED_E, SEED_T), B=B, lr=LR,
               class_token_id=CLASS_TOKEN_ID, batch_seed0=42, losses=[], **pins)
    for it in range(args.steps):
        t1 = time.time()
        batch = O.synth_batch(B, seed=42 + it)
        out = step(batch)
        opt.zero_grad(set_to_none=True)
        out["loss"].backward()
        rec["losses"].append([out[k].item() for k in ("loss", "loss_diff", "loss_reg")])
        if it == 0:
            rec["pred"] = out["pred"].detach().clone()
            rec["domain_embed"] = out["domain_embed"].detach().clone()
            rec["placeholder_idxs"] = out["placeholder_idxs"]
            # below 1 MB: every scalar entry, a fixed fifth of the others
            rec["wo_grads"] = sample_grads(summarise({k: p.grad for k, p in wo_params.items()}), 5)
            rec["head_grads"] = sample_grads(summarise({k: p.grad for k, p in head.items()}), 5)
            # conditioning of the 96 scalar `.v` gradients: dv = w1·dβ1 + w2·dβ2 is a cancelling sum of these terms
            vs = {}
            for k in wo_params:
                if k.endswith(".v"):
                    b = k[:-1]
                    vs[k] = (wo_params[b + "linear1.weight"].detach().norm() * wo_params[b + "linear1.bias"].grad.norm()
                             + wo_params[b + "linear2.weight"].detach().norm() * wo_params[b + "linear2.bias"].grad.norm()).clone()
            rec["v_scale"] = vs
        opt.step()
        print(f"step {it}: loss {rec['losses'][-1]}  ({time.time()-t1:.1f}s)", flush=True)
        torch.save(rec, os.path.join(OUT, "step_sd14_vith.pt"))
    print("wrote", os.path.join(OUT, "step_sd14_vith.pt"), os.path.getsize(os.path.join(OUT, "step_sd14_vith.pt")))


if __name__ == "__main__":
    main()
