"""Pin the CPU oracle (oracle/e4t_oracle.py) against the golden vectors produced by the REFERENCE's own modules
(oracle/gen_golden.py, run with a checkout of the original project importable).  fp32, tolerance 1e-4 relative
(summation-order differences only)."""
import os

import pytest
import torch

from oracle import e4t_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _rel(a, b):
    a = a.double(); b = b.double()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt().clamp_min(1e-30)).item()


def test_wo_literal_and_closed_form_match_reference():
    gold = torch.load(os.path.join(GOLD, "wo.pt"))
    for (R, C), ref in gold.items():
        shapes = O._wo_shapes("p.", R, C)
        sd = O.synth_state_dict(shapes, 3)
        got = O.wo_delta(sd, "p.")
        assert got.shape == (C, R)
        assert _rel(got[::ref["row_stride"]], ref["rows"]) < 1e-5
        sd64 = {k: v.double() for k, v in sd.items()}
        assert _rel(O.wo_delta_closed_form(sd64, "p."), O.wo_delta(sd64, "p.")) < 1e-12


def test_inventory_matches_reference_state_dict():
    import hashlib
    inv = torch.load(os.path.join(GOLD, "inventory.pt"))
    shapes = O.unet_param_shapes(O.SD14_UNET)
    keys = sorted(shapes)
    sha = hashlib.sha256("\n".join(f"{k}:{tuple(shapes[k])}" for k in keys).encode()).hexdigest()
    assert sha == inv["sha256"] and len(keys) == inv["n_keys"]
    n = lambda pred: sum(int(torch.Size(s).numel()) for k, s in shapes.items() if pred(k))
    assert n(lambda k: "wo" not in k) == inv["n_base"] == 859520964        # SURVEY.md §7 pins
    assert n(lambda k: "wo" in k) == inv["n_wo"] == 143226592
    assert sum(1 for k in keys if "wo" in k) == inv["n_wo_tensors"] == 864
    assert O.pooled_feature_dim(O.SD14_UNET) == 10880                      # encoder.py:102, unet_2d_condition.py:586


def _check_unet(name, grads):
    gold = torch.load(os.path.join(GOLD, name))
    cfg = gold["cfg"]
    sd = O.synth_state_dict(O.unet_param_shapes(cfg), gold["seed"])
    hw = gold["x"].shape[-1]
    x, t, ehs, w, wenc = O.golden_unet_inputs(cfg, gold["B"], gold["seed"], hw, gold["enc_shapes"])
    assert torch.equal(x, gold["x"]) and torch.equal(t, gold["t"]) and torch.equal(ehs, gold["ehs"])
    if grads:
        ehs.requires_grad_(True)
        for k in sd:
            if "wo" in k:
                sd[k].requires_grad_(True)
    with torch.set_grad_enabled(grads):
        out = O.unet_forward(sd, cfg, x, t, ehs)
        enc = O.unet_forward(sd, cfg, x, t, ehs, return_encoder_outputs=True)["down_block_samples"]
    assert [tuple(e.shape) for e in enc] == gold["enc_shapes"]
    assert _rel(out, gold["out"]) < 1e-4
    assert _rel(torch.cat([e.mean(dim=(2, 3)) for e in enc], -1), gold["enc_pooled"]) < 1e-4
    if grads:
        loss = (out * w).sum() + sum((e * we).sum() for e, we in zip(enc, wenc))
        loss.backward()
        assert _rel(ehs.grad, gold["d_ehs"]) < 1e-4
        for k, ref in gold["wo_grads"].items():
            if k.endswith("#corner"):
                got = sd[k[:-7]].grad[:16, :16]
            elif k.endswith("#norm"):
                got = sd[k[:-5]].grad.norm()
            else:
                got = sd[k].grad
            # '.v' is a single scalar formed by a heavily cancelling fp32 sum -> looser
            assert _rel(got, ref) < (5e-3 if k.endswith('.v') else 2e-4), k


def test_unet_tiny_matches_reference_fwd_bwd():
    _check_unet("unet_tiny.pt", grads=True)


def test_unet_sd14_matches_reference_fwd():
    torch.set_num_threads(os.cpu_count())
    _check_unet("unet_sd14.pt", grads=False)


def test_token_index_bookkeeping():
    ids, idxs = O.synth_input_ids(list(range(len(O.TEMPLATES))))
    assert ids.shape == (10, 77) and ids.dtype == torch.int64
    assert idxs == [4, 4, 5, 5, 5, 6, 6, 6, 5, 6]
    for row, i in zip(ids.tolist(), idxs):
        assert row[0] == O.BOS and row[i] == O.PLACEHOLDER_ID and row.index(O.PLACEHOLDER_ID) == i
        assert all(t == O.EOS for t in row[i + 1:])


def test_vit_matches_transformers_clip_vision():
    """Independent second implementation: HF CLIPVisionModel (pre-LN ViT, class token, learned positions)."""
    from transformers import CLIPVisionConfig, CLIPVisionModel
    v = O.VIT_TINY
    cfg = CLIPVisionConfig(hidden_size=v["width"], intermediate_size=v["mlp"], num_hidden_layers=v["layers"],
                           num_attention_heads=v["heads"], image_size=v["image"], patch_size=v["patch"],
                           hidden_act="gelu", layer_norm_eps=1e-5)
    hf = CLIPVisionModel(cfg).eval()
    sd = O.synth_state_dict(O.vit_param_shapes(v), 4)
    p = "clip_vision."
    m = {"vision_model.embeddings.class_embedding": sd[p + "class_embedding"],
         "vision_model.embeddings.patch_embedding.weight": sd[p + "conv1.weight"],
         "vision_model.embeddings.position_embedding.weight": sd[p + "positional_embedding"],
         "vision_model.pre_layrnorm.weight": sd[p + "ln_pre.weight"], "vision_model.pre_layrnorm.bias": sd[p + "ln_pre.bias"],
         "vision_model.post_layernorm.weight": sd[p + "ln_post.weight"], "vision_model.post_layernorm.bias": sd[p + "ln_post.bias"]}
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
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        o = hf(pixel_values=x)
        pooled, tokens = O.vit_forward(sd, v, x)
    assert _rel(pooled, o.pooler_output) < 1e-4
    assert _rel(tokens, o.last_hidden_state[:, 1:]) < 1e-4


def test_text_matches_transformers_clip_text():
    from transformers import CLIPTextConfig, CLIPTextModel
    t = O.CLIP_TEXT_TINY
    cfg = CLIPTextConfig(vocab_size=t["vocab"], hidden_size=t["width"], intermediate_size=t["mlp"],
                         num_hidden_layers=t["layers"], num_attention_heads=t["heads"],
                         max_position_embeddings=t["positions"], hidden_act="quick_gelu", layer_norm_eps=1e-5,
                         eos_token_id=O.EOS, bos_token_id=O.BOS, pad_token_id=O.EOS)
    hf = CLIPTextModel(cfg).eval()
    sd = O.synth_state_dict(O.text_param_shapes(t), 5)
    missing, unexpected = hf.load_state_dict(sd, strict=False)
    assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
    ids, _ = O.synth_input_ids([0, 5, 9])
    ids = ids.clamp(max=t["vocab"] - 1)
    with torch.no_grad():
        ref = hf(input_ids=ids).last_hidden_state
        got = O.text_forward(sd, t, input_ids=ids)
        got2 = O.text_forward(sd, t, inputs_embeds=sd["text_model.embeddings.token_embedding.weight"][ids])
    assert _rel(got, ref) < 1e-4 and torch.equal(got, got2)
