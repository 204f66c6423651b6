"""CPU ORACLE for the E4T pre-training hot path — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this file.
The product path (e4t-diffusion_b200/) never does; it fails loudly when the CUDA library is missing.

Plain-torch (fp32/fp64, CPU) functional restatement of the reference algorithm, operating on state dicts that use
the reference's exact key names.  Each function cites the reference file:line it follows
(mkshing/e4t-diffusion @ a1d2593).

Pinning status
  * UNet + WeightOffsets + attention + transformer blocks: PINNED — oracle/gen_golden.py imports the reference's own
    e4t/models/*.py from a checkout of the original project (through oracle/shim for the absent diffusers package) and
    the outputs / gradients it produced are committed under tests/golden/ (tests/test_oracle_cpu.py checks this file against them).
  * diffusers 0.14.0 pieces (ResnetBlock2D, Downsample2D, Upsample2D, Timesteps, TimestepEmbedding, DDPM add_noise):
    restated from the published 0.14.0 behaviour — **parity unpinned** (diffusers is not installed, no network).
  * E4TEncoder (e4t/encoder.py:78-168): open_clip and kornia are absent, so the ViT-H/14 tower follows open_clip's
    published VisionTransformer.forward and kornia.geometry.resize is taken to be F.interpolate(bicubic,
    align_corners=True) — **parity unpinned**; the ViT restatement is cross-checked against
    transformers.CLIPVisionModel (an independent implementation) in tests/test_oracle_cpu.py.
  * CLIP text model with inputs_embeds (e4t/models/modeling_clip.py:10-82): restated; cross-checked against
    transformers.CLIPTextModel — **parity unpinned** w.r.t. the reference's pinned-era transformers.
"""
import math
import zlib

import torch
import torch.nn.functional as F

# ------------------------------------------------------------------------------------------------
# configs
# ------------------------------------------------------------------------------------------------
SD14_UNET = dict(in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280), layers_per_block=2,
                 attention_head_dim=8, cross_attention_dim=768, norm_num_groups=32, norm_eps=1e-5, sample_size=64,
                 flip_sin_to_cos=True, freq_shift=0)
TINY_UNET = dict(in_channels=4, out_channels=4, block_out_channels=(64, 128), layers_per_block=1,
                 attention_head_dim=4, cross_attention_dim=64, norm_num_groups=32, norm_eps=1e-5, sample_size=16,
                 flip_sin_to_cos=True, freq_shift=0)
VIT_H14 = dict(width=1280, layers=32, heads=16, mlp=5120, patch=14, image=224)
VIT_TINY = dict(width=64, layers=2, heads=4, mlp=128, patch=14, image=224)
CLIP_TEXT_L = dict(width=768, layers=12, heads=12, mlp=3072, vocab=49409, positions=77)
CLIP_TEXT_TINY = dict(width=64, layers=2, heads=4, mlp=128, vocab=49409, positions=77)


def block_types(cfg):
    n = len(cfg["block_out_channels"])
    down = ["CrossAttnDownBlock2D"] * (n - 1) + ["DownBlock2D"]
    up = ["UpBlock2D"] + ["CrossAttnUpBlock2D"] * (n - 1)
    return down, up


def ref_unet_kwargs(cfg):
    """kwargs for the reference's UNet2DConditionModel(**kw) (unet_2d_condition.py:39-78)."""
    down, up = block_types(cfg)
    kw = dict(cfg)
    kw["down_block_types"] = tuple(down)
    kw["up_block_types"] = tuple(up)
    return kw


# ------------------------------------------------------------------------------------------------
# parameter inventory (key -> shape), identical to the reference module tree's state_dict
# ------------------------------------------------------------------------------------------------
def _wo_shapes(p, R, C):
    # e4t/weightoffsets.py:6-12
    return {p + "v": (1,), p + "linear1.weight": (R, 1), p + "linear1.bias": (R,), p + "linear2.weight": (C, 1),
            p + "linear2.bias": (C,), p + "linear_column.weight": (R, R), p + "linear_column.bias": (R,),
            p + "linear_row.weight": (C, C), p + "linear_row.bias": (C,)}


def _attn_shapes(p, C, ctx):
    # e4t/models/cross_attention.py:77-99
    s = {p + "to_q.weight": (C, C), p + "to_k.weight": (C, ctx), p + "to_v.weight": (C, ctx),
         p + "to_out.0.weight": (C, C), p + "to_out.0.bias": (C,)}
    s.update(_wo_shapes(p + "wo_q.", C, C))
    s.update(_wo_shapes(p + "wo_k.", ctx, C))
    s.update(_wo_shapes(p + "wo_v.", ctx, C))
    return s


def _tf_shapes(p, C, ctx):
    # e4t/models/transformer_2d.py:149-209, attention.py:181-273,335-384
    s = {p + "norm.weight": (C,), p + "norm.bias": (C,), p + "proj_in.weight": (C, C, 1, 1), p + "proj_in.bias": (C,),
         p + "proj_out.weight": (C, C, 1, 1), p + "proj_out.bias": (C,)}
    b = p + "transformer_blocks.0."
    for n in ("norm1", "norm2", "norm3"):
        s[b + n + ".weight"] = (C,)
        s[b + n + ".bias"] = (C,)
    s.update(_attn_shapes(b + "attn1.", C, C))
    s.update(_attn_shapes(b + "attn2.", C, ctx))
    s[b + "ff.net.0.proj.weight"] = (8 * C, C)
    s[b + "ff.net.0.proj.bias"] = (8 * C,)
    s[b + "ff.net.2.weight"] = (C, 4 * C)
    s[b + "ff.net.2.bias"] = (C,)
    return s


def _res_shapes(p, cin, cout, temb):
    s = {p + "norm1.weight": (cin,), p + "norm1.bias": (cin,), p + "conv1.weight": (cout, cin, 3, 3),
         p + "conv1.bias": (cout,), p + "time_emb_proj.weight": (cout, temb), p + "time_emb_proj.bias": (cout,),
         p + "norm2.weight": (cout,), p + "norm2.bias": (cout,), p + "conv2.weight": (cout, cout, 3, 3),
         p + "conv2.bias": (cout,)}
    if cin != cout:
        s[p + "conv_shortcut.weight"] = (cout, cin, 1, 1)
        s[p + "conv_shortcut.bias"] = (cout,)
    return s


def unet_param_shapes(cfg):
    """Follows the construction order of e4t/models/unet_2d_condition.py:110-299 (keys only; order irrelevant)."""
    boc = cfg["block_out_channels"]
    L = cfg["layers_per_block"]
    ctx = cfg["cross_attention_dim"]
    temb = boc[0] * 4
    s = {"conv_in.weight": (boc[0], cfg["in_channels"], 3, 3), "conv_in.bias": (boc[0],),
         "time_embedding.linear_1.weight": (temb, boc[0]), "time_embedding.linear_1.bias": (temb,),
         "time_embedding.linear_2.weight": (temb, temb), "time_embedding.linear_2.bias": (temb,)}
    n = len(boc)
    out_c = boc[0]
    for i in range(n):
        in_c, out_c = out_c, boc[i]
        last = i == n - 1
        for j in range(L):
            s.update(_res_shapes(f"down_blocks.{i}.resnets.{j}.", in_c if j == 0 else out_c, out_c, temb))
            if not last:
                s.update(_tf_shapes(f"down_blocks.{i}.attentions.{j}.", out_c, ctx))
        if not last:
            s[f"down_blocks.{i}.downsamplers.0.conv.weight"] = (out_c, out_c, 3, 3)
            s[f"down_blocks.{i}.downsamplers.0.conv.bias"] = (out_c,)
    mid = boc[-1]
    s.update(_res_shapes("mid_block.resnets.0.", mid, mid, temb))
    s.update(_tf_shapes("mid_block.attentions.0.", mid, ctx))
    s.update(_res_shapes("mid_block.resnets.1.", mid, mid, temb))
    rev = list(reversed(boc))
    out_c = rev[0]
    for i in range(n):
        prev = out_c
        out_c = rev[i]
        in_c = rev[min(i + 1, n - 1)]
        last = i == n - 1
        for j in range(L + 1):
            res_skip = in_c if j == L else out_c
            res_in = prev if j == 0 else out_c
            s.update(_res_shapes(f"up_blocks.{i}.resnets.{j}.", res_in + res_skip, out_c, temb))
            if i > 0:
                s.update(_tf_shapes(f"up_blocks.{i}.attentions.{j}.", out_c, ctx))
        if not last:
            s[f"up_blocks.{i}.upsamplers.0.conv.weight"] = (out_c, out_c, 3, 3)
            s[f"up_blocks.{i}.upsamplers.0.conv.bias"] = (out_c,)
    s["conv_norm_out.weight"] = (boc[0],)
    s["conv_norm_out.bias"] = (boc[0],)
    s["conv_out.weight"] = (cfg["out_channels"], boc[0], 3, 3)
    s["conv_out.bias"] = (cfg["out_channels"],)
    return s


def pooled_feature_dim(cfg):
    boc = cfg["block_out_channels"]
    L = cfg["layers_per_block"]
    n = len(boc)
    d = boc[0]
    for i in range(n):
        d += boc[i] * L + (boc[i] if i < n - 1 else 0)
    return d + boc[-1]


def vit_param_shapes(v, p="clip_vision."):
    # open_clip VisionTransformer naming (SURVEY.md §8b)
    W = v["width"]
    g = v["image"] // v["patch"]
    s = {p + "conv1.weight": (W, 3, v["patch"], v["patch"]), p + "class_embedding": (W,),
         p + "positional_embedding": (g * g + 1, W), p + "ln_pre.weight": (W,), p + "ln_pre.bias": (W,),
         p + "ln_post.weight": (W,), p + "ln_post.bias": (W,)}
    for i in range(v["layers"]):
        b = p + f"transformer.resblocks.{i}."
        s.update({b + "ln_1.weight": (W,), b + "ln_1.bias": (W,), b + "attn.in_proj_weight": (3 * W, W),
                  b + "attn.in_proj_bias": (3 * W,), b + "attn.out_proj.weight": (W, W), b + "attn.out_proj.bias": (W,),
                  b + "ln_2.weight": (W,), b + "ln_2.bias": (W,), b + "mlp.c_fc.weight": (v["mlp"], W),
                  b + "mlp.c_fc.bias": (v["mlp"],), b + "mlp.c_proj.weight": (W, v["mlp"]), b + "mlp.c_proj.bias": (W,)})
    return s


def encoder_param_shapes(v, feat_dim=10880, word_dim=768, n_layers=129):
    # e4t/encoder.py:101-125
    W = v["width"]
    s = vit_param_shapes(v)
    s.update({"unet_feature_embedder.0.weight": (W, feat_dim), "unet_feature_embedder.0.bias": (W,),
              "unet_feature_embedder.2.weight": (W, W), "unet_feature_embedder.2.bias": (W,),
              "feature_linear.weight": (W, 2 * W), "feature_linear.bias": (W,),
              "final_linear.weight": (word_dim, W), "final_linear.bias": (word_dim,)})
    for i in range(n_layers):
        s[f"first_linears.{i}.weight"] = (W, W)
        s[f"first_linears.{i}.bias"] = (W,)
    return s


def text_param_shapes(t, p="text_model."):
    W = t["width"]
    s = {p + "embeddings.token_embedding.weight": (t["vocab"], W),
         p + "embeddings.position_embedding.weight": (t["positions"], W),
         p + "final_layer_norm.weight": (W,), p + "final_layer_norm.bias": (W,)}
    for i in range(t["layers"]):
        b = p + f"encoder.layers.{i}."
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            s[b + f"self_attn.{n}.weight"] = (W, W)
            s[b + f"self_attn.{n}.bias"] = (W,)
        s.update({b + "layer_norm1.weight": (W,), b + "layer_norm1.bias": (W,), b + "layer_norm2.weight": (W,),
                  b + "layer_norm2.bias": (W,), b + "mlp.fc1.weight": (t["mlp"], W), b + "mlp.fc1.bias": (t["mlp"],),
                  b + "mlp.fc2.weight": (W, t["mlp"]), b + "mlp.fc2.bias": (W,)})
    return s


def synth_state_dict(shapes, seed=0, dtype=torch.float32):
    """Deterministic random-init weights, one independent stream per key (crc32(key) ^ seed), torch-default-like
    scales: matrices/convs U(±1/sqrt(fan_in)); norm gains 1+0.1·N; biases/embeddings small; WeightOffsets.v = 1
    (e4t/weightoffsets.py:8).  The same function feeds the reference (golden generation), this oracle and the CUDA
    implementation, so all three see bit-identical parameters."""
    sd = {}
    for k in sorted(shapes):
        shp = tuple(shapes[k])
        g = torch.Generator().manual_seed((zlib.crc32(k.encode()) ^ (seed * 2654435761)) & 0x7FFFFFFF)
        if k.endswith(".v") and shp == (1,):
            t = torch.ones(1)
        elif len(shp) >= 2:
            fan_in = 1
            for d in shp[1:]:
                fan_in *= d
            if "embedding" in k:
                t = torch.randn(shp, generator=g) * 0.02
            else:
                t = (torch.rand(shp, generator=g) * 2 - 1) / math.sqrt(fan_in)
        elif k.endswith("weight") and ("norm" in k or "ln_" in k):
            t = 1 + 0.1 * torch.randn(shp, generator=g)
        elif k.endswith("class_embedding"):
            t = torch.randn(shp, generator=g) * 0.02
        else:
            t = (torch.rand(shp, generator=g) * 2 - 1) * 0.05
            if ".wo_" in k:  # linear1/linear2/linear_column/linear_row biases: torch default is U(±1/sqrt(fan_in))
                t = t * 4
        sd[k] = t.to(dtype)
    return sd


# ------------------------------------------------------------------------------------------------
# WeightOffsets + attention (L0 operators)
# ------------------------------------------------------------------------------------------------
def wo_delta(sd, p):
    """Literal e4t/weightoffsets.py:14-23 -> Δ of shape (column_dim, row_dim)."""
    v = sd[p + "v"]
    vx = F.linear(v, sd[p + "linear1.weight"], sd[p + "linear1.bias"])
    vy = F.linear(v, sd[p + "linear2.weight"], sd[p + "linear2.bias"])
    m = vx.unsqueeze(0).T * vy.unsqueeze(0)
    m = F.linear(m.T, sd[p + "linear_column.weight"], sd[p + "linear_column.bias"])
    m = F.linear(m.T, sd[p + "linear_row.weight"], sd[p + "linear_row.bias"])
    return m.T


def wo_delta_closed_form(sd, p):
    """SURVEY.md Appendix A: Δ = b·aᵀ + s·b_cᵀ + b_r·1ᵀ."""
    v = sd[p + "v"]
    vx = sd[p + "linear1.weight"][:, 0] * v + sd[p + "linear1.bias"]
    vy = sd[p + "linear2.weight"][:, 0] * v + sd[p + "linear2.bias"]
    Wc, bc = sd[p + "linear_column.weight"], sd[p + "linear_column.bias"]
    Wr, br = sd[p + "linear_row.weight"], sd[p + "linear_row.bias"]
    a, b, s = Wc @ vx, Wr @ vy, Wr.sum(1)
    return b[:, None] * a[None, :] + s[:, None] * bc[None, :] + br[:, None]


USE_SDPA = False


def cross_attention(sd, p, x, ctx, heads):
    """CrossAttnProcessor.__call__ (cross_attention.py:285-322) == AttnProcessor2_0 (:490-538) numerically."""
    ctx = x if ctx is None else ctx
    q = F.linear(x, sd[p + "to_q.weight"] * (1 + wo_delta(sd, p + "wo_q.")))      # :297 / :506
    k = F.linear(ctx, sd[p + "to_k.weight"] * (1 + wo_delta(sd, p + "wo_k.")))    # :305 / :516
    v = F.linear(ctx, sd[p + "to_v.weight"] * (1 + wo_delta(sd, p + "wo_v.")))    # :307 / :518
    B, N, C = q.shape
    dh = C // heads
    q = q.view(B, N, heads, dh).transpose(1, 2)
    k = k.view(B, -1, heads, dh).transpose(1, 2)
    v = v.view(B, -1, heads, dh).transpose(1, 2)
    if USE_SDPA:   # AttnProcessor2_0 literally (:527-529); used by bench.py's on-GPU stock-torch comparator
        o = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B, N, C)
    else:
        s = (q @ k.transpose(-1, -2)) * dh ** -0.5                                 # scale = dim_head**-0.5 (:59)
        o = (s.softmax(-1) @ v).transpose(1, 2).reshape(B, N, C)
    return F.linear(o, sd[p + "to_out.0.weight"], sd[p + "to_out.0.bias"])        # :534


def transformer_block(sd, p, x, ctx, heads):
    """BasicTransformerBlock.forward (attention.py:275-332) + FeedForward/GEGLU (:335-384,409-430)."""
    C = x.shape[-1]
    h = F.layer_norm(x, (C,), sd[p + "norm1.weight"], sd[p + "norm1.bias"], 1e-5)
    x = cross_attention(sd, p + "attn1.", h, None, heads) + x
    h = F.layer_norm(x, (C,), sd[p + "norm2.weight"], sd[p + "norm2.bias"], 1e-5)
    x = cross_attention(sd, p + "attn2.", h, ctx, heads) + x
    h = F.layer_norm(x, (C,), sd[p + "norm3.weight"], sd[p + "norm3.bias"], 1e-5)
    u, g = F.linear(h, sd[p + "ff.net.0.proj.weight"], sd[p + "ff.net.0.proj.bias"]).chunk(2, dim=-1)
    return F.linear(u * F.gelu(g), sd[p + "ff.net.2.weight"], sd[p + "ff.net.2.bias"]) + x


def transformer_2d(sd, p, x, ctx, heads, groups):
    """Transformer2DModel.forward, continuous path (transformer_2d.py:248-286)."""
    B, C, H, W = x.shape
    res = x
    h = F.group_norm(x, groups, sd[p + "norm.weight"], sd[p + "norm.bias"], 1e-6)   # eps 1e-6 (:149)
    h = F.conv2d(h, sd[p + "proj_in.weight"], sd[p + "proj_in.bias"])
    h = h.permute(0, 2, 3, 1).reshape(B, H * W, C)
    h = transformer_block(sd, p + "transformer_blocks.0.", h, ctx, heads)
    h = h.reshape(B, H, W, C).permute(0, 3, 1, 2)
    return F.conv2d(h, sd[p + "proj_out.weight"], sd[p + "proj_out.bias"]) + res


def resnet_block(sd, p, x, temb, groups, eps):
    """diffusers 0.14.0 ResnetBlock2D.forward (restated; SURVEY.md §8 a-8)."""
    h = F.conv2d(F.silu(F.group_norm(x, groups, sd[p + "norm1.weight"], sd[p + "norm1.bias"], eps)),
                 sd[p + "conv1.weight"], sd[p + "conv1.bias"], padding=1)
    h = h + F.linear(F.silu(temb), sd[p + "time_emb_proj.weight"], sd[p + "time_emb_proj.bias"])[:, :, None, None]
    h = F.conv2d(F.silu(F.group_norm(h, groups, sd[p + "norm2.weight"], sd[p + "norm2.bias"], eps)),
                 sd[p + "conv2.weight"], sd[p + "conv2.bias"], padding=1)
    if p + "conv_shortcut.weight" in sd:
        x = F.conv2d(x, sd[p + "conv_shortcut.weight"], sd[p + "conv_shortcut.bias"])
    return x + h


def timestep_embedding(t, dim, flip_sin_to_cos=True, freq_shift=0):
    """diffusers 0.14.0 get_timestep_embedding (restated; SURVEY.md §8 a-11)."""
    half = dim // 2
    exponent = -math.log(10000) * torch.arange(half, dtype=torch.float32, device=t.device) / (half - freq_shift)
    emb = t[:, None].float() * torch.exp(exponent)[None, :]
    emb = torch.cat([torch.sin(emb), torch.cos(emb)], dim=-1)
    if flip_sin_to_cos:
        emb = torch.cat([emb[:, half:], emb[:, :half]], dim=-1)
    return emb


def unet_forward(sd, cfg, sample, timesteps, ehs, return_encoder_outputs=False):
    """UNet2DConditionModel.forward (unet_2d_condition.py:410-562)."""
    boc, L = cfg["block_out_channels"], cfg["layers_per_block"]
    heads, groups, eps = cfg["attention_head_dim"], cfg["norm_num_groups"], cfg["norm_eps"]
    n = len(boc)
    dt = sample.dtype
    if not torch.is_tensor(timesteps):
        timesteps = torch.tensor([timesteps], dtype=torch.int64)
    elif timesteps.dim() == 0:
        timesteps = timesteps[None]
    timesteps = timesteps.expand(sample.shape[0])
    t_emb = timestep_embedding(timesteps, boc[0], cfg["flip_sin_to_cos"], cfg["freq_shift"]).to(dt)   # :461-466
    emb = F.linear(F.silu(F.linear(t_emb, sd["time_embedding.linear_1.weight"], sd["time_embedding.linear_1.bias"])),
                   sd["time_embedding.linear_2.weight"], sd["time_embedding.linear_2.bias"])          # :468
    x = F.conv2d(sample, sd["conv_in.weight"], sd["conv_in.bias"], padding=1)                          # :481
    res = [x]
    for i in range(n):                                                                                 # :485-496
        for j in range(L):
            x = resnet_block(sd, f"down_blocks.{i}.resnets.{j}.", x, emb, groups, eps)
            if i < n - 1:
                x = transformer_2d(sd, f"down_blocks.{i}.attentions.{j}.", x, ehs, heads, groups)
            res.append(x)
        if i < n - 1:
            x = F.conv2d(x, sd[f"down_blocks.{i}.downsamplers.0.conv.weight"],
                         sd[f"down_blocks.{i}.downsamplers.0.conv.bias"], stride=2, padding=1)
            res.append(x)
    x = resnet_block(sd, "mid_block.resnets.0.", x, emb, groups, eps)                                  # :508-515
    x = transformer_2d(sd, "mid_block.attentions.0.", x, ehs, heads, groups)
    x = resnet_block(sd, "mid_block.resnets.1.", x, emb, groups, eps)
    if return_encoder_outputs:                                                                         # :517-521
        return dict(down_block_samples=tuple(res) + (x,))
    for i in range(n):                                                                                 # :527-551
        for j in range(L + 1):
            x = torch.cat([x, res.pop()], dim=1)
            x = resnet_block(sd, f"up_blocks.{i}.resnets.{j}.", x, emb, groups, eps)
            if i > 0:
                x = transformer_2d(sd, f"up_blocks.{i}.attentions.{j}.", x, ehs, heads, groups)
        if i < n - 1:
            x = F.interpolate(x, scale_factor=2.0, mode="nearest")
            x = F.conv2d(x, sd[f"up_blocks.{i}.upsamplers.0.conv.weight"],
                         sd[f"up_blocks.{i}.upsamplers.0.conv.bias"], padding=1)
    x = F.silu(F.group_norm(x, groups, sd["conv_norm_out.weight"], sd["conv_norm_out.bias"], eps))     # :554-556
    return F.conv2d(x, sd["conv_out.weight"], sd["conv_out.bias"], padding=1)                          # :557


# ------------------------------------------------------------------------------------------------
# E4T encoder (e4t/encoder.py:78-168)
# ------------------------------------------------------------------------------------------------
CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)      # encoder.py:128
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)      # encoder.py:129


def _mha(x, w_in, b_in, w_out, b_out, heads, causal=False):
    B, N, W = x.shape
    q, k, v = F.linear(x, w_in, b_in).chunk(3, dim=-1)
    dh = W // heads
    q, k, v = (t.view(B, N, heads, dh).transpose(1, 2) for t in (q, k, v))
    s = (q @ k.transpose(-1, -2)) * dh ** -0.5
    if causal:
        s = s + torch.full((N, N), float("-inf"), dtype=s.dtype, device=s.device).triu(1)
    return F.linear((s.softmax(-1) @ v).transpose(1, 2).reshape(B, N, W), w_out, b_out)


def vit_forward(sd, v, x, p="clip_vision.", ln_post_on_tokens=False):
    """open_clip VisionTransformer.forward with proj=None, output_tokens=True (encoder.py:91-96,154; SURVEY §8 a-12)."""
    W = v["width"]
    x = F.conv2d(x, sd[p + "conv1.weight"], stride=v["patch"])
    x = x.reshape(x.shape[0], W, -1).permute(0, 2, 1)
    cls = sd[p + "class_embedding"].to(x.dtype) + torch.zeros(x.shape[0], 1, W, dtype=x.dtype, device=x.device)
    x = torch.cat([cls, x], dim=1) + sd[p + "positional_embedding"]
    x = F.layer_norm(x, (W,), sd[p + "ln_pre.weight"], sd[p + "ln_pre.bias"], 1e-5)
    for i in range(v["layers"]):
        b = p + f"transformer.resblocks.{i}."
        h = F.layer_norm(x, (W,), sd[b + "ln_1.weight"], sd[b + "ln_1.bias"], 1e-5)
        x = x + _mha(h, sd[b + "attn.in_proj_weight"], sd[b + "attn.in_proj_bias"], sd[b + "attn.out_proj.weight"],
                     sd[b + "attn.out_proj.bias"], v["heads"])
        h = F.layer_norm(x, (W,), sd[b + "ln_2.weight"], sd[b + "ln_2.bias"], 1e-5)
        x = x + F.linear(F.gelu(F.linear(h, sd[b + "mlp.c_fc.weight"], sd[b + "mlp.c_fc.bias"])),
                         sd[b + "mlp.c_proj.weight"], sd[b + "mlp.c_proj.bias"])
    pooled = F.layer_norm(x[:, 0], (W,), sd[p + "ln_post.weight"], sd[p + "ln_post.bias"], 1e-5)
    tokens = x[:, 1:]
    if ln_post_on_tokens:
        tokens = F.layer_norm(tokens, (W,), sd[p + "ln_post.weight"], sd[p + "ln_post.bias"], 1e-5)
    return pooled, tokens


def encoder_preprocess(x, image_size=224):
    """encoder.py:131-139 (kornia bicubic resize, align_corners=True, no antialias; then CLIP normalisation)."""
    x = F.interpolate(x, size=(image_size, image_size), mode="bicubic", align_corners=True)
    x = (x + 1.0) / 2.0
    mean = torch.tensor(CLIP_MEAN, dtype=x.dtype, device=x.device).view(1, 3, 1, 1)
    std = torch.tensor(CLIP_STD, dtype=x.dtype, device=x.device).view(1, 3, 1, 1)
    return (x - mean) / std


def encoder_forward(sd, v, x, maps):
    """E4TEncoder.forward (encoder.py:141-168)."""
    u = torch.cat([m.mean(dim=(2, 3)) for m in maps], dim=-1)                                         # :147-148
    u = F.linear(F.leaky_relu(F.linear(u, sd["unet_feature_embedder.0.weight"], sd["unet_feature_embedder.0.bias"])),
                 sd["unet_feature_embedder.2.weight"], sd["unet_feature_embedder.2.bias"])            # :149
    pooled, tokens = vit_forward(sd, v, encoder_preprocess(x, v["image"]))                           # :153-154
    hs = torch.cat([pooled.unsqueeze(1), tokens[:, 1::2, :]], dim=1)                                  # :155-156
    outs = []
    for i in range(hs.shape[1]):                                                                      # :159-162
        h = F.linear(torch.cat([hs[:, i, :], u], dim=-1), sd["feature_linear.weight"], sd["feature_linear.bias"])
        outs.append(F.linear(h, sd[f"first_linears.{i}.weight"], sd[f"first_linears.{i}.bias"]))
    h = F.leaky_relu(torch.stack(outs).mean(dim=0))                                                   # :163-166
    return F.linear(h, sd["final_linear.weight"], sd["final_linear.bias"])                            # :168


# ------------------------------------------------------------------------------------------------
# CLIP text model with inputs_embeds (e4t/models/modeling_clip.py:10-82)
# ------------------------------------------------------------------------------------------------
def text_forward(sd, t, inputs_embeds=None, input_ids=None, p="text_model."):
    if inputs_embeds is None:
        inputs_embeds = sd[p + "embeddings.token_embedding.weight"][input_ids]
    W = t["width"]
    N = inputs_embeds.shape[1]
    x = inputs_embeds + sd[p + "embeddings.position_embedding.weight"][:N]                           # :37-41
    for i in range(t["layers"]):
        b = p + f"encoder.layers.{i}."
        h = F.layer_norm(x, (W,), sd[b + "layer_norm1.weight"], sd[b + "layer_norm1.bias"], 1e-5)
        w_in = torch.cat([sd[b + f"self_attn.{n}.weight"] for n in ("q_proj", "k_proj", "v_proj")])
        b_in = torch.cat([sd[b + f"self_attn.{n}.bias"] for n in ("q_proj", "k_proj", "v_proj")])
        x = x + _mha(h, w_in, b_in, sd[b + "self_attn.out_proj.weight"], sd[b + "self_attn.out_proj.bias"],
                     t["heads"], causal=True)                                                         # :45-51
        h = F.layer_norm(x, (W,), sd[b + "layer_norm2.weight"], sd[b + "layer_norm2.bias"], 1e-5)
        h = F.linear(h, sd[b + "mlp.fc1.weight"], sd[b + "mlp.fc1.bias"])
        x = x + F.linear(h * torch.sigmoid(1.702 * h), sd[b + "mlp.fc2.weight"], sd[b + "mlp.fc2.bias"])  # quick_gelu
    return F.layer_norm(x, (W,), sd[p + "final_layer_norm.weight"], sd[p + "final_layer_norm.bias"], 1e-5)  # :69


# ------------------------------------------------------------------------------------------------
# the pre-training step (pretrain_e4t.py:595-654)
# ------------------------------------------------------------------------------------------------
TEMPLATES = [  # pretrain_e4t.py:36-47, as word counts before the placeholder (tokenizer is not available offline)
    "a photo of *", "the photo of *", "a photo of a *", "a photo of the *", "a photo of one *",
    "a close-up photo of the *", "a bright photo of the *", "a photo of a nice *", "a good photo of *",
    "a photo of a cool *"]
BOS, EOS, PLACEHOLDER_ID = 49406, 49407, 49408
_WORD_IDS = {"a": 320, "photo": 1125, "of": 539, "the": 518, "one": 637, "close-up": 3469, "bright": 3928,
             "nice": 2527, "good": 886, "cool": 2077}


def synth_input_ids(template_idxs, max_len=77):
    """(B,77) int64 ids '[BOS] w.. PLACEHOLDER [EOS]*' and the placeholder index per row (pretrain_e4t.py:610-617).
    Word ids are fixed stand-ins (<49406); 'close-up' is taken as ONE word-piece."""
    ids, idxs = [], []
    for ti in template_idxs:
        words = TEMPLATES[ti].split()
        row = [BOS] + [PLACEHOLDER_ID if w == "*" else _WORD_IDS[w] for w in words]
        row = row + [EOS] * (max_len - len(row))
        ids.append(row)
        idxs.append(row.index(PLACEHOLDER_ID))                                                        # :617
    return torch.tensor(ids, dtype=torch.int64), idxs


def ddpm_alphas_cumprod(n=1000, beta_start=0.00085, beta_end=0.012):
    """SD-v1.x DDPMScheduler(scaled_linear) (restated from diffusers 0.14.0)."""
    betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, n, dtype=torch.float32) ** 2
    return torch.cumprod(1.0 - betas, dim=0)


def add_noise(latents, noise, timesteps, acp=None):
    acp = (ddpm_alphas_cumprod() if acp is None else acp).to(latents.device)
    a = acp[timesteps].to(latents.dtype) ** 0.5
    s = (1 - acp[timesteps].to(latents.dtype)) ** 0.5
    return a.view(-1, 1, 1, 1) * latents + s.view(-1, 1, 1, 1) * noise                               # :621


def pretrain_step(sd_unet, ucfg, sd_enc, vcfg, sd_text, tcfg, batch, class_token_id=320, domain_embed_scale=0.1,
                  reg_lambda=0.01):
    """Loop body pretrain_e4t.py:616-647 given explicit (pixel_values, latents, noise, timesteps, input_ids)."""
    pixel_values, latents, noise = batch["pixel_values"], batch["latents"], batch["noise"]
    timesteps, input_ids = batch["timesteps"], batch["input_ids"]
    B = latents.shape[0]
    emb_w = sd_text["text_model.embeddings.token_embedding.weight"]
    class_embed = emb_w[class_token_id].detach()                                                      # :561-564
    ids_e4t = torch.tensor([[BOS] + [EOS] * 76], dtype=torch.int64, device=latents.device)
    with torch.no_grad():
        ehs_e4t = text_forward(sd_text, tcfg, input_ids=ids_e4t)                                      # :565-583
    inputs_embeds = emb_w[input_ids].detach().clone()                                                 # :616
    idxs = [row.index(PLACEHOLDER_ID) for row in input_ids.tolist()]                                  # :617
    noisy = add_noise(latents, noise, timesteps)                                                      # :621
    enc = unet_forward(sd_unet, ucfg, noisy, timesteps, ehs_e4t.expand(B, -1, -1), return_encoder_outputs=True)
    domain_embed = encoder_forward(sd_enc, vcfg, pixel_values, enc["down_block_samples"])             # :626
    domain_embed = class_embed.clone().expand(B, -1) + domain_embed_scale * domain_embed              # :628
    for i, idx in enumerate(idxs):                                                                    # :630-631
        inputs_embeds[i, idx, :] = domain_embed[i]
    ehs = text_forward(sd_text, tcfg, inputs_embeds=inputs_embeds)                                    # :634
    pred = unet_forward(sd_unet, ucfg, noisy, timesteps, ehs)                                         # :636
    loss_diff = F.mse_loss(pred.float(), noise.float(), reduction="mean")                             # :645
    loss_reg = reg_lambda * domain_embed.pow(2).sum()                                                 # :646
    return dict(loss=loss_diff + loss_reg, loss_diff=loss_diff, loss_reg=loss_reg, pred=pred,
                domain_embed=domain_embed, placeholder_idxs=idxs)


def synth_batch(B, seed, latent_hw=64, image_hw=512):
    """SURVEY.md §8(d): seeded synthetic inputs of one step."""
    g = torch.Generator().manual_seed(seed)
    import random
    rnd = random.Random(seed)
    tids = rnd.choices(range(len(TEMPLATES)), k=B)
    ids, _ = synth_input_ids(tids)
    return dict(pixel_values=torch.rand(B, 3, image_hw, image_hw, generator=g) * 2 - 1,
                latents=torch.randn(B, 4, latent_hw, latent_hw, generator=g) * 0.18215,
                noise=torch.randn(B, 4, latent_hw, latent_hw, generator=g),
                timesteps=torch.randint(0, 1000, (B,), generator=g, dtype=torch.int64), input_ids=ids)


# ------------------------------------------------------------------------------------------------
# helpers shared by tests/golden generation
# ------------------------------------------------------------------------------------------------
def golden_unet_inputs(cfg, B, seed, hw, enc_shapes=None):
    """Re-draw the inputs oracle/gen_golden.py:unet_case used (same generator, same order)."""
    g = torch.Generator().manual_seed(seed + 17)
    x = torch.randn(B, 4, hw, hw, generator=g)
    t = torch.randint(0, 1000, (B,), generator=g)
    ehs = torch.randn(B, 77, cfg["cross_attention_dim"], generator=g)
    w = torch.randn(B, 4, hw, hw, generator=g)
    wenc = [torch.randn(tuple(s), generator=g) for s in enc_shapes] if enc_shapes is not None else None
    return x, t, ehs, w, wenc


# ------------------------------------------------------------------------------------------------
# inference: StableDiffusionE4TPipeline.__call__ (e4t/pipeline_stable_diffusion_e4t.py:91-250) with the SD-v1.x DDIM
# scheduler of diffusers 0.14.0 (restated: scaled-linear betas, steps_offset 1, clip_sample False, set_alpha_to_one False)
# ------------------------------------------------------------------------------------------------
def ddim_timesteps(num_inference_steps, num_train=1000, steps_offset=1):
    ratio = num_train // num_inference_steps
    return ((torch.arange(0, num_inference_steps) * ratio).round().flip(0).to(torch.int64) + steps_offset).tolist()


def ddim_step(eps, t, x, num_inference_steps, acp=None, num_train=1000):
    acp = ddpm_alphas_cumprod() if acp is None else acp
    prev_t = t - num_train // num_inference_steps
    a_t = acp[t]
    a_prev = acp[prev_t] if prev_t >= 0 else acp[0]
    pred_x0 = (x - (1 - a_t) ** 0.5 * eps) / a_t ** 0.5
    return a_prev ** 0.5 * pred_x0 + (1 - a_prev) ** 0.5 * eps


def pipeline_sample(sd_unet, ucfg, sd_enc, vcfg, sd_text, tcfg, image, input_ids, latents, num_inference_steps=4,
                    guidance_scale=7.5, class_token_id=320, domain_embed_scale=0.1):
    """The denoising loop of pipeline_stable_diffusion_e4t.py:181-216 on explicit prompt ids / starting latents."""
    emb_w = sd_text["text_model.embeddings.token_embedding.weight"]
    bsz = latents.shape[0]
    idx = input_ids[0].tolist().index(PLACEHOLDER_ID)                                                  # :77
    with torch.no_grad():
        ehs_e4t = text_forward(sd_text, tcfg, input_ids=torch.tensor([[BOS] + [EOS] * 76])).expand(bsz, -1, -1)
        base_embeds = emb_w[input_ids]
        class_embed = emb_w[class_token_id]
        pix = image.expand(bsz, -1, -1, -1)
        x = latents.clone()
        for t in ddim_timesteps(num_inference_steps):
            tt = torch.full((bsz,), t, dtype=torch.int64)
            enc = unet_forward(sd_unet, ucfg, x, tt, ehs_e4t, return_encoder_outputs=True)             # :191
            dom = class_embed.expand(bsz, -1) + domain_embed_scale * encoder_forward(sd_enc, vcfg, pix, enc["down_block_samples"])
            emb = base_embeds.expand(bsz, -1, -1).clone()
            emb[:, idx, :] = dom                                                                       # :197-198
            ehs = text_forward(sd_text, tcfg, inputs_embeds=emb)                                       # :200
            if guidance_scale > 1.0:
                eps = unet_forward(sd_unet, ucfg, torch.cat([x, x]), torch.cat([tt, tt]), torch.cat([ehs_e4t, ehs]))
                u, c = eps.chunk(2)
                eps = u + guidance_scale * (c - u)                                                     # :211-213
            else:
                eps = unet_forward(sd_unet, ucfg, x, tt, ehs)
            x = ddim_step(eps, t, x, num_inference_steps)                                              # :216
    return x
