"""StableDiffusionE4TPipeline — mirror of e4t/pipeline_stable_diffusion_e4t.py:30-250 (BASELINE.json configs[4]) on the
sm_100a kernels, forward-only.

Per denoising step the reference runs (pipeline_stable_diffusion_e4t.py:181-216)
    UNet encoder half on the B latents with the empty-prompt context            (:191)
    E4TEncoder(image, 13 feature maps) -> domain embedding                      (:194)
    placeholder row of the prompt embedding <- class_embed + scale * domain      (:196-198)   [same index for every row, :77]
    CLIP text encoder(inputs_embeds)                                            (:200)
    full UNet on 2B rows under classifier-free guidance [uncond = empty prompt] (:201-208)
    guidance mix, scheduler step                                                (:211-216)
Everything heavy goes through the same modules as pre-training (no-grad: W_eff is rebuilt from the current parameters at
each UNet call, no autograd state is kept).  The CLIP ViT-H/14 features of the conditioning image do not depend on the
denoising step — only the pooled UNet features do — so they are computed ONCE per call (`E4TEncoder.image_features`)
instead of once per step (SURVEY.md §8 f-2).

diffusers is not a dependency: the SD-v1.x DDIM scheduler (scaled-linear betas, steps_offset 1, no sample clipping,
eta) is `DDIMScheduler` below; any object with set_timesteps / scale_model_input / step(...).prev_sample works.
With `vae=None` the pipeline returns latents (`output_type="latent"`); with a VAE attached (e.g.
e4t.models.autoencoder_kl.AutoencoderKL, decoded on the sm_100a kernels) `vae.decode(z).sample` is called as the
reference does (decode_latents)."""
from dataclasses import dataclass
from typing import List, Optional, Union

import torch

from e4t._mixins import BaseOutput


@dataclass
class StableDiffusionPipelineOutput(BaseOutput):
    images: object = None
    nsfw_content_detected: object = None


@dataclass
class _StepOutput(BaseOutput):
    prev_sample: torch.Tensor = None
    pred_original_sample: torch.Tensor = None


class DDIMScheduler:
    """diffusers 0.14 DDIMScheduler as configured by SD-v1.x (scheduler/scheduler_config.json): scaled_linear betas
    0.00085..0.012, 1000 train steps, clip_sample False, set_alpha_to_one False, steps_offset 1, epsilon prediction."""
    order = 1
    init_noise_sigma = 1.0

    def __init__(self, num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, steps_offset=1,
                 set_alpha_to_one=False):
        betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
        self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.num_train_timesteps = num_train_timesteps
        self.steps_offset = steps_offset
        self.num_inference_steps = None
        self.timesteps = torch.arange(num_train_timesteps - 1, -1, -1)

    def set_timesteps(self, num_inference_steps, device=None):
        self.num_inference_steps = num_inference_steps
        ratio = self.num_train_timesteps // num_inference_steps
        ts = (torch.arange(0, num_inference_steps) * ratio).round().flip(0).to(torch.int64) + self.steps_offset
        self.timesteps = ts.to(device) if device is not None else ts

    def scale_model_input(self, sample, timestep=None):
        return sample

    def step(self, model_output, timestep, sample, eta=0.0, generator=None, **kw):
        t = int(timestep)
        prev_t = t - self.num_train_timesteps // self.num_inference_steps
        a_t = self.alphas_cumprod[t].to(sample.device)
        a_prev = (self.alphas_cumprod[prev_t] if prev_t >= 0 else self.final_alpha_cumprod).to(sample.device)
        eps = model_output.to(torch.float32)
        x = sample.to(torch.float32)
        pred_x0 = (x - (1 - a_t) ** 0.5 * eps) / a_t ** 0.5
        var = (1 - a_prev) / (1 - a_t) * (1 - a_t / a_prev)
        std = eta * var ** 0.5
        prev = a_prev ** 0.5 * pred_x0 + (1 - a_prev - std ** 2) ** 0.5 * eps
        if eta > 0:
            prev = prev + std * torch.randn(x.shape, generator=generator, device=x.device, dtype=x.dtype)
        return _StepOutput(prev_sample=prev.to(sample.dtype), pred_original_sample=pred_x0.to(sample.dtype))


def preprocess(image):
    """PIL image(s) / tensor -> (n,3,H,W) float tensor in [-1,1] (pipeline_stable_diffusion_e4t.py:12-27)."""
    if isinstance(image, torch.Tensor):
        return image
    import numpy as np
    if not isinstance(image, (list, tuple)):
        image = [image]
    if isinstance(image[0], torch.Tensor):
        return torch.cat(list(image), dim=0)
    arr = np.concatenate([np.array(i)[None, :] for i in image], axis=0).astype(np.float32) / 255.0
    return torch.from_numpy(2.0 * arr.transpose(0, 3, 1, 2) - 1.0)


class StableDiffusionE4TPipeline:
    def __init__(self, vae, text_encoder, tokenizer, unet, e4t_encoder, scheduler, safety_checker=None,
                 feature_extractor=None, e4t_config=None, requires_safety_checker: bool = False,
                 already_added_placeholder_token: bool = False):
        self.vae, self.text_encoder, self.tokenizer, self.unet = vae, text_encoder, tokenizer, unet
        self.e4t_encoder, self.scheduler = e4t_encoder, scheduler
        self.safety_checker, self.feature_extractor = safety_checker, feature_extractor
        if not already_added_placeholder_token:                                  # :45-53
            if self.tokenizer.add_tokens(e4t_config.placeholder_token) == 0:
                raise ValueError(f"The tokenizer already contains the token {e4t_config.placeholder_token}. Please pass "
                                 "a different `placeholder_token` that is not already in the tokenizer.")
            text_encoder.resize_token_embeddings(len(tokenizer))
        self.placeholder_token = e4t_config.placeholder_token
        self.placeholder_token_id = tokenizer.convert_tokens_to_ids(e4t_config.placeholder_token)
        ids = self.tokenizer(e4t_config.domain_class_token, add_special_tokens=False, return_tensors="pt").input_ids[0]
        assert ids.size(0) == 1                                                  # :57-58 single-token class word
        with torch.no_grad():
            self.class_embed = text_encoder.get_input_embeddings()(ids.to(text_encoder.device))      # :60
        self.domain_embed_scale = e4t_config.domain_embed_scale
        # diffusers: 2 ** (len(vae.config.block_out_channels) - 1); 8 (the SD-v1.x VAE) when no VAE is attached
        self.vae_scale_factor = 2 ** (len(vae.config.block_out_channels) - 1) if vae is not None else 8

    @property
    def _execution_device(self):
        return self.unet.device

    def prepare_for_e4t(self, prompt, device):
        """pipeline_stable_diffusion_e4t.py:64-88 (the placeholder index of the FIRST prompt is used for every row)."""
        tk = dict(padding="max_length", truncation=True, max_length=self.tokenizer.model_max_length, return_tensors="pt")
        ids_empty = self.tokenizer("", **tk).input_ids
        input_ids = self.tokenizer(prompt, **tk).input_ids
        try:
            idx = input_ids[0].tolist().index(self.placeholder_token_id)
        except ValueError:
            raise ValueError(f"Your prompt may not have the placeholder_token={self.placeholder_token}")
        ehs_e4t = self.text_encoder(ids_empty.to(device))[0]
        emb = self.text_encoder.get_input_embeddings()(input_ids.to(device)).to(dtype=self.text_encoder.dtype, device=device)
        return dict(placeholder_token_id_idx=idx, encoder_hidden_states_for_e4t=ehs_e4t, inputs_embeds=emb)

    def prepare_latents(self, batch, channels, height, width, dtype, device, generator, latents=None):
        shape = (batch, channels, height // self.vae_scale_factor, width // self.vae_scale_factor)
        if latents is None:
            if isinstance(generator, list):
                latents = torch.cat([torch.randn((1,) + shape[1:], generator=g, device=g.device, dtype=torch.float32)
                                     for g in generator]).to(device)
            else:
                gdev = generator.device if generator is not None else device
                latents = torch.randn(shape, generator=generator, device=gdev, dtype=torch.float32).to(device)
        else:
            latents = latents.to(device)
        return latents * getattr(self.scheduler, "init_noise_sigma", 1.0)

    def decode_latents(self, latents):
        if self.vae is None:
            raise NotImplementedError("no VAE attached: pass vae=AutoencoderKL(...) or use output_type='latent'")
        image = self.vae.decode(latents / 0.18215).sample
        return (image / 2 + 0.5).clamp(0, 1).cpu().permute(0, 2, 3, 1).float().numpy()

    @torch.no_grad()
    def __call__(self, prompt: Union[str, List[str]] = None, height: Optional[int] = None, width: Optional[int] = None,
                 num_inference_steps: int = 50, guidance_scale: float = 7.5, negative_prompt=None,
                 num_images_per_prompt: Optional[int] = 1, eta: float = 0.0, generator=None, latents=None,
                 output_type: Optional[str] = "pil", return_dict: bool = True, callback=None, callback_steps: int = 1,
                 cross_attention_kwargs=None, image=None, domain_embed_scale: Optional[float] = None):
        domain_embed_scale = self.domain_embed_scale if domain_embed_scale is None else domain_embed_scale
        height = height or self.unet.config.sample_size * self.vae_scale_factor
        width = width or self.unet.config.sample_size * self.vae_scale_factor
        assert negative_prompt is None, "negative_prompt is not supported"            # :153
        batch_size = 1 if isinstance(prompt, str) else len(prompt)
        device = self._execution_device
        cfg = guidance_scale > 1.0
        image = preprocess(image)
        e4t = self.prepare_for_e4t(prompt, device)
        self.scheduler.set_timesteps(num_inference_steps, device=device)
        timesteps = self.scheduler.timesteps
        latents = self.prepare_latents(batch_size * num_images_per_prompt, self.unet.in_channels, height, width,
                                       e4t["encoder_hidden_states_for_e4t"].dtype, device, generator, latents)
        bsz = latents.shape[0]
        ehs_e4t = e4t["encoder_hidden_states_for_e4t"].expand(bsz, -1, -1)
        pixel_values = image.expand(bsz, -1, -1, -1).to(device)
        # the ViT-H/14 features of the conditioning image are step-invariant: compute them once
        clip_feats = self.e4t_encoder.image_features(pixel_values) if hasattr(self.e4t_encoder, "image_features") else None
        class_embed = self.class_embed.clone().expand(bsz, -1).to(device)
        kw = {} if cross_attention_kwargs is None else dict(cross_attention_kwargs=cross_attention_kwargs)
        for i, t in enumerate(timesteps):
            model_in = torch.cat([latents] * 2) if cfg else latents                   # :183-184
            model_in = self.scheduler.scale_model_input(model_in, t)
            latents_in = self.scheduler.scale_model_input(latents, t)                 # :187
            enc = self.unet(latents_in, t, ehs_e4t, return_encoder_outputs=True)      # :191
            if clip_feats is not None:
                dom = self.e4t_encoder(x=pixel_values, unet_down_block_samples=enc["down_block_samples"],
                                       clip_features=clip_feats)
            else:
                dom = self.e4t_encoder(x=pixel_values, unet_down_block_samples=enc["down_block_samples"])   # :194
            dom = class_embed + domain_embed_scale * dom.to(class_embed.dtype)        # :196
            emb = e4t["inputs_embeds"].expand(bsz, -1, -1).clone().to(dtype=self.text_encoder.dtype, device=device)
            emb[:, e4t["placeholder_token_id_idx"], :] = dom.to(emb.dtype)            # :197-198
            ehs = self.text_encoder(inputs_embeds=emb)[0].to(dtype=self.unet.dtype, device=device)         # :200
            ctx = torch.cat([ehs_e4t.to(ehs.dtype), ehs]) if cfg else ehs             # :201
            noise_pred = self.unet(model_in, t, encoder_hidden_states=ctx, **kw).sample                     # :203-208
            if cfg:
                u, c = noise_pred.chunk(2)
                noise_pred = u + guidance_scale * (c - u)                             # :211-213
            latents = self.scheduler.step(noise_pred, t, latents, eta=eta, generator=generator).prev_sample  # :216
            if callback is not None and i % callback_steps == 0:
                callback(i, t, latents)
        if output_type == "latent":
            out = latents
        else:
            out = self.decode_latents(latents)
            if output_type == "pil":
                from PIL import Image
                out = [Image.fromarray((im * 255).round().astype("uint8")) for im in out]
        if not return_dict:
            return (out, None)
        return StableDiffusionPipelineOutput(images=out, nsfw_content_detected=None)
