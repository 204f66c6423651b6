"""The E4T pre-training step (pretrain_e4t.py:595-654) assembled from the `e4t` module mirror, with the pieces the
reference gets from accelerate/torch.optim rebuilt B200-first:

  * FlatAdamW     — all trainable parameters (WeightOffsets + encoder) re-homed into ONE fp32 arena with a matching
                    gradient arena; the optimiser is a single fused sm_100a kernel over the arena and the
                    data-parallel gradient exchange is ONE NCCL all-reduce of the gradient arena
                    (reference: DDP buckets over every requires_grad parameter, ≈4.9 GB; here 1.5 GB).
  * PretrainStep  — the loop body given explicit (pixel_values, latents, noise, timesteps, input_ids); with a VAE
                    attached, `latents` may be replaced by `latent_eps` and are then encoded on the device.
"""
import os

import torch
import torch.distributed as dist
import torch.nn.functional as F

from . import functional as FN
from . import ops

PLACEHOLDER_FALLBACK = 49408


def ddpm_alphas_cumprod(n=1000, beta_start=0.00085, beta_end=0.012, device="cpu"):
    """SD-v1.x DDPMScheduler (scaled_linear betas), as used by noise_scheduler.add_noise (pretrain_e4t.py:621)."""
    betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, n, dtype=torch.float32, device=device) ** 2
    return torch.cumprod(1.0 - betas, dim=0)


def add_noise(latents, noise, timesteps, acp):
    a = acp[timesteps] ** 0.5
    s = (1 - acp[timesteps]) ** 0.5
    return a.view(-1, 1, 1, 1) * latents + s.view(-1, 1, 1, 1) * noise


def all_reduce_sum_(flat, group=None):
    """Data-parallel exchange of a flat gradient arena: ONE all-reduce(SUM) (NCCL over NVLink/NVSwitch on GPUs,
    gloo in the CPU tests).  Returns the scale (1/world) that turns the sum into the DDP average; FlatAdamW folds it
    into the optimiser kernel instead of spending another pass over the arena."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        return 1.0 / dist.get_world_size(group)
    return 1.0


def shard_seed(base_seed, rank):
    """Per-rank data seed (the batch shards over images; ranks never exchange activations)."""
    return base_seed + 1000 * rank


class FlatAdamW:
    """torch.optim.AdamW semantics over a flat arena (amsgrad=False).  `params`: iterable of nn.Parameter."""

    def __init__(self, params, lr=1.6e-5, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8, process_group=None):
        seen, plist = set(), []
        for p in params:
            if p.requires_grad and id(p) not in seen:
                seen.add(id(p))
                plist.append(p)
        assert plist, "no trainable parameters"
        dev = plist[0].device
        assert dev.type == "cuda", "FlatAdamW runs the fused sm_100a kernel: parameters must be on a CUDA device"
        self.params = plist
        self.lr, self.betas, self.weight_decay, self.eps = lr, betas, weight_decay, eps
        self.process_group = process_group
        # storages shared by several parameters (E4TEncoder's stacked first_linears) must stay contiguous: group by
        # untyped storage and move each storage once
        groups = {}
        for p in plist:
            groups.setdefault(p.untyped_storage().data_ptr(), []).append(p)
        total = 0
        layout = []
        for sp, ps in groups.items():
            base = min(p.data_ptr() for p in ps)
            end = max(p.data_ptr() + p.numel() * 4 for p in ps)
            n = (end - base) // 4
            n_pad = (n + 3) // 4 * 4
            layout.append((ps, base, n, total))
            total += n_pad
        self.numel = total
        self.arena = torch.zeros(total, device=dev, dtype=torch.float32)
        self.grad = torch.zeros(total, device=dev, dtype=torch.float32)
        self.exp_avg = torch.zeros(total, device=dev, dtype=torch.float32)
        self.exp_avg_sq = torch.zeros(total, device=dev, dtype=torch.float32)
        with torch.no_grad():
            for ps, base, n, off in layout:
                for p in ps:
                    assert p.dtype == torch.float32 and p.is_contiguous()
                    o = off + (p.data_ptr() - base) // 4
                    self.arena[o:o + p.numel()].copy_(p.detach().reshape(-1))
                for p in ps:
                    o = off + (p.data_ptr() - base) // 4
                    p.data = self.arena[o:o + p.numel()].view(p.shape)
                    p.grad = self.grad[o:o + p.numel()].view(p.shape)
                    p._e4t_arena = True
        self.offsets = {}                                                # id(param) -> (offset, numel) in the arena
        for ps, base, n, off in layout:
            for p in ps:
                self.offsets[id(p)] = (off + (p.data_ptr() - self.arena.data_ptr()) // 4 - off, p.numel())
        self.step_count = 0
        self.step_dev = torch.zeros(1, device=dev, dtype=torch.int32)   # device-side counter: graph-replayable
        FN.DIRECT_GRAD_WRITE = True     # .grad views are zeroed by zero_grad(); WO kernels write them directly
        FN.bump_param_epoch()
        # modules that cache views of re-homed storages refresh themselves lazily (E4TEncoder._stacked)

    def zero_grad(self, set_to_none=False):
        self.grad.zero_()

    def all_reduce_grads(self, start=0, end=None):
        """Data-parallel gradient exchange: NCCL all-reduce (SUM) of the gradient arena (or of the slice
        [start, end)); the 1/world average is folded into the optimiser kernel's grad_scale."""
        g = self.grad if (start == 0 and end is None) else self.grad[start:end]
        return all_reduce_sum_(g, self.process_group)

    def prefix_end(self, params):
        """End offset of the arena prefix that holds exactly `params` (None if they are not a contiguous prefix)."""
        ids = {id(p) for p in params}
        if not ids:
            return None
        end = max(self.offsets[i][0] + self.offsets[i][1] for i in ids)
        inside = sum(n for i, (o, n) in self.offsets.items() if o < end)
        mine = sum(self.offsets[i][1] for i in ids)
        return (end + 3) // 4 * 4 if inside == mine else None

    def step(self, grad_scale=1.0):
        self.step_count += 1
        ops.adamw_step_dev(self.arena, self.grad, self.exp_avg, self.exp_avg_sq, self.lr, self.betas[0], self.betas[1],
                           self.eps, self.weight_decay, self.step_dev, grad_scale)
        FN.bump_param_epoch()


    # ---- checkpoint / resume (pretrain_e4t.py:536-558 resumes optimizer state through accelerator.load_state) ------
    def state_dict(self):
        """Moments and step count (clones, not arena views).  Parameters themselves travel in weight_offsets.pt /
        encoder.pt; `numel` guards against loading into a differently laid-out arena."""
        return dict(numel=self.numel, step=self.step_count, exp_avg=self.exp_avg.detach().clone(),
                    exp_avg_sq=self.exp_avg_sq.detach().clone(), lr=self.lr, betas=self.betas,
                    weight_decay=self.weight_decay, eps=self.eps)

    def load_state_dict(self, sd):
        if int(sd["numel"]) != self.numel:
            raise ValueError(f"optimizer arena size mismatch: checkpoint {sd['numel']} vs {self.numel}")
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.step_count = int(sd["step"])
        self.step_dev.fill_(self.step_count)
        for k in ("lr", "betas", "weight_decay", "eps"):
            if k in sd:
                setattr(self, k, tuple(sd[k]) if k == "betas" else sd[k])


def trainable_parameters(unet, e4t_encoder, tune_unet=False):
    """Pre-training (pretrain_e4t.py:274-278): encoder params with requires_grad + UNet params whose name has 'wo'.
    The reference leaves every base UNet weight at requires_grad=True, computes (and all-reduces) their gradients and
    never applies them; here they are frozen, which changes no result and lets the kernels skip ~0.8 TFLOP/img of
    weight-gradient work.  Domain tuning (tuning_e4t.py:139-146, tune_unet=True): encoder params + ALL UNet params."""
    ps = [p for p in e4t_encoder.parameters() if p.requires_grad]
    for n, p in unet.named_parameters():
        p.requires_grad_(bool(tune_unet) or "wo" in n)
        if p.requires_grad:
            ps.append(p)
    return ps


class PretrainStep:
    """One optimisation step == pretrain_e4t.py:595-654 on explicit inputs."""

    def __init__(self, unet, e4t_encoder, text_encoder, placeholder_token_id, class_token_id, lr=1.6e-5,
                 betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8, domain_embed_scale=0.1, reg_lambda=0.01,
                 bos_id=49406, eos_id=49407, weight_dtype=torch.bfloat16, optimizer=True, tune_unet=False,
                 max_grad_norm=None, vae=None):
        self.unet, self.enc, self.text = unet, e4t_encoder, text_encoder
        # frozen AutoencoderKL (pretrain_e4t.py:262): batches without `latents` are encoded from their pixel_values
        self.vae = vae
        if vae is not None:
            vae.requires_grad_(False)
        self.placeholder_token_id = placeholder_token_id
        self.domain_embed_scale, self.reg_lambda = domain_embed_scale, reg_lambda
        self.weight_dtype = weight_dtype
        dev = unet.device
        self.acp = ddpm_alphas_cumprod(device=dev)
        self.text.requires_grad_(False)                                                  # pretrain_e4t.py:262-263
        emb = self.text.get_input_embeddings()
        with torch.no_grad():
            self.class_embed = emb(torch.tensor([class_token_id], device=dev)).float()   # :561-564  (1,768)
            ids = torch.tensor([[bos_id] + [eos_id] * 76], device=dev)
            self.ehs_e4t = self.text(input_ids=ids)[0].to(weight_dtype)                  # :565-583  (1,77,768)
        # tune_unet / max_grad_norm: the domain-tuning step (tuning_e4t.py:270-338): every UNet weight trainable,
        # global gradient-norm clipping over UNet + encoder parameters (:329-335)
        self.tune_unet, self.max_grad_norm = tune_unet, max_grad_norm
        self.opt = FlatAdamW(trainable_parameters(unet, e4t_encoder, tune_unet), lr=lr, betas=betas,
                             weight_decay=weight_decay, eps=eps) if optimizer else None
        self._graph = None
        self.wo_bank = None
        self._wo_factor_exchange = False
        # Data parallel: the encoder-head gradients (925 MB of the 1.5 GB arena, an arena prefix) are final as soon as
        # the head's backward has run — before the encoder-half UNet backward.  Their all-reduce is issued at that
        # moment on a communication stream and overlaps that backward; only the WeightOffsets slice (produced by the
        # bank at the very end of backward) is exchanged after it.  (Round 1: one exposed 1.5 GB all-reduce, 3.8 ms.)
        self._comm = None
        self._early_end = None
        self._early_fired = False
        if (self.opt is not None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
                and not any(p.requires_grad for p in e4t_encoder.clip_vision.parameters())):
            self._early_end = self.opt.prefix_end([p for p in e4t_encoder.parameters() if p.requires_grad])
            if self._early_end is not None:
                self._comm = torch.cuda.Stream()
                FN.GRAD_READY_HOOKS["encoder_head"] = self._early_all_reduce
        if self.opt is not None:
            from .wobank import WOBank
            from e4t.models.cross_attention import CrossAttention
            attns = [m for m in unet.modules() if isinstance(m, CrossAttention)]
            self.wo_bank = WOBank(attns)
            for m in attns:
                m._wo_bank = self.wo_bank
            # Data parallel, head slice exchanged early, and everything behind it in the arena is WeightOffsets
            # parameters: the bank exchanges its ~2 MB of G reductions inside backward and the 573 MB parameter-gradient
            # slice is never all-reduced (E4T_WO_FACTOR_EXCHANGE=0 keeps the slice exchange).
            self._wo_factor_exchange = False
            if self._early_end is not None and os.environ.get("E4T_WO_FACTOR_EXCHANGE", "1") != "0":
                rest = {i for i, (o, n) in self.opt.offsets.items() if o >= self._early_end}
                if rest == {id(p) for p in self.wo_bank.params}:
                    self.wo_bank.dp_group = True
                    self._wo_factor_exchange = True

    def placeholder_idxs(self, input_ids):
        """[ids.index(placeholder_id) for ids in input_ids] (pretrain_e4t.py:617) — exact integer bookkeeping."""
        return [row.index(self.placeholder_token_id) for row in input_ids.cpu().tolist()]

    def forward_loss(self, batch):
        pixel_values, noise = batch["pixel_values"], batch["noise"]
        timesteps, input_ids = batch["timesteps"], batch["input_ids"]
        latents = batch.get("latents")
        if latents is None and self.vae is not None:
            # pretrain_e4t.py:597-599 with the sample's ε taken from the batch (like `noise`), so that the encode is
            # part of a captured step: latent_dist.sample() == mean + std * ε
            with torch.no_grad():
                d = self.vae.encode(pixel_values).latent_dist
                latents = (d.mean + d.std * batch["latent_eps"]) * self.vae.config.scaling_factor
        elif latents is None:
            raise KeyError("batch has no 'latents' and no VAE is attached to encode its pixel_values")
        B = latents.shape[0]
        emb = self.text.get_input_embeddings()
        with torch.no_grad():
            inputs_embeds = emb(input_ids)                                               # :616
        idxs = batch.get("placeholder_idxs")
        if idxs is None:
            idxs = self.placeholder_idxs(input_ids)                                      # :617
        noisy = add_noise(latents, noise, timesteps, self.acp)                           # :621
        enc = self.unet(noisy, timesteps, self.ehs_e4t.expand(B, -1, -1), return_encoder_outputs=True)   # :624
        domain_embed = self.enc(x=pixel_values, unet_down_block_samples=enc["down_block_samples"])       # :626
        domain_embed = self.class_embed.clone().expand(B, -1) + self.domain_embed_scale * domain_embed.float()  # :628
        # per-sample in-place row overwrite (:630-631) as one differentiable index_put
        rows = torch.arange(B, device=latents.device)
        cols = torch.as_tensor(idxs, device=latents.device)
        inputs_embeds = inputs_embeds.to(domain_embed.dtype).index_put((rows, cols), domain_embed)
        ehs = self.text(inputs_embeds=inputs_embeds.to(self.text.dtype))[0].to(self.weight_dtype)        # :634
        pred = self.unet(noisy, timesteps, ehs).sample                                   # :636
        loss_diff = F.mse_loss(pred.float(), noise.float(), reduction="mean")            # :645
        loss_reg = self.reg_lambda * domain_embed.pow(2).sum()                           # :646
        return dict(loss=loss_diff + loss_reg, loss_diff=loss_diff, loss_reg=loss_reg, pred=pred,
                    domain_embed=domain_embed, placeholder_idxs=idxs)

    # ---- whole-step CUDA graph (forward + backward + all-reduce + AdamW) -------------------------------------
    def enable_cuda_graph(self, example_batch, warmup=3):
        """Capture one full step into a CUDA graph.  `example_batch` fixes shapes; it must carry `placeholder_idxs`
        as a device tensor (the host-side index search of pretrain_e4t.py:617 cannot run inside a graph).
        Afterwards __call__ copies the batch into the static input buffers and replays."""
        assert self.opt is not None and torch.is_tensor(example_batch.get("placeholder_idxs"))
        import gc
        self._static = {k: v.clone() for k, v in example_batch.items()}
        # Warm-up and capture run on ONE side stream, and every reference to earlier autograd graphs is dropped
        # first: an AccumulateGrad node that survives from an eager step on the default stream would make the captured
        # backward synchronise with the legacy stream and invalidate the capture.
        self._drop_autograd_refs()
        gc.collect()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        # Data parallel runs keep the NCCL all-reduce and the optimiser kernel OUTSIDE the graph (three eager launches):
        # collectives captured into a graph must be captured identically on every rank and interact with the
        # process-group watchdog; the compute part (forward + backward) is what has thousands of launches.
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        with torch.cuda.stream(side):
            for _ in range(warmup):
                out = self._eager_step(self._static)
                del out
            self._drop_autograd_refs()
        gc.collect()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()

        def capture(body, mode):
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side, capture_error_mode=mode):
                out = body(self._static)
                self._static_out = {k: out[k].detach() for k in ("loss", "loss_diff", "loss_reg")}
                del out
            return graph

        # Data parallel: first try to capture the WHOLE step including the NCCL all-reduces (forked onto the comm stream
        # inside the capture) and AdamW; if this torch/NCCL build refuses, capture forward+backward only and keep the
        # exchange + optimiser as three eager launches (the round-1 behaviour).
        self._graph_has_opt = True
        if multi and os.environ.get("E4T_GRAPH_NCCL", "1") != "0":
            try:
                graph = capture(self._eager_step, "thread_local")
            except Exception as ex:   # noqa: BLE001
                self._capture_note = f"NCCL-in-graph capture failed ({type(ex).__name__}: {str(ex)[:120]}); compute-only graph"
                self._early_fired = False
                self._comm = None               # no collective inside the compute-only graph
                self._disable_wo_factor_exchange()
                torch.cuda.synchronize()
                self._drop_autograd_refs()
                gc.collect()
                self._graph_has_opt = False
                graph = capture(self._fwd_bwd, "thread_local")
        elif multi:
            self._comm = None
            self._disable_wo_factor_exchange()
            self._graph_has_opt = False
            graph = capture(self._fwd_bwd, "thread_local")
        else:
            graph = capture(self._eager_step, "global")
        self._drop_autograd_refs()
        self._graph = graph
        return self

    def _disable_wo_factor_exchange(self):
        """Compute-only graph (no collective may be captured): the bank's in-backward all-reduce goes too; the
        WeightOffsets slice is then exchanged with the rest of the arena after the graph."""
        if self.wo_bank is not None:
            self.wo_bank.dp_group = None
        self._wo_factor_exchange = False

    def release_cuda_graph(self):
        """Drop the captured step (and its static buffers).  Call before `dist.destroy_process_group()`: a live graph
        with captured NCCL kernels keeps the communicator referenced and the destroy waits for it."""
        self._graph = None
        self._static_out = None
        self._static = None
        self._drop_autograd_refs()
        import gc
        gc.collect()
        if torch.cuda.is_available():
            torch.cuda.synchronize()

    def _drop_autograd_refs(self):
        if self.wo_bank is not None:
            self.wo_bank.drop_autograd_refs()
        for m in self.unet.modules():
            c = getattr(m, "_weff_cache", None)
            if c is not None:
                c.clear()

    def __call__(self, batch):
        if self._graph is not None:
            for k, v in batch.items():
                self._static[k].copy_(v, non_blocking=True)
            self._graph.replay()
            FN.bump_param_epoch()        # the replayed AdamW moved the parameters behind torch's version counters
            if not self._graph_has_opt:
                self._apply_optimizer()
            return dict(self._static_out)
        return self._eager_step(batch)

    def _fwd_bwd(self, batch):
        out = self.forward_loss(batch)
        out["loss"].backward()                                                           # :648
        return out

    def _early_all_reduce(self):
        """Fired from inside backward (functional.MeanPoolCatFn): all-reduce the encoder-head slice on the comm stream."""
        if self._comm is None or self._early_fired:
            return
        main = torch.cuda.current_stream()
        self._comm.wait_stream(main)
        with torch.cuda.stream(self._comm):
            self.opt.all_reduce_grads(0, self._early_end)
        self._early_fired = True

    def _apply_optimizer(self):
        if self.opt is not None:
            if self._early_fired:
                torch.cuda.current_stream().wait_stream(self._comm)
                if self._wo_factor_exchange:      # the bank summed its gradients over the ranks inside backward
                    scale = 1.0 / dist.get_world_size()
                else:
                    scale = self.opt.all_reduce_grads(self._early_end, None)
                self._early_fired = False
            elif self._wo_factor_exchange:        # head hook did not fire: its slice still needs the exchange, the bank's does not
                scale = self.opt.all_reduce_grads(0, self._early_end)
            else:
                scale = self.opt.all_reduce_grads()
            if self.max_grad_norm is not None:
                # accelerator.clip_grad_norm_ (tuning_e4t.py:329-335) == torch clip_grad_norm_: one norm over the flat
                # gradient arena (its padding is zero), coefficient kept on the device (graph-replayable)
                total = torch.linalg.vector_norm(self.opt.grad) * scale
                self.opt.grad.mul_(torch.clamp(self.max_grad_norm / (total + 1e-6), max=1.0))
            self.opt.step(scale)                                                         # :652
            self.opt.zero_grad()                                                         # :654

    def _eager_step(self, batch):
        out = self._fwd_bwd(batch)
        self._apply_optimizer()
        return out


def TuningStep(unet, e4t_encoder, text_encoder, placeholder_token_id, class_token_id, lr=1.6e-5, reg_lambda=1e-4,
               max_grad_norm=1.0, **kw):
    """One optimisation step of tuning_e4t.py:270-338 (BASELINE.json configs[3]): the pre-training step with every UNet
    weight and the encoder trainable, reg_lambda 1e-4 (tuning_e4t.py:31) and gradient-norm clipping at 1.0 (:38)."""
    return PretrainStep(unet, e4t_encoder, text_encoder, placeholder_token_id, class_token_id, lr=lr,
                        reg_lambda=reg_lambda, tune_unet=True, max_grad_norm=max_grad_norm, **kw)
