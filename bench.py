#!/usr/bin/env python
"""bench.py — E4T pre-training throughput on B200 (BASELINE.json metric: images/sec @512², per-GPU bs16, SD-v1.4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 16] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (pretrain_e4t.py:595-654: UNet encoder-half -> E4T encoder -> text encoder ->
full UNet -> loss -> backward -> AdamW) over one batch of synthetic 512² inputs with random-init SD-v1.4 + ViT-H/14
weights.  Prints ONE JSON line (rank 0).  `value` = device-resident throughput (inputs already in HBM), `e2e` = the
same through the public API with pinned-host inputs copied every step and the loss read back every step.
`--impl reference` times the CPU oracle (oracle/e4t_oracle.py, the restated reference path) on the host cores.
`--dump-outputs DIR` writes what the last timed step produced as DIR/<name>.npy (float32), so that two builds run with
the same arguments (hence the same seeded weights and inputs) can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "e4t-diffusion_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "E4T pretrain images/sec @512^2 bs16 SD-v1.4"
SD14 = dict(in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280), layers_per_block=2,
            attention_head_dim=8, cross_attention_dim=768, norm_num_groups=32, norm_eps=1e-5, sample_size=64)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16, help="per-GPU batch (BASELINE config: 16)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_stock"],
                    help="reference = the reference's CPU path on the host cores; torch_stock = the same step in stock torch "
                         "ops (cuBLAS/cuDNN/SDPA, bf16 autocast) on the GPU: the on-box library comparator")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's losses and a fixed sample of the updated trainable "
                         "parameters and AdamW first moments as DIR/<name>.npy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-micro", action="store_true")
    ap.add_argument("--profile-one-step", action="store_true", help="run W warm-up + 1 step and exit (for ncu)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of the whole-step CUDA graph")
    ap.add_argument("--unfreeze-clip-vision", action="store_true",
                    help="the README recipe's variant (README.md:52, pretrain_e4t.py:78,249): the ViT-H/14 tower trains too "
                         "(+630.8 M parameters in the optimiser and the all-reduce); reported separately, SURVEY.md §8d")
    ap.add_argument("--tuning", action="store_true",
                    help="BASELINE configs[3]: the domain-tuning step (tuning_e4t.py:270-338): every UNet weight trainable, "
                         "one image repeated over the batch, grad-norm clipping at 1.0")
    return ap.parse_args()


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(bf16_burst=d.get("bf16_tflops", 1590.0), bf16_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi, DURING the timed region)
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# model / data
# ------------------------------------------------------------------------------------------------------------------
def build_models(device, freeze_clip_vision=True):
    from e4t.encoder import E4TEncoder
    from e4t.models.modeling_clip import CLIPTextConfig, CLIPTextModel
    from e4t.models.unet_2d_condition import UNet2DConditionModel
    torch.manual_seed(0)
    with torch.device(device):
        unet = UNet2DConditionModel(cross_attention_dim=768, sample_size=64)     # SD-v1.4 config (defaults + 768)
        enc = E4TEncoder(word_embedding_dim=768, arch="ViT-H-14", freeze_clip_vision=freeze_clip_vision)
        text = CLIPTextModel(CLIPTextConfig(vocab_size=49409))
    text.to(torch.bfloat16)                                                      # pretrain_e4t.py:422-423
    return unet, enc, text


TEMPLATE_WORDS = [4, 4, 5, 5, 5, 6, 6, 6, 5, 6]   # placeholder index for the 10 templates (pretrain_e4t.py:36-47)


def host_batch(B, seed, pinned=True):
    """Synthetic per-step inputs on the host (SURVEY.md §8d)."""
    import random
    g = torch.Generator().manual_seed(seed)
    rnd = random.Random(seed)
    idxs = [TEMPLATE_WORDS[t] for t in rnd.choices(range(10), k=B)]
    ids = torch.full((B, 77), 49407, dtype=torch.int64)
    ids[:, 0] = 49406
    for i, ix in enumerate(idxs):
        ids[i, 1:ix] = torch.randint(300, 4000, (ix - 1,), generator=g)
        ids[i, ix] = 49408
    b = dict(pixel_values=torch.rand(B, 3, 512, 512, generator=g) * 2 - 1,
             latents=torch.randn(B, 4, 64, 64, generator=g) * 0.18215, noise=torch.randn(B, 4, 64, 64, generator=g),
             timesteps=torch.randint(0, 1000, (B,), generator=g, dtype=torch.int64), input_ids=ids,
             placeholder_idxs=torch.tensor(idxs, dtype=torch.int64))
    if pinned:
        b = {k: v.pin_memory() for k, v in b.items()}
    return b


DUMP_SAMPLE = 1 << 22      # entries of each sampled optimiser buffer: 2 x 16 MB of float32


def dump_outputs(dirname, out, opt):
    """The step's loss terms as returned to the caller, and the same seeded sample of the flat parameter arena and of
    AdamW's first moment (the latter carries the gradients, which the sign-like early AdamW update mostly hides)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    idx = torch.randint(0, opt.arena.numel(), (min(DUMP_SAMPLE, opt.arena.numel()),),
                        generator=torch.Generator().manual_seed(0)).to(opt.arena.device)
    arrays = {k: v.detach().float() for k, v in out.items() if torch.is_tensor(v) and v.is_floating_point()}
    arrays.update(params_sample=opt.arena[idx], exp_avg_sample=opt.exp_avg[idx])
    for k, v in arrays.items():
        np.save(os.path.join(dirname, f"{k}.npy"), v.cpu().numpy().astype(np.float32))


def to_device(b, device):
    return {k: v.to(device, non_blocking=True) for k, v in b.items()}


def batch_bytes(b):
    return int(sum(v.numel() * v.element_size() for v in b.values()))


# ------------------------------------------------------------------------------------------------------------------
# micro-timing of the dominant kernels (CUDA events on the launching stream, L2 flushed between launches)
# ------------------------------------------------------------------------------------------------------------------
def micro_rooflines(B, peaks, device):
    from e4t_b200 import ops
    res = {}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)   # > 126 MB L2

    def timeit(fn, iters=8):
        fn(); fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2] * 1e-3

    g = torch.Generator(device=device).manual_seed(1)
    # (1) attention core, level-0 self-attention: N=M=4096, 8 heads x dh 40  (59% of attention FLOPs, SURVEY §7)
    N, C, H = 4096, 320, 8
    qkv = (torch.randn(B, N, 3 * C, device=device, generator=g) * 0.5).to(torch.bfloat16)
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    t = timeit(lambda: ops.attn_fwd(q, k, v, H))
    fl = 4.0 * N * N * C * B
    res["attn_fwd_L0_self"] = dict(ms=t * 1e3, tflops=fl / t / 1e12, flops=fl)
    o, lse = ops.attn_fwd(q, k, v, H)
    do = torch.randn_like(o)
    t = timeit(lambda: ops.attn_bwd(q, k, v, o, do, lse, H))
    res["attn_bwd_fused_L0_self"] = dict(ms=t * 1e3, tflops=2.0 * fl / t / 1e12, flops=2.0 * fl,
                                         note="SURVEY.md §8d: backward = 2x forward (dQ, dK, dV, dP; the S recompute is not counted)")
    # (2) fused WO-modulated QKV projection GEMM, level 0: (B*4096, 320) x (960, 320)^T
    x = (torch.randn(B * N, C, device=device, generator=g)).to(torch.bfloat16)
    w = (torch.randn(3 * C, C, device=device, generator=g) * 0.05).to(torch.bfloat16)
    t = timeit(lambda: ops.gemm(x, w))
    fl2 = 2.0 * B * N * C * 3 * C
    res["qkv_proj_L0"] = dict(ms=t * 1e3, tflops=fl2 / t / 1e12, flops=fl2)
    # (3) GEGLU projection GEMM level 1 (B*1024, 640) x (5120, 640)^T and (4) 3x3 conv 320->320 @64x64
    x1 = torch.randn(B * 1024, 640, device=device, generator=g).to(torch.bfloat16)
    w1 = (torch.randn(5120, 640, device=device, generator=g) * 0.05).to(torch.bfloat16)
    t = timeit(lambda: ops.gemm(x1, w1))
    res["ff_proj_L1"] = dict(ms=t * 1e3, tflops=2.0 * B * 1024 * 640 * 5120 / t / 1e12)
    xc = torch.randn(B, 64, 64, 320, device=device, generator=g).to(torch.bfloat16)
    wc = (torch.randn(9, 320, 320, device=device, generator=g) * 0.05).to(torch.bfloat16)
    t = timeit(lambda: ops.conv3x3(xc, wc))
    res["conv3x3_320_64"] = dict(ms=t * 1e3, tflops=2.0 * B * 4096 * 9 * 320 * 320 / t / 1e12)
    # (5) HBM-bound: GroupNorm+SiLU 320ch @64x64
    gam = torch.ones(320, device=device); bet = torch.zeros(320, device=device)
    t = timeit(lambda: ops.groupnorm_fwd(xc, gam, bet, 32, 1e-5, True))
    byts = xc.numel() * 2 * 3  # stats read + apply read + write
    res["groupnorm_silu_320_64"] = dict(ms=t * 1e3, gbs=byts / t / 1e9, frac_hbm=byts / t / 1e9 / peaks["hbm"])
    del flush
    return res


def attention_aggregate(B, peaks, device):
    """SURVEY.md §8d aggregate for the 'fused WeightOffsets-attention' of north_star: WO-modulated QKV projections +
    attention core, forward and backward, over BOTH UNet passes of a step (759 GFLOP per image per step, out-proj
    excluded, backward = 2x forward).  Every distinct kernel signature is timed alone (CUDA events, L2 flushed) and
    weighted by its call count in the step; FLOPs are the analytic figure F = 2·N·Rq·C + 4·M·Rkv·C + 4·N·M·C per module."""
    from e4t_b200 import ops
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)

    def timeit(fn, iters=5):
        fn(); fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2] * 1e-3

    bf = torch.bfloat16
    levels = [(4096, 320, 5, 2), (1024, 640, 5, 2), (256, 1280, 5, 2), (64, 1280, 1, 1)]   # (N, C, modules full, enc-half)
    H, Mx, Rx = 8, 77, 768
    tot_t = tot_f = 0.0
    rows = []
    for N, C, n_full, n_enc in levels:
        cnt = n_full + n_enc
        x = torch.randn(B, N, C, device=device).to(bf)
        ctx = torch.randn(B, Mx, Rx, device=device).to(bf)
        w3 = (torch.randn(3 * C, C, device=device) * 0.05).to(bf)
        w1 = (torch.randn(C, C, device=device) * 0.05).to(bf)
        wkv = (torch.randn(2 * C, Rx, device=device) * 0.05).to(bf)
        x2, c2 = x.view(-1, C), ctx.view(-1, Rx)
        # ---- self-attention module
        qkv = ops.gemm(x2, w3).view(B, N, 3 * C)
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        o, lse = ops.attn_fwd(q, k, v, H)
        do, dqkv = torch.randn_like(o), torch.randn_like(qkv)
        dw = torch.zeros(3 * C, C, device=device)
        t_self = (timeit(lambda: ops.gemm(x2, w3)) + timeit(lambda: ops.attn_fwd(q, k, v, H))
                  + timeit(lambda: ops.attn_bwd(q, k, v, o, do, lse, H))
                  + timeit(lambda: ops.gemm(dqkv.view(-1, 3 * C), w3, b_mn=True))
                  + timeit(lambda: ops.gemm(dqkv.view(-1, 3 * C), x2, a_mn=True, b_mn=True, out=dw, accumulate=True, splits=8)))
        f_self = 3.0 * B * (2.0 * N * C * 3 * C + 4.0 * N * N * C)
        # ---- cross-attention module
        qc = ops.gemm(x2, w1).view(B, N, C)
        kv = ops.gemm(c2, wkv).view(B, Mx, 2 * C)
        kc, vc = kv[..., :C], kv[..., C:]
        oc, lsec = ops.attn_fwd(qc, kc, vc, H)
        dkv = torch.randn_like(kv)
        dw1, dwkv = torch.zeros(C, C, device=device), torch.zeros(2 * C, Rx, device=device)
        t_cross = (timeit(lambda: ops.gemm(x2, w1)) + timeit(lambda: ops.gemm(c2, wkv))
                   + timeit(lambda: ops.attn_fwd(qc, kc, vc, H)) + timeit(lambda: ops.attn_bwd(qc, kc, vc, oc, do, lsec, H))
                   + timeit(lambda: ops.gemm(do.view(-1, C), w1, b_mn=True)) + timeit(lambda: ops.gemm(dkv.view(-1, 2 * C), wkv, b_mn=True))
                   + timeit(lambda: ops.gemm(do.view(-1, C), x2, a_mn=True, b_mn=True, out=dw1, accumulate=True, splits=8))
                   + timeit(lambda: ops.gemm(dkv.view(-1, 2 * C), c2, a_mn=True, b_mn=True, out=dwkv, accumulate=True, splits=2)))
        f_cross = 3.0 * B * (2.0 * N * C * C + 4.0 * Mx * Rx * C + 4.0 * N * Mx * C)
        tot_t += cnt * (t_self + t_cross)
        tot_f += cnt * (f_self + f_cross)
        rows.append(dict(N=N, C=C, modules=cnt, self_ms=t_self * 1e3, self_tflops=f_self / t_self / 1e12,
                         cross_ms=t_cross * 1e3, cross_tflops=f_cross / t_cross / 1e12))
        del x, ctx, qkv, o, do, dqkv, qc, kv, oc
    del flush
    ach = tot_f / tot_t / 1e12
    return dict(kernels="WO-modulated QKV projection GEMMs + attention core, fwd + bwd, all 32 modules x both UNet passes",
                gflop_per_image_per_step=tot_f / B / 1e9, ms_per_step=tot_t * 1e3, achieved=ach,
                peak=peaks["bf16_sustained"], unit="TFLOP/s", frac=ach / peaks["bf16_sustained"],
                peak_source=peaks["source"] + ", sustained figure (kernels run inside a long step)", by_level=rows)


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference path) — bounded sample
# ------------------------------------------------------------------------------------------------------------------
def cpu_oracle_setup():
    from oracle import e4t_oracle as O
    # more threads than ~32 only add synchronisation overhead to these (small-batch) CPU GEMMs/convs
    torch.set_num_threads(min(os.cpu_count(), 32))
    g = torch.Generator().manual_seed(0)

    def rnd_sd(shapes):
        sd = {}
        for k, s in shapes.items():
            if k.endswith(".v"):
                sd[k] = torch.ones(1)
            elif len(s) >= 2:
                fan = 1
                for d in s[1:]:
                    fan *= d
                sd[k] = torch.empty(s).uniform_(-1, 1, generator=g) / fan ** 0.5
            elif k.endswith("weight"):
                sd[k] = torch.ones(s)
            else:
                sd[k] = torch.zeros(s)
        return sd

    sd_u = rnd_sd(O.unet_param_shapes(O.SD14_UNET))
    sd_e = rnd_sd(O.encoder_param_shapes(O.VIT_H14))
    sd_t = rnd_sd(O.text_param_shapes(O.CLIP_TEXT_L))
    train = [v for k, v in sd_u.items() if "wo" in k] + [v for k, v in sd_e.items() if not k.startswith("clip_vision.")]
    for v in train:
        v.requires_grad_(True)
    opt = torch.optim.AdamW(train, lr=1.6e-5)
    return O, sd_u, sd_e, sd_t, opt


def cpu_oracle_step(state, B, seed):
    O, sd_u, sd_e, sd_t, opt = state
    batch = O.synth_batch(B, seed)
    t0 = time.perf_counter()
    out = O.pretrain_step(sd_u, O.SD14_UNET, sd_e, O.VIT_H14, sd_t, O.CLIP_TEXT_L, batch)
    opt.zero_grad()
    out["loss"].backward()
    opt.step()
    return time.perf_counter() - t0, float(out["loss"])


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    state = cpu_oracle_setup()
    cores = torch.get_num_threads()
    B = 2                                                      # BASELINE.json configs[0]: bs=2, 10 steps, CPU fp32
    t_w, _ = cpu_oracle_step(state, B, 1)                      # 1 warm-up step (also sizes the run)
    budget = 240.0
    want = 10 if args.steps <= 0 else min(args.steps, 10)
    steps = max(1, min(want, int(budget // max(t_w, 1e-3))))
    ts = []
    for i in range(steps):
        t, _ = cpu_oracle_step(state, B, 2 + i)
        ts.append(t)
    tot = sum(ts)
    val = B * steps / tot
    sample = (f"BASELINE configs[0] (bs=2, 10 steps, CPU fp32): {steps} timed step(s) after 1 warm-up"
              f"{'' if steps == 10 else ' (capped to ~%d s of CPU work)' % int(budget)} of the full pre-training step, "
              f"SD-v1.4 UNet + ViT-H/14 + CLIP-L text, torch.set_num_threads({cores}) of {os.cpu_count()} host cores")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/sec", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": tot / steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "SD-v1.4 E4T pretrain step, random-init, 512^2 (CPU oracle port of the reference path)",
                       "per_step_batch": B, "device": "host CPU", "same_model_as_gpu_arm": True},
            "cpu_baseline": {"value": val, "unit": "images/sec", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def run_torch_stock(args):
    """--impl torch_stock: the SAME step expressed in stock torch ops on the GPU (F.conv2d / F.linear -> cuDNN / cuBLAS,
    F.scaled_dot_product_attention, torch autograd, torch.optim.AdamW(fused), bf16 autocast, fp32 masters): what the
    reference's modules would launch on this B200 (SURVEY.md §2.2).  Comparator only — never on the product path."""
    from oracle import e4t_oracle as O
    assert torch.cuda.is_available()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    O.USE_SDPA = True
    state = cpu_oracle_setup()
    _, sd_u, sd_e, sd_t, _ = state
    for sd in (sd_u, sd_e, sd_t):
        for k in list(sd):
            rg = sd[k].requires_grad
            sd[k] = sd[k].detach().to(dev).requires_grad_(rg)
    train = [v for v in list(sd_u.values()) + list(sd_e.values()) if v.requires_grad]
    opt = torch.optim.AdamW(train, lr=1.6e-5, fused=True)
    B = args.batch
    batches = [{k: v.to(dev) for k, v in O.synth_batch(B, 42 + i).items()} for i in range(2)]

    def one(b):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = O.pretrain_step(sd_u, O.SD14_UNET, sd_e, O.VIT_H14, sd_t, O.CLIP_TEXT_L, b)
        opt.zero_grad(set_to_none=True)
        out["loss"].backward()
        opt.step()
        return out["loss"]
    for i in range(max(args.warmup, 1)):
        one(batches[i % 2])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = one(batches[i % 2])
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    print(json.dumps({"impl": "torch_stock", "metric": METRIC, "value": B * args.steps / t, "unit": "images/sec",
                      "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3,
                      "higher_is_better": True, "dtype": "bf16 autocast", "data": "synthetic", "loss": float(loss),
                      "config": {"workload": "same step in stock torch ops (cuBLAS/cuDNN/SDPA), eager, all base-weight "
                                             "gradients skipped like our arm (only wo + encoder head require grad)",
                                 "per_gpu_batch": B}}))


# ------------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.impl == "torch_stock":
        run_torch_stock(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback "
                         "(use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    from e4t_b200 import _lib
    from e4t_b200.engine import PretrainStep
    _lib.load()
    peaks = load_peaks()
    B = args.batch

    unet, enc, text = build_models(device, freeze_clip_vision=not args.unfreeze_clip_vision)
    if args.tuning:
        from e4t_b200.engine import TuningStep
        step = TuningStep(unet, enc, text, placeholder_token_id=49408, class_token_id=320, lr=1.6e-5,
                          weight_dtype=torch.bfloat16)
    else:
        step = PretrainStep(unet, enc, text, placeholder_token_id=49408, class_token_id=320, lr=1.6e-5,
                            weight_dtype=torch.bfloat16)
    n_train = step.opt.numel

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(n, batches, e2e):
        """n steps; returns device time (s) via CUDA events, the last loss and the last step's outputs."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        last = out = None
        for i in range(n):
            hb = batches[i % len(batches)]
            # e2e: pinned host -> device every step (straight into the graph's static inputs when graphed)
            b = (hb if step._graph is not None else to_device(hb, device)) if e2e else hb
            out = step(b)
            if e2e:
                last = out["loss"].item()          # device -> host read of the step result
            else:
                last = out["loss"]
        e1.record()
        barrier()
        t = e0.elapsed_time(e1) * 1e-3
        if world > 1:
            tt = torch.tensor([t], device=device)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = tt.item()
        return t, (last if isinstance(last, float) else float(last)), out

    host_batches = [host_batch(B, 42 + rank * 1000 + i) for i in range(4)]
    if args.tuning:      # one image (and its latents) repeated over the batch, fresh noise / timesteps per step (:266-281)
        for hb in host_batches:
            hb["pixel_values"] = host_batches[0]["pixel_values"][:1].expand(B, -1, -1, -1).contiguous().pin_memory()
            hb["latents"] = host_batches[0]["latents"][:1].expand(B, -1, -1, -1).contiguous().pin_memory()
    dev_batches = [to_device(hb, device) for hb in host_batches]
    h2d = batch_bytes(host_batches[0])

    # warm-up (also builds the bf16 operand caches and first-call attributes)
    run_steps(max(args.warmup, 1), dev_batches, False)
    cuda_graph = False
    if not args.no_graph and not args.profile_one_step:
        try:
            step.enable_cuda_graph(dev_batches[0], warmup=2)
            cuda_graph = True
            run_steps(2, dev_batches, False)
        except Exception as ex:      # stay on eager launches, say so in the JSON line
            step._graph = None
            cuda_graph = f"failed: {type(ex).__name__}: {str(ex)[:200]}"
    if args.profile_one_step:
        run_steps(1, dev_batches, False)
        return

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _lib.reset_launch_count()
    t_dev, loss, out = run_steps(args.steps, dev_batches, False)
    launches = _lib.launch_count()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, step.opt)
    del out
    if cuda_graph is True:
        # under graph replay the host-side counter does not tick: count the launches of one eager step instead
        step_graph, step._graph = step._graph, None
        _lib.reset_launch_count()
        run_steps(1, dev_batches, False)
        launches = _lib.launch_count() * args.steps
        step._graph = step_graph
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / t_dev

    e2e = None
    if not args.no_e2e:
        run_steps(1, host_batches, True)
        t_e2e, _, _ = run_steps(args.steps, host_batches, True)
        e2e = {"value": world * B * args.steps / t_e2e, "unit": "images/sec", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": 4, "ms_per_step": t_e2e / args.steps * 1e3}

    micro, roof = None, None
    if rank == 0 and not args.no_micro:
        del dev_batches
        torch.cuda.empty_cache()
        micro = micro_rooflines(B, peaks, device)
        a = micro["attn_fwd_L0_self"]
        traffic, traffic_src = None, None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of the SHIPPED kernel from its ncu --set full capture
            with open(os.path.join(ROOT, "profiles", "r02_attn_fwd_ncu.json")) as f:
                tj = json.load(f)
            if B == tj.get("batch"):
                traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
        except Exception:
            pass
        roof = {"kernel": ("attention forward core (attn_fwd3_kernel: two S buffers per tile in TMEM, exp2 split 2/8 over MUFU/FMA; "
                           "level-0 self-attention, N=M=4096, 8x40, B=%d)" % B),
                "bound": "tensor", "achieved": a["tflops"], "peak": peaks["bf16_burst"], "unit": "TFLOP/s",
                "frac": a["tflops"] / peaks["bf16_burst"], "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_flops_per_launch": a["flops"],
                "algorithmic_bytes_per_launch": 4 * B * 4096 * 320 * 2,
                "peak_source": peaks["source"] + ", burst figure (kernel timed alone, L2 flushed between launches)",
                "aggregate_wo_attention": attention_aggregate(B, peaks, device)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            state = cpu_oracle_setup()
            cpu_oracle_step(state, 2, 1)                       # warm-up
            t_cpu, _ = cpu_oracle_step(state, 2, 2)
            cpu = {"value": 2.0 / t_cpu, "unit": "images/sec", "cores": torch.get_num_threads(), "kind": "port",
                   "sample": "ONE timed full pre-training step after one warm-up step at B=2 images (BASELINE configs[0] "
                             "batch; SD-v1.4 UNet x2 fwd + ViT-H/14 + CLIP-L text + bwd + AdamW), fp32 CPU oracle "
                             "(oracle/e4t_oracle.py), torch threads = min(host cores, 32)"}
            del state
        except Exception as ex:  # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": "images/sec", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"failed: {type(ex).__name__}: {ex}"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "SD-v1.4 E4T pretrain step (UNet enc-half + E4T encoder ViT-H/14 + CLIP text + "
                                       "full UNet + loss + bwd + AdamW), random-init, 512^2 (64x64 latents)",
                           "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
                           "trainable_params": n_train, "cuda_graph": cuda_graph,
                           "variant": ("domain tuning (configs[3]): all UNet weights trainable, grad clip" if args.tuning else
                                       "unfreeze_clip_vision" if args.unfreeze_clip_vision else "pretrain (configs[1])"),
                           "l2": "inputs rotate over 4 batches; per-step working set (activations ~30 GB) >> 126 MB L2",
                           "grad_allreduce": ("NCCL all-reduce of the flat fp32 grad arena: encoder-head slice issued from "
                                              "inside backward on a comm stream (overlaps the enc-half UNet backward), "
                                              + ("WeightOffsets gradients exchanged as the bank's 2 MB of G reductions inside "
                                                 "backward (the 573 MB slice is not all-reduced); "
                                                 if getattr(step, "_wo_factor_exchange", False) else "WeightOffsets slice after backward; ")
                                              + ("all inside the CUDA graph" if getattr(step, "_graph_has_opt", False)
                                                 else "eager after the compute-only graph")
                                              + ("; " + step._capture_note if getattr(step, "_capture_note", None) else ""))
                           if world > 1 else "none"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
                "gpu_launches_per_step": launches // max(args.steps, 1), "loss": loss, "roofline": roof, "kernels": micro,
                "cpu_baseline": cpu}
        print(json.dumps(line))
    if world > 1:
        sys.stdout.flush()
        dist.barrier()      # rank 0 may still be timing kernels for the roofline object; leave together
        # A CUDA graph that holds captured NCCL kernels keeps the communicator busy: destroying the process group while the
        # graph is alive hung the 2-GPU run at exit (r02 call 9: JSON line printed, then no exit).  Drop the graph first;
        # the timer is the backstop so that a teardown problem can never turn a finished measurement into a time-out.
        step.release_cuda_graph()
        torch.cuda.synchronize()
        import threading
        t = threading.Timer(60.0, lambda: os._exit(0))
        t.daemon = True
        t.start()
        dist.destroy_process_group()
        t.cancel()


if __name__ == "__main__":
    main()
