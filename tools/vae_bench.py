"""AutoencoderKL on the B200: encode / decode throughput, the mid-block attention's share of encode time, the cost of
on-device encode inside the pre-training step, and a stock-torch comparator.  Prints ONE JSON line.

    python tools/vae_bench.py [--batch 16] [--out profiles/vae_bench.json]

Weights are synthetic (oracle.e4t_oracle.synth_state_dict) in the SD-v1.4 vae/config.json layout, cast to bf16 as
pretrain_e4t.py:423 does.  Times are CUDA-event windows of at least --min-window seconds after warm-up.  The working set
of every timed call (>= 1 GB of activations at B = 16) is far above the 126 MB L2.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "e4t-diffusion_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import e4t_oracle as O  # noqa: E402
from oracle import vae_oracle as V  # noqa: E402


def vae_flops(cfg, hw):
    """Multiply-add FLOPs (2 per MAC) of encode and decode of one hw x hw image, from the layer shapes."""
    boc, L, G = cfg["block_out_channels"], cfg["layers_per_block"], None
    conv = lambda cin, cout, k, s: 2.0 * cin * cout * k * k * s * s

    def res(cin, cout, s):
        return conv(cin, cout, 3, s) + conv(cout, cout, 3, s) + (conv(cin, cout, 1, s) if cin != cout else 0.0)

    def mid(c, s):
        n = s * s
        return 2 * res(c, c, s) + 4 * 2.0 * n * c * c + 2 * 2.0 * n * n * c   # q,k,v,proj + QKᵀ, PV

    enc, s, c = conv(3, boc[0], 3, hw), hw, boc[0]
    for i, co in enumerate(boc):
        for j in range(L):
            enc += res(c if j == 0 else co, co, s)
        c = co
        if i < len(boc) - 1:
            s //= 2
            enc += conv(co, co, 3, s)
    enc += mid(c, s) + conv(c, 8, 3, s) + 2.0 * 8 * 8 * s * s
    lat = s
    dec = 2.0 * 4 * 4 * s * s + conv(4, boc[-1], 3, s) + mid(boc[-1], s)
    c = boc[-1]
    for i, co in enumerate(reversed(boc)):
        for j in range(L + 1):
            dec += res(c if j == 0 else co, co, s)
        c = co
        if i < len(boc) - 1:
            s *= 2
            dec += conv(co, co, 3, s)
    dec += conv(boc[0], 3, 3, s)
    return enc, dec, lat


def timed(fn, min_window, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n, t = 1, 0.0
    while True:
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) * 1e-3
        if t >= min_window:
            return t / n
        n = max(n * 2, int(n * min_window / max(t, 1e-6)) + 1)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power, clk = [s.strip() for s in r.stdout.strip().split(",")]
        return dict(gpu=name, power_limit=power, sm_max_clock=clk)
    except Exception as ex:   # noqa: BLE001
        return dict(gpu=torch.cuda.get_device_name(0), power_limit=f"unavailable ({type(ex).__name__})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--min-window", type=float, default=1.0)
    ap.add_argument("--skip-step", action="store_true", help="leave out the PretrainStep comparison")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/vae_bench.py measures on a CUDA device"
    from e4t.models.autoencoder_kl import AutoencoderKL
    from e4t_b200 import _lib
    _lib.load()
    dev = torch.device("cuda", 0)
    B, cfg = args.batch, V.SD14_VAE
    f_enc, f_dec, lat = vae_flops(cfg, 512)
    res = dict(metric="vae_sd14", batch=B, image=512, latent=lat, tflop_per_image=dict(encode=f_enc * 1e-12,
                                                                                     decode=f_dec * 1e-12))
    res.update(gpu_info())
    sd = O.synth_state_dict(V.vae_param_shapes(cfg), 0)
    vae = AutoencoderKL(**cfg)
    vae.load_state_dict(sd, strict=True)
    vae = vae.to(dev, dtype=torch.bfloat16)
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(B, 3, 512, 512, generator=g, device=dev) * 2 - 1
    z = torch.randn(B, 4, lat, lat, generator=g, device=dev)

    t_enc = timed(lambda: vae.encode(x), args.min_window)
    t_dec = timed(lambda: vae.decode(z), args.min_window)
    attn = vae.encoder.mid_block.attentions[0]
    h = torch.randn(B, lat, lat, cfg["block_out_channels"][-1], generator=g, device=dev).to(torch.bfloat16)
    with torch.no_grad():
        t_attn = timed(lambda: attn(h), args.min_window)
    res["ours"] = dict(encode_ms=t_enc * 1e3, decode_ms=t_dec * 1e3, encode_img_s=B / t_enc, decode_img_s=B / t_dec,
                       encode_tflops=B * f_enc / t_enc * 1e-12, decode_tflops=B * f_dec / t_dec * 1e-12,
                       attn_block_ms=t_attn * 1e3, attn_share_of_encode=t_attn / t_enc)

    # stock torch: the oracle on CUDA under bf16 autocast (cuDNN convolutions, SDPA attention)
    sd_dev = {k: v.to(dev) for k, v in sd.items()}
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        s_enc = timed(lambda: V.vae_encode(sd_dev, cfg, x), args.min_window)
        s_dec = timed(lambda: V.vae_decode(sd_dev, cfg, z), args.min_window)
    res["stock_torch_bf16_autocast"] = dict(encode_ms=s_enc * 1e3, decode_ms=s_dec * 1e3, encode_img_s=B / s_enc,
                                            decode_img_s=B / s_dec)
    del sd_dev
    torch.cuda.empty_cache()

    if not args.skip_step:
        import bench
        from e4t_b200.engine import PretrainStep
        unet, enc, text = bench.build_models(dev)
        step = PretrainStep(unet, enc, text, placeholder_token_id=49408, class_token_id=320, lr=1.6e-5,
                            weight_dtype=torch.bfloat16, vae=vae)
        hb = bench.host_batch(B, 42, pinned=False)
        with_lat = {k: v.to(dev) for k, v in hb.items()}
        with_enc = dict(with_lat, latent_eps=torch.randn(B, 4, lat, lat, generator=g, device=dev))
        del with_enc["latents"]
        ms = {}
        for name, b in (("latents_given", with_lat), ("vae_encode_on_device", with_enc)):
            step(b)
            step.enable_cuda_graph(b, warmup=2)
            ms[name] = timed(lambda: step(b), args.min_window) * 1e3
            step.release_cuda_graph()
        res["pretrain_step_ms"] = dict(ms, configs="BASELINE configs[1]: SD-v1.4 + ViT-H/14, 512², bs 16, bf16, "
                                                    "whole-step CUDA graph",
                                       encode_cost_ms=ms["vae_encode_on_device"] - ms["latents_given"])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
