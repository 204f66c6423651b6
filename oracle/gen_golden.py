"""Generate tests/golden/*.pt by running the REFERENCE's own modules (imported unchanged from a checkout of the original
e4t-diffusion project via oracle/shim) on seeded synthetic weights/inputs:

    E4T_REFERENCE=<checkout> python oracle/gen_golden.py    # writes tests/golden/{unet_tiny,unet_sd14,wo,inventory}.pt

The fixtures pin oracle/e4t_oracle.py (tests/test_oracle_cpu.py) and are the parity target of the CUDA path
(tests/test_e2e_gpu.py).  Everything is fp32 on CPU; weights come from e4t_oracle.synth_state_dict so the oracle and
the CUDA implementation can rebuild bit-identical parameters from the seed alone.
"""
import hashlib
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if not os.path.isdir(os.environ.get("E4T_REFERENCE", "")):
    raise SystemExit("set E4T_REFERENCE to a checkout of the original e4t-diffusion project")
sys.path[:0] = [os.environ["E4T_REFERENCE"], os.path.join(HERE, "shim"), ROOT]

from oracle import e4t_oracle as O  # noqa: E402
from oracle.golden import sample_grads, sample_rows  # noqa: E402

from e4t.models.unet_2d_condition import UNet2DConditionModel  # noqa: E402  (the reference's)
from e4t.weightoffsets import WeightOffsets  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
torch.manual_seed(0)
torch.set_num_threads(os.cpu_count())


def build_ref_unet(cfg, seed):
    m = UNet2DConditionModel(**O.ref_unet_kwargs(cfg))
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    mine = O.unet_param_shapes(cfg)
    assert shapes == mine, (set(shapes) ^ set(mine), [k for k in shapes if k in mine and shapes[k] != mine[k]][:5])
    sd = O.synth_state_dict(mine, seed)
    missing, unexpected = m.load_state_dict(sd, strict=True)
    return m, sd


def unet_case(cfg, B, seed, with_grads, hw):
    g = torch.Generator().manual_seed(seed + 17)
    m, sd = build_ref_unet(cfg, seed)
    x = torch.randn(B, 4, hw, hw, generator=g)
    t = torch.randint(0, 1000, (B,), generator=g)
    ehs = torch.randn(B, 77, cfg["cross_attention_dim"], generator=g).requires_grad_(with_grads)
    w = torch.randn(B, 4, hw, hw, generator=g)
    t0 = time.time()
    out = m(x, t, ehs).sample
    enc = m(x, t, ehs, return_encoder_outputs=True)["down_block_samples"]
    rec = dict(cfg=cfg, seed=seed, B=B, x=x, t=t, ehs=ehs.detach().clone(), w=w, out=out.detach().clone(),
               enc_pooled=torch.cat([e.mean(dim=(2, 3)) for e in enc], dim=-1).detach().clone(),
               enc_shapes=[tuple(e.shape) for e in enc])
    if with_grads:
        wenc = [torch.randn(e.shape, generator=g) for e in enc]
        loss = (out * w).sum() + sum((e * we).sum() for e, we in zip(enc, wenc))
        loss.backward()
        rec["wenc_seed_note"] = "wenc tensors are drawn from the same generator after x,t,ehs,w in enc order"
        rec["d_ehs"] = ehs.grad.clone()
        wo = {k: p.grad.clone() for k, p in m.named_parameters() if "wo" in k}
        # all the small WO grads verbatim; for the square matrices keep a 16x16 corner + Frobenius norm
        small = {}
        for k, gr in wo.items():
            if gr.numel() <= 4096:
                small[k] = gr
            else:
                small[k + "#corner"] = gr[:16, :16].clone()
                small[k + "#norm"] = gr.norm()
        rec["wo_grads"] = small
    print(f"  case B={B} hw={hw} boc={cfg['block_out_channels']} done in {time.time()-t0:.1f}s")
    return rec


def wo_case():
    rec = {}
    for R, C in [(32, 16), (320, 320), (768, 640)]:
        mod = WeightOffsets(R, C)
        sd = O.synth_state_dict({("p." + k): tuple(v.shape) for k, v in mod.state_dict().items()}, 3)
        mod.load_state_dict({k[2:]: v for k, v in sd.items()})
        rec[(R, C)] = sample_rows(mod().detach(), 1 if R * C <= 320 * 320 else 4)
    return rec


def main():
    os.makedirs(OUT, exist_ok=True)
    print("weight offsets"); torch.save(wo_case(), os.path.join(OUT, "wo.pt"))
    print("tiny unet"); torch.save(unet_case(O.TINY_UNET, 2, 1, True, 16), os.path.join(OUT, "unet_tiny.pt"))
    print("sd14 unet")
    rec = unet_case(O.SD14_UNET, 1, 2, True, 64)
    # below 1 MB: the tests re-draw `w` from the seed, and keep a fixed sample of the WeightOffsets gradients
    del rec["w"]
    rec["wo_grads"] = sample_grads(rec["wo_grads"], 16)
    torch.save(rec, os.path.join(OUT, "unet_sd14.pt"))
    m = UNet2DConditionModel(**O.ref_unet_kwargs(O.SD14_UNET))
    keys = sorted(m.state_dict().keys())
    n_base = sum(p.numel() for k, p in m.named_parameters() if "wo" not in k)
    n_wo = sum(p.numel() for k, p in m.named_parameters() if "wo" in k)
    inv = dict(sha256=hashlib.sha256("\n".join(f"{k}:{tuple(m.state_dict()[k].shape)}" for k in keys).encode()).hexdigest(),
               n_keys=len(keys), n_base=n_base, n_wo=n_wo,
               n_wo_tensors=sum(1 for k, _ in m.named_parameters() if "wo" in k))
    print(inv)
    torch.save(inv, os.path.join(OUT, "inventory.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
