import sys, os, torch
sys.path[:0] = [os.getcwd(), os.path.join(os.getcwd(), "e4t-diffusion_b200"), os.path.join(os.getcwd(), "tests")]
from oracle import e4t_oracle as O
from oracle import vae_oracle as V
import test_vae_gpu as T
from e4t_b200 import engine
from e4t_b200.engine import PretrainStep
vae, _ = T._vae(V.TINY_VAE, 45)
batch = {k: v.cuda() for k, v in O.synth_batch(2, seed=42, latent_hw=16, image_hw=128).items()}
eps = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(7)).cuda()
x = batch["pixel_values"]
m = [vae.encode(x).latent_dist.mean.clone() for _ in range(3)]
print("encode repeat maxdiff", (m[0]-m[1]).abs().max().item(), (m[0]-m[2]).abs().max().item())
rec = {}
orig = engine.add_noise
def spy(l, n, t, a):
    rec.setdefault("lat", []).append(l.clone()); rec.setdefault("strides", []).append(l.stride())
    return orig(l, n, t, a)
engine.add_noise = spy
seen = {}
enc0 = vae.encode
def espy(x, *a, **k):
    o = enc0(x, *a, **k); seen["d"] = o.latent_dist; return o
vae.encode = espy
def run(b, v):
    unet, enc, text = T._step_models()
    st = PretrainStep(unet, enc, text, O.PLACEHOLDER_ID, class_token_id=320, lr=1e-3, weight_dtype=torch.float32, vae=v)
    out = st.forward_loss(b)
    l = out["loss"].item(); del st, out; torch.cuda.synchronize(); return l
wv = dict(batch, latent_eps=eps); del wv["latents"]
la = run(wv, vae)
L = rec["lat"][-1]; d = seen["d"]
R = ((d.mean + d.std * eps) * vae.config.scaling_factor)
print("vae loss", la, "strides", rec["strides"][-1], "recorded vs reconstructed", (L - R).abs().max().item())
lb = run(dict(batch, latents=L.clone()), None)
lc = run(dict(batch, latents=L.clone()), None)
ld = run(wv, vae)
print("pre(L)", lb, "pre(L) again", lc, "vae again", ld, "lat diff 2nd vae vs 1st", (rec["lat"][-1]-L).abs().max().item())
lp1 = run(batch, None); lp2 = run(batch, None)
print("synthetic latents twice", lp1, lp2)
