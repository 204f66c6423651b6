"""TEST-ONLY shim of the diffusers==0.14.0 symbols the reference imports (requirements.txt:1 of
mkshing/e4t-diffusion; diffusers itself is not installed and there is no network).

Used ONLY by oracle/gen_golden.py so that the reference's own e4t/models/*.py can be imported unchanged from
a checkout of the original project to generate the golden vectors under tests/golden/.  It restates, from the published
diffusers 0.14.0 behaviour, the five un-vendored pieces the UNet needs (ResnetBlock2D, Downsample2D,
Upsample2D, Timesteps, TimestepEmbedding) plus trivial stand-ins for the config/mixin plumbing.
parity unpinned at this boundary: diffusers is absent, so these restatements cannot be checked against it here.
"""
