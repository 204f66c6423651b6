"""Edges of the GEMM / convolution engine and of the VAE's kernels, each against a plain fp64 torch computation on the
same bf16-representable inputs.

Pass criteria follow from the output format:
  - fp32 outputs: relative RMS error <= 2e-3 (1e-4 for conv_out_fwd and pointwise_nchw, which accumulate in fp32 from
    exact products);
  - bf16 outputs: EVERY element within 2^-8 |ref| + 2e-3 rms(ref).  A wrong tail tile, row group or row segment is a
    local error that a whole-tensor RMS would dilute.
Combinations are a seeded sample of each cross product, not all of it.  The worst error of each kernel family (as a
fraction of its bound) is printed at the end of the module (pytest -s).
"""
import itertools
import random

import pytest
import torch
import torch.nn.functional as F

from oracle import vae_oracle as V

pytestmark = pytest.mark.gpu
torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.allow_tf32 = False
BF16, F32, F64 = torch.bfloat16, torch.float32, torch.float64

_WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(_WORST):
        print(f"[edges] {k:<16} worst error / bound {_WORST[k]:.3f}")


def _note(family, frac):
    _WORST[family] = max(_WORST.get(family, 0.0), frac)


def check_bf16(out, ref, family, extra=None):
    """Every element: |out - ref| <= 2^-8 |ref| + 2e-3 rms(ref) (+ extra, a per-element allowance)."""
    assert out.dtype == BF16 and out.shape == ref.shape, (out.dtype, out.shape, ref.shape)
    out, ref = out.double(), ref.double()
    assert torch.isfinite(out).all(), f"{family}: non-finite output"
    bound = 2.0 ** -8 * ref.abs() + 2e-3 * ref.pow(2).mean().sqrt()
    if extra is not None:
        bound = bound + extra
    frac = ((out - ref).abs() / bound.clamp_min(1e-30)).max().item()
    _note(family, frac)
    if frac > 1:
        bad = ((out - ref).abs() > bound).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{family}: {len(bad)} of {ref.numel()} elements out of bound; first at {i}: "
                             f"out {out[i].item():.6g} ref {ref[i].item():.6g} (worst {frac:.2f}x the bound)")


def check_f32(out, ref, family, tol=2e-3):
    assert out.dtype == F32 and out.shape == ref.shape, (out.dtype, out.shape, ref.shape)
    out, ref = out.double(), ref.double()
    assert torch.isfinite(out).all(), f"{family}: non-finite output"
    rel = ((out - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt().clamp_min(1e-30)).item()
    _note(family, rel / tol)
    assert rel <= tol, f"{family}: relative RMS error {rel:.3e} > {tol}"


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _mk(shape, g, scale=1.0):
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(BF16)


def _f32(shape, g, scale=1.0):
    return torch.randn(shape, generator=g, device="cuda") * scale


def _padded(t, inner):
    """The same values in a buffer whose row stride is `inner` (>= t.shape[-1]): a column slice of a wider buffer."""
    buf = torch.zeros(t.shape[:-1] + (inner,), device=t.device, dtype=t.dtype)
    buf[..., :t.shape[-1]] = t
    return buf[..., :t.shape[-1]]


def _r8(n):
    return (n + 7) // 8 * 8


def _sample(items, k, seed):
    items = list(items)
    return random.Random(seed).sample(items, min(k, len(items)))


# =====================================================================================================================
# GEMM engine
# =====================================================================================================================
def _operands(M, N, K, a_mn, b_mn, g, batch=None):
    """Logical A (.., M, K), B (.., N, K) and their stored forms (MN-major rows padded to a multiple of 8)."""
    lead = () if batch is None else (batch,)
    A = _mk(lead + (M, K), g, K ** -0.25)
    B = _mk(lead + (N, K), g, K ** -0.25)
    As = _padded(A.transpose(-1, -2), _r8(M)) if a_mn else A
    Bs = _padded(B.transpose(-1, -2), _r8(N)) if b_mn else B
    return A, B, As, Bs


def _ref(A, B, alpha=1.0, bias=None, rg=None, rpg=1, res=None, base=None):
    r = alpha * (A.double() @ B.double().transpose(-1, -2))
    M = r.shape[-2]
    if bias is not None:
        r = r + bias.double()
    if rg is not None:
        r = r + rg.double().repeat_interleave(rpg, 0)[:M]
    if res is not None:
        r = r + res.double()
    if base is not None:
        r = r + base.double()
    return r


def _out_buf(M, N, dtype, kind):
    """'plain' contiguous; 'ldo' a column slice with a row stride that is not a multiple of 16 bytes; 'off1' an output
    whose pointer is one element past a 16-byte boundary."""
    if kind == "plain":
        return torch.empty((M, N), device="cuda", dtype=dtype)
    if kind == "ldo":
        return torch.empty((M, N + 3), device="cuda", dtype=dtype)[:, :N]
    if kind == "off1":
        return torch.empty(M * N + 1, device="cuda", dtype=dtype)[1:].view(M, N)
    raise ValueError(kind)


# every epilogue path x every addend: (name, N, out dtype, output kind, alpha, bias, rows_per_group, residual kind)
_EPI = [
    # lean TMA-store loop (bf16, N % 8 == 0, alpha 1, no row group)
    ("lean", 320, BF16, "plain", 1.0, False, 0, None),
    ("lean+bias", 320, BF16, "plain", 1.0, True, 0, None),
    ("lean+res", 320, BF16, "plain", 1.0, False, 0, "plain"),
    ("lean+bias+res", 320, BF16, "plain", 1.0, True, 0, "plain"),
    # general TMA-store loop
    ("general alpha", 320, BF16, "plain", 0.37, False, 0, None),
    ("general rg1", 320, BF16, "plain", 1.0, False, 1, None),
    ("general rg77", 320, BF16, "plain", 1.0, False, 77, None),
    ("general rg128", 320, BF16, "plain", 1.0, False, 128, None),
    ("general rg4096", 320, BF16, "plain", 1.0, False, 4096, None),
    ("general all", 320, BF16, "plain", -1.5, True, 77, "plain"),
    # a residual the TMA-store loops cannot read by 16 bytes (unaligned column slice) -> per-thread loop
    ("res unaligned", 320, BF16, "plain", 1.0, True, 0, "slice"),
    # bf16 per-thread loop
    ("bf16 N77", 77, BF16, "plain", 1.0, False, 0, None),
    ("bf16 N77 all", 77, BF16, "plain", 0.5, True, 77, "plain"),
    ("bf16 ldo", 320, BF16, "ldo", 1.0, True, 0, "plain"),
    ("bf16 ldo all", 264, BF16, "ldo", 2.0, True, 128, "slice"),
    ("bf16 off1", 320, BF16, "off1", 1.0, False, 0, None),
    ("bf16 off1 all", 320, BF16, "off1", 0.5, True, 1, "plain"),
    # fp32 store
    ("f32 N77", 77, F32, "plain", 1.0, True, 0, None),
    ("f32 N77 ldo", 77, F32, "ldo", 0.5, True, 77, "slice"),
    ("f32 N320", 320, F32, "plain", 1.0, True, 128, "plain"),
    ("f32 N320 ldo", 320, F32, "ldo", 1.0, False, 0, "plain"),
    ("f32 off1", 320, F32, "off1", 1.0, True, 0, None),
]


@pytest.mark.parametrize("i", range(len(_EPI)), ids=[c[0] for c in _EPI])
def test_gemm_epilogue_paths(i):
    from e4t_b200 import ops
    name, N, dt, kind, alpha, has_bias, rpg, res_kind = _EPI[i]
    M, K = 300, 200
    g = _gen(100 + i)
    A, B, _, _ = _operands(M, N, K, False, False, g)
    bias = _f32((N,), g) if has_bias else None
    rg = _f32((-(-M // rpg), N), g) if rpg else None
    res = None
    if res_kind == "plain":
        res = _mk((M, N), g)
    elif res_kind == "slice":     # pointer 2 bytes past 16-byte alignment, row stride N + 5
        res = _padded(_mk((M, N + 1), g), N + 5)[:, 1:]
    out = _out_buf(M, N, dt, kind)
    ops.gemm(A, B, out=out, bias=bias, rowgroup=rg, rows_per_group=max(rpg, 1), residual=res, alpha=alpha)
    ref = _ref(A, B, alpha, bias, rg, max(rpg, 1), res)
    (check_bf16 if dt == BF16 else check_f32)(out, ref, "gemm epilogue")


@pytest.mark.parametrize("splits", [1, 3, 0, "kchunks"])
@pytest.mark.parametrize("N,ldo", [(77, 77), (320, 323)])
def test_gemm_atomic_accumulate(splits, N, ldo):
    from e4t_b200 import ops
    M, K = 257, 1232
    g = _gen(N + ldo)
    for a_mn, b_mn in ((True, True), (False, False)):
        A, B, As, Bs = _operands(M, N, K, a_mn, b_mn, g)
        base = _f32((M, N), g)
        out = _padded(base.clone(), ldo)
        sp = -(-K // 64) if splits == "kchunks" else splits
        addends = {}
        if sp == 1:       # addends are taken only without split-K (each split would add them again)
            addends = dict(bias=_f32((N,), g), residual=_mk((M, N), g))
        ops.gemm(As, Bs, a_mn=a_mn, b_mn=b_mn, out=out, accumulate=True, splits=sp, **addends)
        ref = _ref(A, B, bias=addends.get("bias"), res=addends.get("residual"), base=base)
        check_f32(out, ref, "gemm atomic")


_TAILS = _sample(itertools.product([1, 127, 129, 300], [8, 40, 77, 264, 1000], [8, 56, 64, 72, 1232],
                                   [(False, False), (False, True), (True, False), (True, True)]), 28, 1)


@pytest.mark.parametrize("M,N,K,majors", _TAILS)
def test_gemm_ragged_tails(M, N, K, majors):
    from e4t_b200 import ops
    a_mn, b_mn = majors
    g = _gen(M * 131 + N * 7 + K)
    A, B, As, Bs = _operands(M, N, K, a_mn, b_mn, g)
    ref = _ref(A, B)
    check_bf16(ops.gemm(As, Bs, a_mn=a_mn, b_mn=b_mn), ref, "gemm tails")
    check_f32(ops.gemm(As, Bs, a_mn=a_mn, b_mn=b_mn, out_dtype=F32), ref, "gemm tails")


_BNS = [(False, bn) for bn in range(32, 257, 32)] + [(True, bn) for bn in (64, 128, 192, 256)]


@pytest.mark.parametrize("b_mn,bn", _BNS)
def test_gemm_every_tile_width(b_mn, bn):
    """N = 1000 leaves the last N tile partial at every width."""
    from e4t_b200 import ops
    M, N, K = 300, 1000, 200
    g = _gen(bn + 1000 * b_mn)
    A, B, As, Bs = _operands(M, N, K, False, b_mn, g)
    bias = _f32((N,), g)
    res = _mk((M, N), g)
    rg = _f32((3, N), g)
    out = ops.gemm(As, Bs, b_mn=b_mn, bias=bias, residual=res, force_bn=bn)
    check_bf16(out, _ref(A, B, bias=bias, res=res), "gemm tile width")
    out = ops.gemm(As, Bs, b_mn=b_mn, rowgroup=rg, rows_per_group=128, alpha=0.5, force_bn=bn)
    check_bf16(out, _ref(A, B, 0.5, rg=rg, rpg=128), "gemm tile width")
    out = ops.gemm(As, Bs, b_mn=b_mn, bias=bias, out_dtype=F32, force_bn=bn)
    check_f32(out, _ref(A, B, bias=bias), "gemm tile width")


def test_gemm_batching():
    from e4t_b200 import ops
    g = _gen(77)
    Bt, M, N, K = 3, 300, 264, 200
    A, B, _, _ = _operands(M, N, K, False, False, g, batch=Bt)
    ref = _ref(A, B)
    check_bf16(ops.gemm(A, B), ref, "gemm batched")
    check_f32(ops.gemm(A, B, out_dtype=F32), ref, "gemm batched")
    # a shared 2-D operand on either side
    check_bf16(ops.gemm(A[1], B), _ref(A[1].expand(Bt, M, K), B), "gemm batched")
    check_bf16(ops.gemm(A, B[2]), _ref(A, B[2].expand(Bt, N, K)), "gemm batched")
    # MN-major batched operands
    Am = _padded(A.transpose(1, 2), _r8(M))
    Bm = _padded(B.transpose(1, 2), _r8(N))
    check_bf16(ops.gemm(Am, Bm, a_mn=True, b_mn=True), ref, "gemm batched")
    # batched residual and bias
    res = _mk((Bt, M, N), g)
    bias = _f32((N,), g)
    check_bf16(ops.gemm(A, B, bias=bias, residual=res), _ref(A, B, bias=bias, res=res), "gemm batched")
    check_bf16(ops.gemm(A, B, residual=res, alpha=0.25), _ref(A, B, 0.25, res=res), "gemm batched")
    # batched output that is a slice of a larger buffer (out_bstride != M * ldo): TMA-store and per-thread loops
    for rows, cols, dt in ((M + 8, N + 8, BF16), (M + 5, N + 3, BF16), (M + 1, N + 1, F32)):
        buf = torch.full((Bt, rows, cols), 7.0, device="cuda", dtype=dt)
        out = buf[:, :M, :N]
        ops.gemm(A, B, out=out, bias=bias, residual=res)
        (check_bf16 if dt == BF16 else check_f32)(out, _ref(A, B, bias=bias, res=res), "gemm batched")
        assert (buf[:, M:, :] == 7).all() and (buf[:, :, N:] == 7).all(), "wrote outside the output slice"
    # rows aligned (ldo = N) but a batch stride that is not a multiple of 16 bytes
    for dt in (BF16, F32):
        flat = torch.full((Bt * (M * N + 4),), 7.0, device="cuda", dtype=dt)
        out = flat.as_strided((Bt, M, N), (M * N + 4, N, 1))
        ops.gemm(A, B, out=out, bias=bias, residual=res)
        (check_bf16 if dt == BF16 else check_f32)(out, _ref(A, B, bias=bias, res=res), "gemm batched")
        assert (flat.view(Bt, -1)[:, M * N:] == 7).all(), "wrote outside the output"


def test_gemm_qkv_column_slices():
    """The VAE mid-block attention: q, k, v are column slices of one (B, T, 3C) projection (lda = 3C)."""
    from e4t_b200 import ops
    g = _gen(512)
    Bt, T, C = 2, 1024, 512
    qkv = _mk((Bt, T, 3 * C), g)
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    s = ops.gemm(q, k, out_dtype=F32, alpha=C ** -0.5)
    s_ref = C ** -0.5 * (q.double() @ k.double().transpose(1, 2))
    check_f32(s, s_ref, "gemm qkv")
    p = _mk((Bt, T, T), g, 0.03)
    o = ops.gemm(p, v, b_mn=True)
    check_bf16(o, p.double() @ v.double(), "gemm qkv")


def test_gemm_refusals():
    """Inputs the ABI refuses raise E4TError from the host-side check and launch nothing."""
    from e4t_b200 import _lib, ops
    from e4t_b200._lib import E4TError, c_float, c_int, c_ll, ptr, stream
    g = _gen(3)
    M, N, K = 256, 320, 128
    A, B = _mk((M, K), g), _mk((N, K), g)
    bias = _f32((N + 1,), g)
    rg = _f32((2 * N + 1,), g)

    def call(A, B, out, lda, ldb, *, bias=None, rg=None, res=None, mode=0, splits=1, force_bn=0, b_mn=0):
        _lib.call("e4t_gemm_bf16", ptr(A), ptr(B), ptr(out), c_int(M), c_int(N), c_int(K), c_int(1), c_int(0),
                  c_int(b_mn), c_ll(lda), c_ll(ldb), c_ll(0), c_ll(0), c_int(mode), c_ll(N), c_ll(0), ptr(bias),
                  ptr(rg), c_int(128), ptr(res), c_ll(N), c_ll(0), c_float(1.0), c_int(splits), c_int(force_bn),
                  stream())

    out = torch.full((M, N), 3.0, device="cuda", dtype=BF16)
    out32 = torch.full((M, N), 3.0, device="cuda", dtype=F32)
    A132 = _padded(A, K + 4)                   # lda = 132: not a multiple of 8
    # lda fine, pointer 2 bytes past 16-byte alignment
    Aoff = torch.zeros(M * (K + 8) + 1, device="cuda", dtype=BF16)[1:].view(M, K + 8)
    Boff = torch.zeros(N * (K + 8) + 1, device="cuda", dtype=BF16)[1:].view(N, K + 8)
    refused = [
        ("lda % 8", lambda: call(A132, B, out, K + 4, K)),
        ("ldb % 8", lambda: call(A, _padded(B, K + 4), out, K, K + 4)),
        ("misaligned A", lambda: call(Aoff, B, out, K + 8, K)),
        ("misaligned B", lambda: call(A, Boff, out, K, K + 8)),
        ("misaligned bias", lambda: call(A, B, out, K, K, bias=bias[1:])),
        ("misaligned rowgroup", lambda: call(A, B, out, K, K, rg=rg[1:])),
        ("split-K with bias", lambda: call(A, B, out32, K, K, bias=bias[:N], mode=2, splits=2)),
        ("split-K without atomics", lambda: call(A, B, out32, K, K, mode=1, splits=2)),
        ("force_bn 48", lambda: call(A, B, out, K, K, force_bn=48)),
        ("force_bn 288", lambda: call(A, B, out, K, K, force_bn=288)),
        ("force_bn 96, MN-major B", lambda: call(A, B.t().contiguous(), out, K, N, force_bn=96, b_mn=1)),
    ]
    torch.cuda.synchronize()
    for what, fn in refused:
        _lib.reset_launch_count()
        with pytest.raises(E4TError):
            fn()
        assert _lib.launch_count() == 0, what
    torch.cuda.synchronize()
    assert (out == 3).all() and (out32 == 3).all()
    # the Python wrapper raises the same error
    with pytest.raises(E4TError):
        ops.gemm(A, B, bias=bias[1:])


# =====================================================================================================================
# Convolution
# =====================================================================================================================
def _w9(w):
    return w.permute(2, 3, 0, 1).reshape(9, w.shape[0], w.shape[1]).contiguous()


def _conv_ref(x, w, bias=None, stride=1, pad=1):
    """fp64 3x3 convolution of NHWC x with w (Cout, Cin, 3, 3) -> NHWC; pad 0 is F.pad(x, (0,1,0,1)) then stride 2.
    im2col + one fp64 matrix product per image."""
    xn = x.permute(0, 3, 1, 2).double()
    if pad == 0:
        xn = F.pad(xn, (0, 1, 0, 1))
    B, _, Hin, Win = xn.shape
    Ho = (Hin + 2 * pad - 3) // stride + 1
    Wo = (Win + 2 * pad - 3) // stride + 1
    wm = w.double().reshape(w.shape[0], -1)
    outs = []
    for b in range(B):
        cols = F.unfold(xn[b:b + 1], 3, padding=pad, stride=stride)[0]     # (Cin*9, L)
        o = wm @ cols
        outs.append(o.t().reshape(Ho, Wo, -1))
    out = torch.stack(outs)
    if bias is not None:
        out = out + bias.double()
    return out


# (H, W) = OUTPUT size per tiling: several images per tile, several rows per tile, one row segment per tile
_TILINGS = ([("images", h, h, b) for h in (2, 4, 8) for b in (1, 3, 5)]
            + [("rows", 128 // w * k, w, b) for w in (16, 32, 64) for k, b in ((1, 1), (2, 2), (3, 1))]
            + [("segment", h, w, 1) for w in (128, 256, 384, 512) for h in (1, 3, 5)])
_SP = [(1, 1), (2, 1), (2, 0)]
_CIN = [64, 192, 512]
_COUT = [32, 96, 128, 200, 512, 3, 77]
_BN = [0, 32, 64, 96, 128, 160, 224, 256]


def _conv_cases():
    """Two cases per tiling, the (stride, pad) pairs in turn; Cin, Cout and force_bn (0 = heuristic, often a width
    that does not divide Cout) drawn from a seeded generator."""
    rnd = random.Random(11)
    cases = []
    for i, t in enumerate(_TILINGS):
        for j in range(2):
            cases.append((t, _SP[(2 * i + j) % 3], rnd.choice(_CIN), rnd.choice(_COUT), rnd.choice(_BN)))
    return cases


@pytest.mark.parametrize("tiling,sp,cin,cout,bn", _conv_cases())
def test_conv3x3_tilings(tiling, sp, cin, cout, bn):
    from e4t_b200 import ops
    kind, H, W, B = tiling
    stride, pad = sp
    g = _gen(H * 1000 + W * 10 + cin + cout + bn)
    x = _mk((B, H * stride, W * stride, cin), g)
    w = _mk((cout, cin, 3, 3), g, (9 * cin) ** -0.5)
    bias = _f32((cout,), g)
    res = _mk((B, H, W, cout), g)
    ref = _conv_ref(x, w, bias, stride, pad)
    out = ops.conv3x3_ex(x, _w9(w), stride=stride, pad=pad, bias=bias, residual=res, force_bn=bn)
    check_bf16(out, ref + res.double(), f"conv {kind}")
    if stride == 1:
        out = ops.conv3x3_ex(x, _w9(w), bias=bias, force_bn=bn)
        check_bf16(out, ref, f"conv {kind}")
        rg = _f32((B, cout), g)
        ref_rg = ref + rg.double()[:, None, None, :] + res.double()
        check_bf16(ops.conv3x3(x, _w9(w), bias=bias, rowgroup=rg, residual=res, force_bn=bn), ref_rg, f"conv {kind}")
        check_f32(ops.conv3x3(x, _w9(w), bias=bias, rowgroup=rg, residual=res, out_dtype=F32, force_bn=bn), ref_rg,
                  f"conv {kind}")


def test_conv3x3_refusals():
    from e4t_b200 import _lib, ops
    from e4t_b200._lib import E4TError
    g = _gen(4)
    x, w = _mk((1, 16, 16, 64), g), _mk((9, 64, 64), g)
    refused = [
        ("Cin % 64", lambda: ops.conv3x3(_mk((1, 16, 16, 32), g), _mk((9, 64, 32), g))),
        ("width 96", lambda: ops.conv3x3(_mk((1, 4, 96, 64), g), w)),
        ("pad 0, stride 1", lambda: ops.conv3x3_ex(x, w, stride=1, pad=0)),
        ("odd input, stride 2", lambda: ops.conv3x3_ex(_mk((1, 15, 16, 64), g), w, stride=2)),
        ("force_bn 48", lambda: ops.conv3x3(x, w, force_bn=48)),
        ("force_bn 288", lambda: ops.conv3x3(x, w, force_bn=288)),
        ("misaligned bias", lambda: ops.conv3x3(x, w, bias=_f32((65,), g)[1:])),
    ]
    torch.cuda.synchronize()
    for what, fn in refused:
        _lib.reset_launch_count()
        with pytest.raises(E4TError):
            fn()
        assert _lib.launch_count() == 0, what


def _sd14_convs():
    """(Cin, Cout, H_in, W_in, stride, pad, residual) of every 3x3 convolution on the GEMM engine that the SD-v1.4 VAE
    runs to encode a 512^2 image and decode a 64^2 latent."""
    cfg = V.SD14_VAE
    boc, L = cfg["block_out_channels"], cfg["layers_per_block"]
    hw = cfg["sample_size"]
    sig = set()

    def resnet(cin, cout, s):
        sig.add((cin, cout, s, s, 1, 1, False))      # conv1
        sig.add((cout, cout, s, s, 1, 1, True))      # conv2 (+ shortcut / input as residual)

    s, c = hw, boc[0]
    for i, co in enumerate(boc):
        for j in range(L):
            resnet(c if j == 0 else co, co, s)
        c = co
        if i < len(boc) - 1:
            sig.add((co, co, s, s, 2, 0, False))
            s //= 2
    resnet(c, c, s)                                  # mid block (encoder)
    rev = list(reversed(boc))
    s, c = hw // 8, rev[0]
    resnet(c, c, s)                                  # mid block (decoder)
    for i, co in enumerate(rev):
        for j in range(L + 1):
            resnet(c if j == 0 else co, co, s)
        c = co
        if i < len(rev) - 1:
            s *= 2
            sig.add((co, co, s, s, 1, 1, False))    # upsampler conv after nearest x2
    return sorted(sig)


@pytest.mark.parametrize("cin,cout,H,W,stride,pad,has_res", _sd14_convs())
def test_conv3x3_sd14_vae_sizes(cin, cout, H, W, stride, pad, has_res):
    from e4t_b200 import ops
    g = _gen(cin + cout + H + stride)
    x = _mk((1, H, W, cin), g)
    w = _mk((cout, cin, 3, 3), g, (9 * cin) ** -0.5)
    bias = _f32((cout,), g, 0.1)
    res = _mk((1, H // stride, W // stride, cout), g) if has_res else None
    ref = _conv_ref(x, w, bias, stride, pad)
    if res is not None:
        ref = ref + res.double()
    if stride == 1:
        out = ops.conv3x3(x, _w9(w), bias=bias, residual=res)
    else:
        out = ops.conv3x3_ex(x, _w9(w), stride=stride, pad=pad, bias=bias)
    check_bf16(out, ref, "conv sd14 vae")


# =====================================================================================================================
# The VAE's small kernels
# =====================================================================================================================
@pytest.mark.parametrize("cin,cout,H,W", [(3, 128, 512, 512), (4, 512, 64, 64), (3, 64, 8, 8), (16, 40, 8, 24)])
def test_conv_in_fwd(cin, cout, H, W):
    from e4t_b200 import ops
    g = _gen(cin * cout + H)
    x = _f32((2, cin, H, W), g)
    w = _f32((cout, cin, 3, 3), g, (9 * cin) ** -0.5)
    bias = _f32((cout,), g, 0.1)
    ref = F.conv2d(x.double(), w.double(), bias.double(), padding=1).permute(0, 2, 3, 1)
    check_bf16(ops.conv_in_fwd(x, w, bias), ref, "conv_in_fwd")


@pytest.mark.parametrize("C,cout,H,W", [(512, 8, 64, 64), (128, 3, 512, 512), (64, 1, 8, 8)])
def test_conv_out_fwd(C, cout, H, W):
    from e4t_b200 import ops
    g = _gen(C * cout + H)
    x = _mk((2, H, W, C), g)
    w = _f32((cout, C, 3, 3), g, (9 * C) ** -0.5)
    bias = _f32((cout,), g, 0.1)
    ref = F.conv2d(x.permute(0, 3, 1, 2).double(), w.double(), bias.double(), padding=1)
    check_f32(ops.conv_out_fwd(x, w, bias), ref, "conv_out_fwd", tol=1e-4)


@pytest.mark.parametrize("HW", [1, 4096, 4097])
@pytest.mark.parametrize("cin,cout", [(4, 4), (8, 8), (1, 3)])
@pytest.mark.parametrize("with_bias", [False, True])
def test_pointwise_nchw(HW, cin, cout, with_bias):
    from e4t_b200 import ops
    g = _gen(HW + cin * 10 + cout)
    x = _f32((2, cin, 1, HW), g)
    w = _f32((cout, cin), g)
    bias = _f32((cout,), g) if with_bias else None
    ref = torch.einsum("oc,bchw->bohw", w.double(), x.double())
    if bias is not None:
        ref = ref + bias.double()[None, :, None, None]
    check_f32(ops.pointwise_nchw(x, w, bias), ref, "pointwise_nchw", tol=1e-4)


def _scores(rows, M, kind, g):
    s = torch.randn(rows, M, generator=g, device="cuda")
    if kind == "gauss30":
        s = s * 30
    elif kind == "peak":
        idx = torch.randint(0, M, (rows,), generator=g, device="cuda")
        s[torch.arange(rows, device="cuda"), idx] += 1e4
    elif kind == "equal":
        s = torch.full((rows, M), 0.75, device="cuda")
    elif kind == "neginf":
        # some (not all) entries masked: at random, plus the whole first half of odd rows (so that entire threads see
        # only -inf before their first finite value)
        s = s * 4
        mask = torch.rand(rows, M, generator=g, device="cuda") < 0.5
        mask[1::2, :M // 2] = True
        mask[:, -1] = False
        s[mask] = float("-inf")
    return s


_SOFTMAX = _sample([(r, m, k) for r in (1, 3, 4096) for m in (4, 8, 100, 1028, 4096, 16384, 65536)
                    for k in ("gauss1", "gauss30", "peak", "equal", "neginf") if r * m <= 1 << 26], 40, 5)
# the masked pattern at every length
_SOFTMAX += [(3, m, "neginf") for m in (4, 8, 100, 1028, 4096, 16384, 65536) if (3, m, "neginf") not in _SOFTMAX]


@pytest.mark.parametrize("rows,M,kind", _SOFTMAX)
def test_softmax_rows(rows, M, kind):
    from e4t_b200 import ops
    g = _gen(rows + M)
    s = _scores(rows, M, kind, g)
    p = ops.softmax_rows(s)
    check_bf16(p, torch.softmax(s.double(), -1), "softmax_rows")


@pytest.mark.parametrize("rows,M,pad", [(3, 100, 4), (5, 1028, 60), (64, 4096, 8), (2, 16384, 4)])
def test_softmax_rows_strided(rows, M, pad):
    """ld > M through the C-ABI: P's pad columns keep their sentinel."""
    from e4t_b200 import _lib
    from e4t_b200._lib import c_int, c_ll, ptr, stream
    g = _gen(M + pad)
    ld = M + pad
    S = torch.full((rows, ld), 1e4, device="cuda")
    S[:, :M] = _scores(rows, M, "gauss30", g)
    P = torch.full((rows, ld), -7.0, device="cuda", dtype=BF16)
    _lib.call("e4t_softmax_rows", ptr(S), ptr(P), c_ll(rows), c_int(M), c_ll(ld), stream())
    check_bf16(P[:, :M], torch.softmax(S[:, :M].double(), -1), "softmax_rows")
    assert (P[:, M:] == -7.0).all(), "softmax_rows wrote into the pad columns"


# =====================================================================================================================
# GroupNorm
# =====================================================================================================================
def _gn_input(B, HW, C, G, ratio, g):
    """Groups with offsets of either sign at |mean| / std = ratio, std varying across groups."""
    std = torch.exp(torch.rand(B, G, generator=g, device="cuda") * 2 - 1)
    sign = torch.where(torch.rand(B, G, generator=g, device="cuda") < 0.5, -1.0, 1.0)
    off = sign * ratio * std
    cpg = C // G
    x = torch.randn(B, HW, C, generator=g, device="cuda")
    x = x * std.repeat_interleave(cpg, 1)[:, None, :] + off.repeat_interleave(cpg, 1)[:, None, :]
    return x.to(BF16)


def _gn_check(B, HW, C, ratio, silu, eps, seed, grads):
    from e4t_b200 import ops
    G = 32
    g = _gen(seed)
    x = _gn_input(B, HW, C, G, ratio, g)
    gamma = 1 + 0.1 * _f32((C,), g)
    beta = 0.1 * _f32((C,), g)
    xr = x.double().permute(0, 2, 1).requires_grad_(grads)
    gr = gamma.double().requires_grad_(grads)
    br = beta.double().requires_grad_(grads)
    z = F.group_norm(xr, G, gr, br, eps)
    yr = F.silu(z) if silu else z
    y, stats = ops.groupnorm_fwd(x, gamma, beta, G, eps, silu)
    zt = z.detach().permute(0, 2, 1)
    # the fused SiLU's sigmoid is one tanh.approx (|error| <= 2^-12 on the sigmoid): allow 2^-11 |z| on top
    check_bf16(y, yr.detach().permute(0, 2, 1), "groupnorm fwd", extra=2.0 ** -11 * zt.abs() if silu else None)
    if not grads:
        return
    dy = _mk((B, HW, C), g)
    yr.backward(dy.double().permute(0, 2, 1))
    dx = ops.groupnorm_bwd(x, dy, gamma, beta, stats, G, eps, silu)
    extra = None
    if silu:   # the same approximation inside silu'(z): 2^-11 (1 + |z|) |dy gamma| rstd
        var = x.double().view(B, HW, G, C // G).var(dim=(1, 3), unbiased=False)
        rstd = (var + eps).rsqrt().repeat_interleave(C // G, 1)[:, None, :]
        extra = 2.0 ** -11 * (1 + zt.abs()) * (dy.double() * gamma.double()).abs() * rstd
    check_bf16(dx, xr.grad.permute(0, 2, 1), "groupnorm bwd", extra=extra)
    dg, db = ops.groupnorm_param_grad(x, dy, stats, gamma, beta, G, eps, silu)
    check_f32(dg, gr.grad, "groupnorm dgamma")
    check_f32(db, br.grad, "groupnorm dbeta")


_GN = [(C, HW, r) for C, HW in ((128, 512 * 512), (512, 64 * 64), (320, 64 * 64)) for r in (0, 8, 32, 128)]
_GN_VARIANTS = [(False, 1e-6), (True, 1e-6), (False, 1e-5), (True, 1e-5)]


@pytest.mark.parametrize("i", range(len(_GN)), ids=[f"C{c}-HW{hw}-r{r}" for c, hw, r in _GN])
def test_groupnorm_offset_groups(i):
    C, HW, ratio = _GN[i]
    B = 1 if HW > 64 * 64 else 2
    for silu, eps in (_GN_VARIANTS[i % 4], _GN_VARIANTS[(i + 1) % 4]):
        _gn_check(B, HW, C, ratio, silu, eps, seed=i * 10 + silu, grads=ratio <= 32)


def test_groupnorm_vae_batch():
    """B = 16 at 512^2 x 128: the grid heuristic divides its row chunks by B."""
    _gn_check(16, 512 * 512, 128, 8, True, 1e-6, seed=16, grads=False)


# =====================================================================================================================
# VAE end to end at 512^2
# =====================================================================================================================
def test_vae_sd14_512_end_to_end():
    """SD-v1.4 AutoencoderKL with synthetic weights at its real resolution, B = 2, against the fp32 oracle on the GPU.
    Bound: twice the oracle's own bf16-autocast error, measured here (the convention of the committed fixtures)."""
    from test_vae_gpu import _vae
    m, sd = _vae(V.SD14_VAE, 21)
    sd = {k: v.cuda() for k, v in sd.items()}
    gen = torch.Generator().manual_seed(22)
    x = (torch.rand(2, 3, 512, 512, generator=gen) * 2 - 1).cuda()
    z = torch.randn(2, 4, 64, 64, generator=gen).cuda()
    with torch.no_grad():
        d = m.encode(x).latent_dist
        dec = m.decode(z).sample
        mean, logvar = V.vae_encode(sd, V.SD14_VAE, x)
        ref_dec = V.vae_decode(sd, V.SD14_VAE, z)
        with torch.autocast("cuda", dtype=BF16):
            mean_a, logvar_a = V.vae_encode(sd, V.SD14_VAE, x)
            dec_a = V.vae_decode(sd, V.SD14_VAE, z)
    for name, ours, ref, auto in (("mean", d.mean, mean, mean_a), ("logvar", d.logvar, logvar, logvar_a),
                                  ("decode", dec, ref_dec, dec_a)):
        err = (ours.float() - ref).abs().max().item()
        tol = (auto.float() - ref).abs().max().item()
        _note("vae 512 e2e", err / (2 * tol))
        print(f"[vae sd14 512] {name}: max err {err:.3e}, bf16-autocast oracle {tol:.3e}")
        assert ours.shape == ref.shape and torch.isfinite(ours).all()
        assert err <= 2 * tol, (name, err, tol)
