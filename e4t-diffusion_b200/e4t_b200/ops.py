"""Raw (non-autograd) wrappers over the C-ABI entry points declared in include/e4t_b200.h.

Every function takes CUDA tensors, launches hand-written sm_100a kernels on torch's current stream and
returns torch tensors that merely own the output memory.
"""
import ctypes

import torch

from . import _lib
from ._lib import c_float, c_int, c_ll, c_void_p, ptr, stream

BF16 = torch.bfloat16
F32 = torch.float32


def _fp(t):
    return ptr(t)


def gemm(A, B, *, a_mn=False, b_mn=False, out=None, out_dtype=BF16, bias=None, rowgroup=None,
         rows_per_group=1, residual=None, alpha=1.0, splits=1, accumulate=False, force_bn=0):
    """out[b] = alpha * op(A[b]) @ op(B[b])^T (+bias +rowgroup +residual).

    K-major operands are (.., rows, K) with K contiguous; MN-major operands are (.., K, rows) with rows
    contiguous (i.e. the transposed storage).  A 2-D operand is shared across the batch.
    accumulate=True -> fp32 atomic accumulation into `out` (required for split-K).
    """
    assert A.dtype == BF16 and B.dtype == BF16
    assert A.stride(-1) == 1 and B.stride(-1) == 1
    batch = 1
    if A.dim() == 3:
        batch = A.shape[0]
    if B.dim() == 3:
        batch = max(batch, B.shape[0])
    if a_mn:
        K, M = A.shape[-2], A.shape[-1]
    else:
        M, K = A.shape[-2], A.shape[-1]
    if b_mn:
        Kb, N = B.shape[-2], B.shape[-1]
    else:
        N, Kb = B.shape[-2], B.shape[-1]
    assert K == Kb, (A.shape, B.shape, a_mn, b_mn)
    a_bs = A.stride(0) if A.dim() == 3 and batch > 1 else 0
    b_bs = B.stride(0) if B.dim() == 3 and batch > 1 else 0
    if accumulate:
        assert out is not None and out.dtype == F32
        out_mode = 2
    else:
        if out is None:
            shape = (batch, M, N) if (A.dim() == 3 or B.dim() == 3) else (M, N)
            out = torch.empty(shape, device=A.device, dtype=out_dtype)
        out_mode = 0 if out.dtype == BF16 else 1
    assert out.stride(-1) == 1
    o_bs = out.stride(0) if out.dim() == 3 and batch > 1 else 0
    r_bs = 0
    ldr = 0
    if residual is not None:
        assert residual.dtype == BF16 and residual.stride(-1) == 1
        ldr = residual.stride(-2)
        r_bs = residual.stride(0) if residual.dim() == 3 and batch > 1 else 0
    if bias is not None:
        assert bias.dtype == F32 and bias.is_contiguous()
    if rowgroup is not None:
        assert rowgroup.dtype == F32 and rowgroup.is_contiguous()
    _lib.call("e4t_gemm_bf16", ptr(A), ptr(B), ptr(out), c_int(M), c_int(N), c_int(K), c_int(batch),
              c_int(int(a_mn)), c_int(int(b_mn)), c_ll(A.stride(-2)), c_ll(B.stride(-2)), c_ll(a_bs), c_ll(b_bs),
              c_int(out_mode), c_ll(out.stride(-2)), c_ll(o_bs), ptr(bias), ptr(rowgroup), c_int(rows_per_group),
              ptr(residual), c_ll(ldr), c_ll(r_bs), c_float(alpha), c_int(splits), c_int(force_bn), stream())
    return out


def conv3x3(x, w9, *, bias=None, rowgroup=None, residual=None, out_dtype=BF16, force_bn=0):
    """3x3 stride-1 pad-1 convolution on NHWC bf16.  x: (B,H,W,Cin); w9: (9,Cout,Cin) bf16, tap = ky*3+kx."""
    assert x.dtype == BF16 and w9.dtype == BF16 and x.is_contiguous() and w9.is_contiguous()
    Bn, H, W, Cin = x.shape
    Cout = w9.shape[1]
    assert w9.shape == (9, Cout, Cin)
    out = torch.empty((Bn, H, W, Cout), device=x.device, dtype=out_dtype)
    if residual is not None:
        assert residual.dtype == BF16 and residual.is_contiguous() and residual.shape == out.shape
    _lib.call("e4t_conv3x3_bf16", ptr(x), ptr(w9), ptr(out), c_int(Bn), c_int(H), c_int(W), c_int(Cin), c_int(Cout),
              c_int(0 if out_dtype == BF16 else 1), ptr(bias), ptr(rowgroup), ptr(residual), c_int(force_bn),
              stream())
    return out


def conv3x3_s2(x, w9, *, bias=None, force_bn=0):
    """3x3 stride-2 pad-1 convolution on NHWC bf16 (Downsample2D): (B,H,W,Cin) -> (B,H/2,W/2,Cout)."""
    assert x.dtype == BF16 and w9.dtype == BF16 and x.is_contiguous() and w9.is_contiguous()
    Bn, H, W, Cin = x.shape
    Cout = w9.shape[1]
    out = torch.empty((Bn, H // 2, W // 2, Cout), device=x.device, dtype=BF16)
    _lib.call("e4t_conv3x3_s2_bf16", ptr(x), ptr(w9), ptr(out), c_int(Bn), c_int(H), c_int(W), c_int(Cin), c_int(Cout),
              ptr(bias), c_int(force_bn), stream())
    return out


def conv3x3_ex(x, w9, *, stride=1, pad=1, bias=None, residual=None, force_bn=0):
    """3x3 convolution on NHWC bf16 with stride 1/2 and top/left padding 1, or 0 with stride 2 (the VAE's
    F.pad(x, (0,1,0,1)) downsample): (B,H,W,Cin) -> (B,H/stride,W/stride,Cout) bf16."""
    assert x.dtype == BF16 and w9.dtype == BF16 and x.is_contiguous() and w9.is_contiguous()
    Bn, H, W, Cin = x.shape
    Cout = w9.shape[1]
    assert w9.shape == (9, Cout, Cin)
    out = torch.empty((Bn, H // stride, W // stride, Cout), device=x.device, dtype=BF16)
    if residual is not None:
        assert residual.dtype == BF16 and residual.is_contiguous() and residual.shape == out.shape
    _lib.call("e4t_conv3x3_ex", ptr(x), ptr(w9), ptr(out), c_int(Bn), c_int(H), c_int(W), c_int(Cin), c_int(Cout),
              c_int(stride), c_int(pad), ptr(bias), ptr(residual), c_int(force_bn), stream())
    return out


def softmax_rows(S, out=None):
    """Row softmax of an fp32 matrix (.., M) (last dim contiguous, rows evenly strided) -> bf16 of the same shape."""
    assert S.dtype == F32 and S.stride(-1) == 1
    M = S.shape[-1]
    S2 = S.reshape(-1, M) if S.dim() != 2 else S
    if out is None:
        out = torch.empty(S.shape, device=S.device, dtype=BF16)
    assert out.is_contiguous() and S2.stride(0) == M
    _lib.call("e4t_softmax_rows", ptr(S2), ptr(out), c_ll(S2.shape[0]), c_int(M), c_ll(M), stream())
    return out


# ----------------------------------------------------------------------------------------------
# normalisation
# ----------------------------------------------------------------------------------------------
def groupnorm_fwd(x, gamma, beta, groups, eps, silu):
    """x: (B,HW,C) or (B,H,W,C) bf16 NHWC.  Returns (y, stats[B,G,2] = (sum, sumsq) of x - p), p = each group's first
    element x[b, 0, g * C // G] (see groupnorm_mean_rstd)."""
    assert x.dtype == BF16 and x.is_contiguous()
    Bn, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (Bn * C)
    y = torch.empty_like(x)
    stats = torch.empty((Bn, groups, 2), device=x.device, dtype=F32)
    _lib.call("e4t_groupnorm_fwd", ptr(x), ptr(gamma), ptr(beta), ptr(y), ptr(stats), c_int(Bn), c_int(HW), c_int(C),
              c_int(groups), c_float(eps), c_int(int(silu)), stream())
    return y, stats


def groupnorm_bwd(x, dy, gamma, beta, stats, groups, eps, silu):
    assert x.dtype == BF16 and dy.dtype == BF16 and x.is_contiguous() and dy.is_contiguous()
    Bn, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (Bn * C)
    dx = torch.empty_like(x)
    scratch = torch.empty((Bn, groups, 2), device=x.device, dtype=F32)
    _lib.call("e4t_groupnorm_bwd", ptr(x), ptr(dy), ptr(gamma), ptr(beta), ptr(stats), ptr(dx), ptr(scratch),
              c_int(Bn), c_int(HW), c_int(C), c_int(groups), c_float(eps), c_int(int(silu)), stream())
    return dx


def layernorm_fwd(x, gamma, beta, eps):
    assert x.dtype == BF16 and x.is_contiguous()
    C = x.shape[-1]
    rows = x.numel() // C
    y = torch.empty_like(x)
    stats = torch.empty((rows, 2), device=x.device, dtype=F32)
    _lib.call("e4t_layernorm_fwd", ptr(x), ptr(gamma), ptr(beta), ptr(y), ptr(stats), c_ll(rows), c_int(C),
              c_float(eps), stream())
    return y, stats


def layernorm_bwd(x, dy, gamma, stats, eps):
    assert x.dtype == BF16 and dy.dtype == BF16 and x.is_contiguous() and dy.is_contiguous()
    C = x.shape[-1]
    rows = x.numel() // C
    dx = torch.empty_like(x)
    _lib.call("e4t_layernorm_bwd", ptr(x), ptr(dy), ptr(gamma), ptr(stats), ptr(dx), c_ll(rows), c_int(C),
              c_float(eps), stream())
    return dx


# ----------------------------------------------------------------------------------------------
# elementwise
# ----------------------------------------------------------------------------------------------
def geglu_fwd(h):
    assert h.dtype == BF16 and h.is_contiguous()
    F = h.shape[-1] // 2
    rows = h.numel() // (2 * F)
    out = torch.empty(h.shape[:-1] + (F,), device=h.device, dtype=BF16)
    _lib.call("e4t_geglu_fwd", ptr(h), ptr(out), c_ll(rows), c_int(F), stream())
    return out


def geglu_bwd(h, dout):
    assert h.dtype == BF16 and dout.dtype == BF16 and h.is_contiguous() and dout.is_contiguous()
    F = h.shape[-1] // 2
    rows = h.numel() // (2 * F)
    dh = torch.empty_like(h)
    _lib.call("e4t_geglu_bwd", ptr(h), ptr(dout), ptr(dh), c_ll(rows), c_int(F), stream())
    return dh


def resample2x(x, mode):
    """NHWC bf16.  mode 0 nearest-up, 1 its adjoint, 2 stride-2 pick, 3 zero-insertion (adjoint of 2)."""
    assert x.dtype == BF16 and x.is_contiguous() and x.dim() == 4
    Bn, Hx, Wx, C = x.shape
    if mode in (0, 3):
        H, W = Hx, Wx
        y = torch.empty((Bn, 2 * H, 2 * W, C), device=x.device, dtype=BF16)
    else:
        H, W = Hx // 2, Wx // 2
        y = torch.empty((Bn, H, W, C), device=x.device, dtype=BF16)
    _lib.call("e4t_resample2x", ptr(x), ptr(y), c_int(Bn), c_int(H), c_int(W), c_int(C), c_int(mode), stream())
    return y


def meanpool_fwd(x, out, c_off):
    """x (B,HW,C)/(B,H,W,C) bf16 -> out[:, c_off:c_off+C] (fp32, (B, ldo))."""
    assert x.dtype == BF16 and x.is_contiguous() and out.dtype == F32 and out.stride(1) == 1
    Bn, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (Bn * C)
    _lib.call("e4t_meanpool_fwd", ptr(x), ptr(out), c_int(Bn), c_int(HW), c_int(C), c_int(out.stride(0)), c_int(c_off),
              stream())


def meanpool_bwd(dout, shape, c_off):
    assert dout.dtype == F32 and dout.stride(1) == 1
    Bn, C = shape[0], shape[-1]
    HW = 1
    for s in shape[1:-1]:
        HW *= s
    dx = torch.empty(shape, device=dout.device, dtype=BF16)
    _lib.call("e4t_meanpool_bwd", ptr(dout), ptr(dx), c_int(Bn), c_int(HW), c_int(C), c_int(dout.stride(0)),
              c_int(c_off), stream())
    return dx


def conv_in_fwd(x, w, bias):
    """x NCHW fp32 (B,Cin,H,W) -> NHWC bf16 (B,H,W,Cout).  w fp32 (Cout,Cin,3,3)."""
    assert x.dtype == F32 and x.is_contiguous() and w.dtype == F32 and w.is_contiguous()
    Bn, Cin, H, W = x.shape
    Cout = w.shape[0]
    y = torch.empty((Bn, H, W, Cout), device=x.device, dtype=BF16)
    _lib.call("e4t_conv_in_fwd", ptr(x), ptr(w), ptr(bias), ptr(y), c_int(Bn), c_int(Cin), c_int(H), c_int(W),
              c_int(Cout), stream())
    return y


def pointwise_nchw(x, w, bias):
    """1x1 convolution on NCHW fp32 (B,Cin,H,W) -> (B,Cout,H,W); w fp32 (Cout,Cin)."""
    assert x.dtype == F32 and x.is_contiguous() and w.dtype == F32 and w.is_contiguous()
    Bn, Cin, H, W = x.shape
    Cout = w.shape[0]
    y = torch.empty((Bn, Cout, H, W), device=x.device, dtype=F32)
    _lib.call("e4t_pointwise_nchw", ptr(x), ptr(w), ptr(bias), ptr(y), c_int(Bn), c_int(Cin), c_int(Cout),
              c_ll(H * W), stream())
    return y


def conv_out_fwd(x, w, bias):
    """x NHWC bf16 (B,H,W,C) -> NCHW fp32 (B,Cout,H,W)."""
    assert x.dtype == BF16 and x.is_contiguous() and w.dtype == F32 and w.is_contiguous()
    Bn, H, W, C = x.shape
    Cout = w.shape[0]
    y = torch.empty((Bn, Cout, H, W), device=x.device, dtype=F32)
    _lib.call("e4t_conv_out_fwd", ptr(x), ptr(w), ptr(bias), ptr(y), c_int(Bn), c_int(H), c_int(W), c_int(C),
              c_int(Cout), stream())
    return y


def conv_out_bwd(dy, w, C):
    assert dy.dtype == F32 and dy.is_contiguous()
    Bn, Cout, H, W = dy.shape
    dx = torch.empty((Bn, H, W, C), device=dy.device, dtype=BF16)
    _lib.call("e4t_conv_out_bwd", ptr(dy), ptr(w), ptr(dx), c_int(Bn), c_int(H), c_int(W), c_int(C), c_int(Cout),
              stream())
    return dx


# ----------------------------------------------------------------------------------------------
# WeightOffsets
# ----------------------------------------------------------------------------------------------
def wo_factors(v, w1, b1, w2, b2, Wc, Wr):
    R, C = Wc.shape[0], Wr.shape[0]
    buf = torch.empty(2 * R + 3 * C, device=v.device, dtype=F32)
    vx, a, vy, b, s = buf[:R], buf[R:2 * R], buf[2 * R:2 * R + C], buf[2 * R + C:2 * R + 2 * C], buf[2 * R + 2 * C:]
    _lib.call("e4t_wo_factors_fwd", ptr(v), ptr(w1), ptr(b1), ptr(w2), ptr(b2), ptr(Wc), ptr(Wr), ptr(vx), ptr(vy),
              ptr(a), ptr(b), ptr(s), c_int(R), c_int(C), stream())
    return vx, vy, a, b, s


def wo_weff(W, a, bc, b, s, br, out=None):
    C, R = W.shape
    if out is None:
        out = torch.empty((C, R), device=W.device, dtype=BF16)
    assert out.is_contiguous() and out.shape == (C, R) and out.dtype == BF16
    _lib.call("e4t_wo_weff_fwd", ptr(W), ptr(a), ptr(bc), ptr(b), ptr(s), ptr(br), ptr(out), c_int(C), c_int(R),
              stream())
    return out


def wo_bwd(dWeff, W, v, w1, w2, Wc, Wr, bc, vx, vy, a, b, s, outs=None):
    """outs: optional 9 preallocated gradient tensors (dv,dw1,db1,dw2,db2,dWc,dbc,dWr,dbr) that are WRITTEN."""
    C, R = W.shape
    dev = W.device
    scratch = torch.empty(3 * C + 2 * R + R + C, device=dev, dtype=F32)
    if outs is not None:
        dv, dw1, db1, dw2, db2, dWc, dbc, dWr, dbr = outs
        for t in outs:
            assert t.dtype == F32 and t.is_contiguous()
    else:
        dv = torch.empty(1, device=dev, dtype=F32)
        dw1 = torch.empty(R, device=dev, dtype=F32); db1 = torch.empty(R, device=dev, dtype=F32)
        dw2 = torch.empty(C, device=dev, dtype=F32); db2 = torch.empty(C, device=dev, dtype=F32)
        dWc = torch.empty((R, R), device=dev, dtype=F32); dbc = torch.empty(R, device=dev, dtype=F32)
        dWr = torch.empty((C, C), device=dev, dtype=F32); dbr = torch.empty(C, device=dev, dtype=F32)
    _lib.call("e4t_wo_bwd", ptr(dWeff), ptr(W), ptr(v), ptr(w1), ptr(w2), ptr(Wc), ptr(Wr), ptr(bc), ptr(vx), ptr(vy),
              ptr(a), ptr(b), ptr(s), ptr(scratch), ptr(dv), ptr(dw1), ptr(db1), ptr(dw2), ptr(db2), ptr(dWc),
              ptr(dbc), ptr(dWr), ptr(dbr), c_int(R), c_int(C), stream())
    return dv, dw1, db1, dw2, db2, dWc, dbc, dWr, dbr


def adamw_step(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0):
    assert p.dtype == F32 and p.is_contiguous() and g.is_contiguous() and m.is_contiguous() and v.is_contiguous()
    _lib.call("e4t_adamw_step", ptr(p), ptr(g), ptr(m), ptr(v), c_ll(p.numel()), c_float(lr), c_float(beta1),
              c_float(beta2), c_float(eps), c_float(weight_decay), c_int(step), c_float(grad_scale), stream())


def adamw_step_dev(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step_dev, grad_scale=1.0):
    """AdamW with the step counter in device memory (int32 tensor, incremented by the call): graph-replayable."""
    assert p.dtype == F32 and step_dev.dtype == torch.int32
    _lib.call("e4t_adamw_step_dev", ptr(p), ptr(g), ptr(m), ptr(v), c_ll(p.numel()), c_float(lr), c_float(beta1),
              c_float(beta2), c_float(eps), c_float(weight_decay), ptr(step_dev), c_float(grad_scale), stream())


# ----------------------------------------------------------------------------------------------
# attention core
# ----------------------------------------------------------------------------------------------
def _bs(t):
    return t.stride(0)


def attn_fwd(q, k, v, heads, scale=None):
    """q (B,N,H*dh), k/v (B,M,H*dh) bf16 (last dim contiguous; may be column slices of a fused projection).
    Returns (o (B,N,H*dh) bf16, lse (B,H,N) fp32)."""
    assert q.dtype == BF16 and k.dtype == BF16 and v.dtype == BF16
    assert q.stride(-1) == 1 and k.stride(-1) == 1 and v.stride(-1) == 1
    Bn, N, C = q.shape
    M = k.shape[1]
    dh = C // heads
    scale = dh ** -0.5 if scale is None else scale
    o = torch.empty((Bn, N, C), device=q.device, dtype=BF16)
    lse = torch.empty((Bn, heads, N), device=q.device, dtype=F32)
    _lib.call("e4t_attn_fwd", ptr(q), ptr(k), ptr(v), ptr(o), ptr(lse), c_int(Bn), c_int(heads), c_int(N), c_int(M),
              c_int(dh), c_ll(q.stride(1)), c_ll(_bs(q)), c_ll(k.stride(1)), c_ll(_bs(k)), c_ll(v.stride(1)),
              c_ll(_bs(v)), c_ll(o.stride(1)), c_ll(_bs(o)), c_float(scale), stream())
    return o, lse


def attn_bwd(q, k, v, o, do, lse, heads, scale=None, dq=None, dk=None, dv=None, fused=True, causal=False):
    """dq/dk/dv may be preallocated (e.g. column slices of one fused (B,N,3C) gradient buffer).
    fused=True: single-pass backward (S/dP computed once per tile pair, dQ reduced in fp32) when the head dim fits
    the TMEM budget (dh <= 80); otherwise / fused=False the two-kernel (dQ, dK/dV) path.
    causal=True (N == M, dh <= 80): key j contributes to query i only if j <= i; o / lse must come from a forward that
    applied the same mask (attn_small_fwd)."""
    assert do.dtype == BF16 and do.stride(-1) == 1
    Bn, N, C = q.shape
    M = k.shape[1]
    dh = C // heads
    scale = dh ** -0.5 if scale is None else scale
    dq = torch.empty((Bn, N, C), device=q.device, dtype=BF16) if dq is None else dq
    dk = torch.empty((Bn, M, C), device=q.device, dtype=BF16) if dk is None else dk
    dv = torch.empty((Bn, M, C), device=q.device, dtype=BF16) if dv is None else dv
    assert dq.stride(-1) == 1 and dk.stride(-1) == 1 and dv.stride(-1) == 1
    dlt = torch.empty((Bn, heads, N), device=q.device, dtype=F32)
    assert not causal or (dh <= 80 and N == M), "causal attention backward: dh <= 80 and N == M"
    if causal or (fused and dh <= 80 and N >= 128):
        dqacc = torch.empty((Bn, N, C), device=q.device, dtype=F32)
        _lib.call("e4t_attn_bwd_fused_causal" if causal else "e4t_attn_bwd_fused", ptr(q), ptr(k), ptr(v), ptr(o), ptr(do), ptr(lse), ptr(dlt), ptr(dqacc),
                  ptr(dq), ptr(dk), ptr(dv), c_int(Bn), c_int(heads), c_int(N), c_int(M), c_int(dh),
                  c_ll(q.stride(1)), c_ll(_bs(q)), c_ll(k.stride(1)), c_ll(_bs(k)), c_ll(v.stride(1)), c_ll(_bs(v)),
                  c_ll(o.stride(1)), c_ll(_bs(o)), c_ll(do.stride(1)), c_ll(_bs(do)), c_ll(dq.stride(1)),
                  c_ll(_bs(dq)), c_ll(dk.stride(1)), c_ll(_bs(dk)), c_ll(dv.stride(1)), c_ll(_bs(dv)),
                  c_float(scale), stream())
        return dq, dk, dv
    _lib.call("e4t_attn_bwd", ptr(q), ptr(k), ptr(v), ptr(o), ptr(do), ptr(lse), ptr(dlt), ptr(dq), ptr(dk), ptr(dv),
              c_int(Bn), c_int(heads), c_int(N), c_int(M), c_int(dh), c_ll(q.stride(1)), c_ll(_bs(q)),
              c_ll(k.stride(1)), c_ll(_bs(k)), c_ll(v.stride(1)), c_ll(_bs(v)), c_ll(o.stride(1)), c_ll(_bs(o)),
              c_ll(do.stride(1)), c_ll(_bs(do)), c_ll(dq.stride(1)), c_ll(_bs(dq)), c_ll(dk.stride(1)), c_ll(_bs(dk)),
              c_ll(dv.stride(1)), c_ll(_bs(dv)), c_float(scale), stream())
    return dq, dk, dv


# ----------------------------------------------------------------------------------------------
# small operators (csrc/small_ops.cu) and weight gradients
# ----------------------------------------------------------------------------------------------
ACT_GELU, ACT_QUICK_GELU, ACT_LEAKY_RELU = 0, 1, 2


def act_fwd(x, mode):
    assert x.dtype == BF16 and x.is_contiguous()
    y = torch.empty_like(x)
    _lib.call("e4t_act_fwd", ptr(x), ptr(y), c_ll(x.numel()), c_int(mode), stream())
    return y


def act_bwd(x, dy, mode):
    assert x.dtype == BF16 and dy.dtype == BF16 and x.is_contiguous() and dy.is_contiguous()
    dx = torch.empty_like(x)
    _lib.call("e4t_act_bwd", ptr(x), ptr(dy), ptr(dx), c_ll(x.numel()), c_int(mode), stream())
    return dx


def colsum_acc(x2, out, rows_per_group=0):
    """out[g][n] += sum of the rows of group g of x2 (bf16 (M,N), row stride = x2.stride(0)); out fp32, pre-initialised."""
    assert x2.dtype == BF16 and x2.dim() == 2 and x2.stride(1) == 1 and out.dtype == F32 and out.is_contiguous()
    _lib.call("e4t_colsum_acc", ptr(x2), ptr(out), c_ll(x2.shape[0]), c_int(x2.shape[1]), c_ll(x2.stride(0)),
              c_ll(rows_per_group), stream())
    return out


def attn_small_fwd(q, k, v, heads, scale=None, causal=False):
    """Short-sequence attention (N, M <= 128, dh <= 64) with optional causal mask; same layout as attn_fwd."""
    assert q.dtype == BF16 and k.dtype == BF16 and v.dtype == BF16
    assert q.stride(-1) == 1 and k.stride(-1) == 1 and v.stride(-1) == 1
    Bn, N, C = q.shape
    M = k.shape[1]
    dh = C // heads
    scale = dh ** -0.5 if scale is None else scale
    o = torch.empty((Bn, N, C), device=q.device, dtype=BF16)
    lse = torch.empty((Bn, heads, N), device=q.device, dtype=F32)
    _lib.call("e4t_attn_small_fwd", ptr(q), ptr(k), ptr(v), ptr(o), ptr(lse), c_int(Bn), c_int(heads), c_int(N),
              c_int(M), c_int(dh), c_ll(q.stride(1)), c_ll(_bs(q)), c_ll(k.stride(1)), c_ll(_bs(k)), c_ll(v.stride(1)),
              c_ll(_bs(v)), c_ll(o.stride(1)), c_ll(_bs(o)), c_float(scale), c_int(int(causal)), stream())
    return o, lse


def attn_small_bwd(q, k, v, o, do, lse, heads, scale=None, causal=False, dq=None, dk=None, dv=None):
    assert do.dtype == BF16 and do.stride(-1) == 1
    Bn, N, C = q.shape
    M = k.shape[1]
    dh = C // heads
    scale = dh ** -0.5 if scale is None else scale
    dq = torch.empty((Bn, N, C), device=q.device, dtype=BF16) if dq is None else dq
    dk = torch.empty((Bn, M, C), device=q.device, dtype=BF16) if dk is None else dk
    dv = torch.empty((Bn, M, C), device=q.device, dtype=BF16) if dv is None else dv
    _lib.call("e4t_attn_small_bwd", ptr(q), ptr(k), ptr(v), ptr(o), ptr(do), ptr(lse), ptr(dq), ptr(dk), ptr(dv),
              c_int(Bn), c_int(heads), c_int(N), c_int(M), c_int(dh), c_ll(q.stride(1)), c_ll(_bs(q)),
              c_ll(k.stride(1)), c_ll(_bs(k)), c_ll(v.stride(1)), c_ll(_bs(v)), c_ll(o.stride(1)), c_ll(_bs(o)),
              c_ll(do.stride(1)), c_ll(_bs(do)), c_ll(dq.stride(1)), c_ll(_bs(dq)), c_ll(dk.stride(1)), c_ll(_bs(dk)),
              c_ll(dv.stride(1)), c_ll(_bs(dv)), c_float(scale), c_int(int(causal)), stream())
    return dq, dk, dv


def layernorm_param_grad(x, dy, stats, gamma):
    """(dgamma, dbeta) fp32 of LayerNorm given the forward's (mean, rstd) stats."""
    C = x.shape[-1]
    rows = x.numel() // C
    dg = torch.zeros(C, device=x.device, dtype=F32)
    db = torch.zeros(C, device=x.device, dtype=F32)
    _lib.call("e4t_layernorm_param_grad", ptr(x), ptr(dy), ptr(stats), ptr(gamma), ptr(dg), ptr(db), c_ll(rows), c_int(C),
              stream())
    return dg, db


def groupnorm_mean_rstd(x, stats, groups, eps):
    """(mean, rstd) fp32 (B, G) from groupnorm_fwd's stats, which are sums about each group's first element."""
    Bn, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (Bn * C)
    n = float(HW * (C // groups))
    pivot = x.reshape(Bn, HW, C)[:, 0, ::C // groups].float()
    d = stats[..., 0] / n
    var = (stats[..., 1] / n - d * d).clamp_min(0.0)
    return pivot + d, torch.rsqrt(var + eps)


def groupnorm_param_grad(x, dy, stats, gamma, beta, groups, eps, silu):
    """(dgamma, dbeta) fp32 of GroupNorm(+SiLU); stats = the forward's per-(image, group) sums."""
    Bn, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (Bn * C)
    mean, rstd = groupnorm_mean_rstd(x, stats, groups, eps)
    mean_c = mean.repeat_interleave(C // groups, dim=1).contiguous()
    rstd_c = rstd.repeat_interleave(C // groups, dim=1).contiguous()
    dg = torch.zeros(C, device=x.device, dtype=F32)
    db = torch.zeros(C, device=x.device, dtype=F32)
    _lib.call("e4t_groupnorm_param_grad", ptr(x), ptr(dy), ptr(mean_c), ptr(rstd_c), ptr(gamma), ptr(beta), ptr(dg),
              ptr(db), c_int(Bn), c_int(HW), c_int(C), c_int(int(silu)), stream())
    return dg, db


def narrow_conv_wgrad(wide, narrow, sgn):
    """acc[w][n][tap] = sum wide[b,y,x,w] * narrow[b,n,y+sgn*(ky-1),x+sgn*(kx-1)] (weight gradients of conv_in / conv_out)."""
    assert wide.dtype == BF16 and wide.is_contiguous() and narrow.dtype == F32 and narrow.is_contiguous()
    Bn, H, W, Cw = wide.shape
    Cn = narrow.shape[1]
    assert narrow.shape == (Bn, Cn, H, W)
    acc = torch.zeros((Cw, Cn, 9), device=wide.device, dtype=F32)
    _lib.call("e4t_narrow_conv_wgrad", ptr(wide), ptr(narrow), ptr(acc), c_int(Bn), c_int(H), c_int(W), c_int(Cw),
              c_int(Cn), c_int(sgn), stream())
    return acc


def conv3x3_wgrad(x, dy):
    """dW9 fp32 (9, Cout, Cin) of a 3x3/s1/p1 convolution on NHWC bf16 (x: (B,H,W,Cin), dy: (B,H,W,Cout))."""
    assert x.dtype == BF16 and dy.dtype == BF16 and x.is_contiguous() and dy.is_contiguous()
    Bn, H, W, Cin = x.shape
    Cout = dy.shape[-1]
    dw9 = torch.zeros((9, Cout, Cin), device=x.device, dtype=F32)
    _lib.call("e4t_conv3x3_wgrad", ptr(x), ptr(dy), ptr(dw9), c_int(Bn), c_int(H), c_int(W), c_int(Cin), c_int(Cout),
              stream())
    return dw9
