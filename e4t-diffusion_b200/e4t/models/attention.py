"""BasicTransformerBlock / FeedForward / GEGLU — mirror of e4t/models/attention.py:181-430 on the sm_100a kernels.
LayerNorm -> attn1 (self) -> LayerNorm -> attn2 (cross) -> LayerNorm -> GEGLU feed-forward, residual adds fused into
the producing GEMM epilogues.  AttentionBlock (attention.py:37-178): the VAE mid-block's single-head spatial
self-attention, forward only."""
from typing import Optional

import torch
from torch import nn

from e4t.models.cross_attention import CrossAttention, _weight_bf16
from e4t.models.resnet import f32
from e4t_b200 import functional as FN
from e4t_b200 import ops


class AttentionBlock(nn.Module):
    """attention.py:37-178 (diffusers 0.14), on channels-last (B,H,W,C) bf16, no-grad (the VAE is frozen):
    GroupNorm -> one q|k|v GEMM with bias -> S = C^-0.5 Q Kᵀ (fp32) -> row softmax -> P V -> proj_attn with the residual
    added in its epilogue.  The single head has dh = C (512 in SD-v1.x), past what the fused attention kernel holds in
    tensor memory; S is materialised instead (1 GB fp32 at B = 16, 4096 tokens)."""

    def __init__(self, channels: int, num_head_channels: Optional[int] = None, norm_num_groups: int = 32,
                 rescale_output_factor: float = 1.0, eps: float = 1e-5):
        super().__init__()
        self.channels = channels
        self.num_heads = channels // num_head_channels if num_head_channels is not None else 1
        self.num_head_size = num_head_channels
        if self.num_heads != 1:
            raise NotImplementedError("AttentionBlock: only num_heads == 1 (the SD-v1.x VAE) is supported")
        if rescale_output_factor != 1.0:
            raise NotImplementedError("AttentionBlock: rescale_output_factor != 1")
        self.group_norm = nn.GroupNorm(num_channels=channels, num_groups=norm_num_groups, eps=eps, affine=True)
        self.query = nn.Linear(channels, channels)
        self.key = nn.Linear(channels, channels)
        self.value = nn.Linear(channels, channels)
        self.rescale_output_factor = rescale_output_factor
        self.proj_attn = nn.Linear(channels, channels, 1)

    def _qkv(self):
        """q|k|v weights row-concatenated into one bf16 GEMM operand + the fp32 concatenated bias."""
        ps = (self.query, self.key, self.value)
        w = FN.prepared(self.query.weight, ("qkv_bf16", self.key.weight._version, self.value.weight._version,
                                            self.key.weight.data_ptr(), self.value.weight.data_ptr()),
                        lambda t: torch.cat([p.weight.detach() for p in ps], dim=0).to(torch.bfloat16).contiguous())
        b = FN.prepared(self.query.bias, ("qkv_f32", self.key.bias._version, self.value.bias._version,
                                          self.key.bias.data_ptr(), self.value.bias.data_ptr()),
                        lambda t: torch.cat([p.bias.detach() for p in ps], dim=0).float().contiguous())
        return w, b

    def forward(self, hidden_states):
        if torch.is_grad_enabled() and (hidden_states.requires_grad or
                                        any(p.requires_grad for p in self.parameters())):
            raise NotImplementedError("AttentionBlock is forward-only (call it under torch.no_grad())")
        x = FN._c(hidden_states)
        B, H, W, C = x.shape
        N = H * W
        gn = self.group_norm
        h = FN.GroupNormFn.apply(x, f32(gn.weight), f32(gn.bias), gn.num_groups, gn.eps, False)
        w_qkv, b_qkv = self._qkv()
        qkv = ops.gemm(h.view(B * N, C), w_qkv, bias=b_qkv).view(B, N, 3 * C)
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        s = ops.gemm(q, k, out_dtype=torch.float32, alpha=C ** -0.5)              # (B,N,N) fp32
        p = ops.softmax_rows(s)
        del s
        o = ops.gemm(p, v, b_mn=True)                                               # (B,N,C)
        out = ops.gemm(o.view(B * N, C), _weight_bf16(self.proj_attn), bias=f32(self.proj_attn.bias),
                       residual=x.view(B * N, C))
        return out.view(B, H, W, C)


class GEGLU(nn.Module):
    """attention.py:409-430: proj: dim_in -> 2*dim_out, out = h * gelu(gate) (exact erf GELU)."""

    def __init__(self, dim_in: int, dim_out: int):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)

    def forward(self, hidden_states):
        h = FN.LinearFn.apply(hidden_states, _weight_bf16(self.proj), self.proj.bias, None, self.proj.weight)
        return FN.GEGLUFn.apply(h)


class FeedForward(nn.Module):
    """attention.py:335-384 (activation_fn='geglu', the only variant SD-v1.x builds)."""

    def __init__(self, dim: int, dim_out: Optional[int] = None, mult: int = 4, dropout: float = 0.0,
                 activation_fn: str = "geglu", final_dropout: bool = False):
        super().__init__()
        if activation_fn != "geglu":
            raise NotImplementedError("only GEGLU feed-forward is on the SD-v1.x path")
        inner_dim = int(dim * mult)
        dim_out = dim_out if dim_out is not None else dim
        self.net = nn.ModuleList([GEGLU(dim, inner_dim), nn.Dropout(dropout), nn.Linear(inner_dim, dim_out)])

    def forward(self, hidden_states, residual=None):
        h = self.net[0](hidden_states)
        return FN.LinearFn.apply(h, _weight_bf16(self.net[2]), self.net[2].bias, residual, self.net[2].weight)


class BasicTransformerBlock(nn.Module):
    """attention.py:181-332."""

    def __init__(self, dim: int, num_attention_heads: int, attention_head_dim: int, dropout=0.0,
                 cross_attention_dim: Optional[int] = None, activation_fn: str = "geglu",
                 num_embeds_ada_norm: Optional[int] = None, attention_bias: bool = False,
                 only_cross_attention: bool = False, upcast_attention: bool = False,
                 norm_elementwise_affine: bool = True, norm_type: str = "layer_norm", final_dropout: bool = False):
        super().__init__()
        if norm_type != "layer_norm" or num_embeds_ada_norm is not None or only_cross_attention:
            raise NotImplementedError("AdaLayerNorm / only_cross_attention are not on the SD-v1.x path")
        self.only_cross_attention = only_cross_attention
        self.attn1 = CrossAttention(query_dim=dim, heads=num_attention_heads, dim_head=attention_head_dim,
                                    dropout=dropout, bias=attention_bias, upcast_attention=upcast_attention)
        self.ff = FeedForward(dim, dropout=dropout, activation_fn=activation_fn, final_dropout=final_dropout)
        self.attn2 = CrossAttention(query_dim=dim, cross_attention_dim=cross_attention_dim, heads=num_attention_heads,
                                    dim_head=attention_head_dim, dropout=dropout, bias=attention_bias,
                                    upcast_attention=upcast_attention) if cross_attention_dim is not None else None
        self.norm1 = nn.LayerNorm(dim, elementwise_affine=norm_elementwise_affine)
        self.norm2 = nn.LayerNorm(dim, elementwise_affine=norm_elementwise_affine) if self.attn2 is not None else None
        self.norm3 = nn.LayerNorm(dim, elementwise_affine=norm_elementwise_affine)

    @staticmethod
    def _ln(norm, x):
        return FN.LayerNormFn.apply(x, norm.weight, norm.bias, norm.eps)

    def forward(self, hidden_states, encoder_hidden_states=None, timestep=None, attention_mask=None,
                cross_attention_kwargs=None, class_labels=None):
        kw = cross_attention_kwargs if cross_attention_kwargs is not None else {}
        x = FN.as_bf16(hidden_states)
        x = self.attn1(self._ln(self.norm1, x), encoder_hidden_states=None, attention_mask=attention_mask,
                       residual=x, **kw)                                                   # attention.py:291-302
        if self.attn2 is not None:
            x = self.attn2(self._ln(self.norm2, x), encoder_hidden_states=encoder_hidden_states,
                           attention_mask=attention_mask, residual=x, **kw)                # :304-316
        return self.ff(self._ln(self.norm3, x), residual=x)                                # :318-330
