"""Drop-ins for ``vision_transformers/dilateformer.py``: ``GlobalAttention`` (dilateformer.py:136-164; SURVEY.md section 8 row
f-2), the multi-scale dilated attention ``MultiDilatelocalAttention`` (dilateformer.py:64-97) and ``DilateBlock``
(dilateformer.py:100-134) of DilateFormer's first two stages.

``GlobalAttention`` is ViT.Attention's math on a channels-last image: ``forward(x[B, H, W, C]) -> [B, H, W, C]`` attends over the
H * W positions (dilateformer.py:151-162).  The tokens of a contiguous ``[B, H, W, C]`` tensor ARE the ``[B, H*W, C]`` matrix, so
the class shares the ViT forward (co-scheduled single-launch kernel for 64-wide heads and <= 240 positions) through a view.

``MultiDilatelocalAttention`` runs as GEMM(qkv) -> this library's dilated-attention kernel -> GEMM(proj), one C-ABI call.
Deviation: for a contiguous x the reference writes the pre-projection attention output into the caller's x
(dilateformer.py:90-93 assign through a view of it); these drop-ins leave x untouched."""
from __future__ import annotations

import torch
from torch import nn

from . import _lib as L
from . import ops, vit
from ._common import StagedModule, check_forward_mode, f32, w16
from .cswin import Mlp


class GlobalAttention(vit.Attention):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0., proj_drop=0.):
        super().__init__(dim, num_heads, qkv_bias, attn_drop, proj_drop)
        if qk_scale:
            self.scale = qk_scale                  # dilateformer.py:144: qk_scale or head_dim ** -0.5

    def forward(self, x):
        B, H, W, C = x.shape
        return super().forward(x.reshape(B, H * W, C)).reshape(B, H, W, C)


class DilateAttention(nn.Module):
    """The per-group settings of dilateformer.py:41-61 (head_dim, scale, kernel_size, dilation, attn_drop).  It has no
    parameters and no forward of its own here: ``MultiDilatelocalAttention`` runs all groups in one kernel."""

    def __init__(self, head_dim, qk_scale=None, attn_drop=0, kernel_size=3, dilation=1):
        super().__init__()
        self.head_dim = head_dim
        self.scale = qk_scale or head_dim ** -0.5
        self.kernel_size = kernel_size
        self.dilation = dilation
        self.attn_drop = nn.Dropout(attn_drop)


def _dilate_args(a, attn, x, y):
    """Fill the pa_dilate_args part shared by the module and the block entry points."""
    B, H, W, C = x.shape
    dil = list(attn.dilation)
    if not 1 <= len(dil) <= 8:
        raise ValueError(f"{len(dil)} dilation groups unsupported (1 to 8)")
    a.dtype, a.out_dtype = ops.dtype_code(x.dtype), ops.dtype_code(y.dtype)
    a.B, a.Himg, a.Wimg, a.C, a.H = B, H, W, C, attn.num_heads
    a.kernel_size, a.n_dilation = int(attn.kernel_size), len(dil)
    for i, d in enumerate(dil):
        a.dilation[i] = int(d)
    a.scale = float(attn.scale)
    a.x, a.y = ops._ptr(x), ops._ptr(y)


class MultiDilatelocalAttention(StagedModule):
    """Same constructor, attributes, ``forward(x[B, H, W, C]) -> [B, H, W, C]`` contract and ``state_dict`` keys
    (``qkv.weight`` [3C, C, 1, 1], [``qkv.bias``], ``proj.weight``, ``proj.bias``) as the reference class (dilateformer.py:64-97).
    The 1x1 qkv conv is staged as a [3C, C] 16-bit matrix.  x is read, never written (see the module docstring)."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None,
                 attn_drop=0., proj_drop=0., kernel_size=3, dilation=[1, 2, 3]):
        super().__init__()
        self.dim = dim
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.dilation = dilation
        self.kernel_size = kernel_size
        self.scale = qk_scale or head_dim ** -0.5
        self.num_dilation = len(dilation)
        assert num_heads % self.num_dilation == 0, f"num_heads{num_heads} must be the times of num_dilation{self.num_dilation}!!"
        self.qkv = nn.Conv2d(dim, dim * 3, 1, bias=qkv_bias)
        self.dilate_attention = nn.ModuleList(
            [DilateAttention(head_dim, qk_scale, attn_drop, kernel_size, dilation[i])
             for i in range(self.num_dilation)])
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        self.out_dtype = None          # None: same dtype as x (fp32 with fp32_input).  torch.float16/float32 selectable
        self._init_stage()

    def _drops(self):
        return (self.dilate_attention[0].attn_drop.p, self.proj_drop.p)

    def _staged(self, dtype):
        q, p = self.qkv, self.proj
        C = self.dim
        return self._stage.get(
            ("w", dtype), (q.weight, q.bias, p.weight, p.bias),
            lambda: (w16(q.weight.reshape(3 * C, C), dtype), f32(q.bias), w16(p.weight, torch.float16), f32(p.bias)))

    def forward(self, x):
        x, y_dtype = self._prepare_input(x)
        check_forward_mode(self, x, self._drops())
        x = x.contiguous()
        wq, bq, wp, bp = self._staged(x.dtype)
        y = torch.empty(x.shape, dtype=self.out_dtype or y_dtype, device=x.device)
        a = L.DilateArgs()
        _dilate_args(a, self, x, y)
        a.qkv_weight, a.qkv_bias, a.proj_weight, a.proj_bias = ops._ptr(wq), ops._ptr(bq), ops._ptr(wp), ops._ptr(bp)
        ops.run_with_workspace(x, a, "pa_dilate_workspace_bytes", "pa_dilate_fwd")
        return y


class DropPath(nn.Module):
    """Stochastic depth (timm's DropPath, used by dilateformer.py:118 when drop_path > 0): the identity at eval.  The B200 path
    is forward-only, so dropping paths in training is an explicit error."""

    def __init__(self, drop_prob=0.):
        super().__init__()
        self.drop_prob = drop_prob

    def forward(self, x):
        if self.training and self.drop_prob > 0:
            raise NotImplementedError("drop_path > 0 in training mode is not implemented on the B200 forward path")
        return x


class DilateBlock(StagedModule):
    """Same constructor and ``state_dict`` keys as the reference block (dilateformer.py:100-124), ``pos_embed.*`` included when
    ``cpe_per_block``.  ``attention_half(x[B, H, W, C])`` = ``x + attn(norm1(x))`` (dilateformer.py:130) as ONE C-ABI call
    (``pa_dilate_block_attn_fwd``): LayerNorm kernel -> qkv GEMM -> dilated-attention kernel -> proj GEMM with the residual in its
    epilogue.  ``forward(x[B, C, H, W])`` runs the depthwise cpe conv, the MLP half and the permutes with the block's own PyTorch
    modules in THEIR parameter dtype (dilateformer.py:126-134), so the block works in a 16-bit model as well as in an fp32 model
    whose attention half is fed 16-bit activations (or fp32 ones with ``fp32_input`` set); the result has x's dtype."""

    def __init__(self, dim, num_heads, mlp_ratio=4., qkv_bias=False, qk_scale=None, drop=0., attn_drop=0.,
                 drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm, kernel_size=3, dilation=[1, 2, 3],
                 cpe_per_block=False):
        super().__init__()
        self.dim = dim
        self.num_heads = num_heads
        self.mlp_ratio = mlp_ratio
        self.kernel_size = kernel_size
        self.dilation = dilation
        self.cpe_per_block = cpe_per_block
        if self.cpe_per_block:
            self.pos_embed = nn.Conv2d(dim, dim, 3, padding=1, groups=dim)
        self.norm1 = norm_layer(dim)
        self.attn = MultiDilatelocalAttention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale,
                                              attn_drop=attn_drop, kernel_size=kernel_size, dilation=dilation)
        self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.norm2 = norm_layer(dim)
        mlp_hidden_dim = int(dim * mlp_ratio)
        self.mlp = Mlp(in_features=dim, hidden_features=mlp_hidden_dim, act_layer=act_layer, drop=drop)
        self.out_dtype = None
        self._init_stage()

    def attention_half(self, x):
        x, y_dtype = self._prepare_input(x)
        at = self.attn
        dp = self.drop_path.drop_prob if isinstance(self.drop_path, DropPath) else 0.
        check_forward_mode(self, x, at._drops())
        if self.training and dp > 0:
            raise NotImplementedError("drop_path > 0 in training mode is not implemented on the B200 forward path")
        if not isinstance(self.norm1, nn.LayerNorm):
            raise NotImplementedError("only norm_layer=nn.LayerNorm is implemented on the B200 path")
        x = x.contiguous()
        n1, q, p = self.norm1, at.qkv, at.proj
        C = self.dim
        wq, bq, wp, bp, g, b = self._stage.get(
            "w", (q.weight, q.bias, p.weight, p.bias, n1.weight, n1.bias),
            lambda: (w16(q.weight.reshape(3 * C, C), torch.float16), f32(q.bias), w16(p.weight, torch.float16), f32(p.bias),
                     f32(n1.weight), f32(n1.bias)))
        y = torch.empty(x.shape, dtype=self.out_dtype or y_dtype, device=x.device)
        a = L.DilateBlockArgs()
        _dilate_args(a.attn, at, x, y)
        a.attn.qkv_weight, a.attn.qkv_bias, a.attn.proj_weight, a.attn.proj_bias = ops._ptr(wq), ops._ptr(bq), ops._ptr(wp), ops._ptr(bp)
        a.ln_weight, a.ln_bias, a.ln_eps = ops._ptr(g), ops._ptr(b), float(n1.eps)
        ops.run_with_workspace(x, a, "pa_dilate_block_attn_workspace_bytes", "pa_dilate_block_attn_fwd")
        return y

    def forward(self, x):
        """dilateformer.py:126-134: NCHW in, NCHW out (a permuted view of a channels-last tensor, as the reference returns)."""
        h = x
        if self.cpe_per_block:
            hc = h.to(self.pos_embed.weight.dtype)
            h = (hc + self.pos_embed(hc)).to(x.dtype)
        y = self.attention_half(h.permute(0, 2, 3, 1))
        y = y.to(self.norm2.weight.dtype)
        y = y + self.drop_path(self.mlp(self.norm2(y)))
        return y.permute(0, 3, 1, 2).to(x.dtype)
