"""fp32 CPU restatement of DilateFormer's multi-scale dilated attention (TEST ORACLE), and its golden cases.

``dilateformer.MultiDilatelocalAttention`` (dilateformer.py:64-97) and ``DilateBlock`` (dilateformer.py:100-134) in explicit
pad / gather / einsum form, independent of the reference's unfold / reshape / permute chains.  The cases live in their own
dict and their golden files in ``tests/golden/dilate/`` (written by ``oracle/make_golden_dilate.py``), apart from
``GOLDEN_CASES`` and the top-level golden files, which other tests enumerate.

Only tests/ and tools/ may import this.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .attention import _dwconv_same, _layer_norm_rows, _lin, _softmax_last

DILATE_CASES = {
    # MultiDilatelocalAttention(dim, num_heads, qkv_bias, qk_scale, attn_drop, proj_drop, kernel_size, dilation)
    # dilateformer_tiny / small stage 1 width: C 72, 3 heads (head_dim 24), one head per dilation group
    "msda_b2_12x12_c72_h3_bias": dict(variant="msda", ctor=dict(dim=72, num_heads=3, qkv_bias=True), x=(2, 12, 12, 72)),
    # dilateformer_base stage 1 width: head_dim 32, non-square map
    "msda_b2_10x14_c96_h3": dict(variant="msda", ctor=dict(dim=96, num_heads=3), x=(2, 10, 14, 96)),
    # k = 5 and dilations [1, 3]: group 1's padding (6) exceeds the 5 x 6 map; two heads per group, head_dim 16
    "msda_b2_5x6_c64_h4_k5_d1_3": dict(variant="msda", ctor=dict(dim=64, num_heads=4, qkv_bias=True, kernel_size=5, dilation=[1, 3]),
                                       x=(2, 5, 6, 64)),
    # DilateBlock attention half on channels-last x: x + attn(norm1(x))       dilateformer.py:130
    "dilateblock_half_b2_12x12_c72_h3": dict(variant="dilate_block_half", ctor=dict(dim=72, num_heads=3, qkv_bias=True),
                                             x=(2, 12, 12, 72), keep=("norm1.", "attn.")),
    # DilateBlock.forward on NCHW x with the per-block cpe conv (the model's default, dilateformer.py:364)
    "dilateblock_b2_c72_h3_14x14_cpe": dict(variant="dilate_block", ctor=dict(dim=72, num_heads=3, qkv_bias=True, cpe_per_block=True),
                                            x=(2, 72, 14, 14)),
}

REF_CLASS = {"msda": "MultiDilatelocalAttention", "dilate_block_half": "DilateBlock", "dilate_block": "DilateBlock"}


def gather_windows(t, kernel_size, dilation):
    """t [..., H, W, d] -> [..., H, W, k*k, d]: entry (y, x, i*k + j) is t[y + i*dil - p, x + j*dil - p] with p = dil*(k-1)//2,
    zero outside the map (nn.Unfold's zero padding, dilateformer.py:48)."""
    H, W = t.shape[-3], t.shape[-2]
    k, dil = kernel_size, dilation
    p = dil * (k - 1) // 2
    tp = F.pad(t, (0, 0, p, p, p, p))
    return torch.stack([tp[..., i * dil:i * dil + H, j * dil:j * dil + W, :] for i in range(k) for j in range(k)], dim=-2)


def dilate_attention_core(qkv, num_heads, kernel_size, dilation, scale):
    """The attention between the two projections.  qkv [B, H, W, 3C] with column s*C + g*Cg + h*hd + d (dilateformer.py:88);
    returns O [B, H, W, C] with column g*Cg + h*hd + d (dilateformer.py:90-94)."""
    B, H, W, C3 = qkv.shape
    C = C3 // 3
    nd = len(dilation)
    hg, hd = num_heads // nd, C // num_heads
    t = qkv.reshape(B, H, W, 3, nd, hg, hd)
    out = torch.empty(B, H, W, nd, hg, hd, dtype=qkv.dtype)
    for g in range(nd):
        q, k, v = (t[:, :, :, s, g].permute(0, 3, 1, 2, 4) for s in range(3))       # [B, hg, H, W, hd]
        kw = gather_windows(k, kernel_size, dilation[g])
        vw = gather_windows(v, kernel_size, dilation[g])
        s = torch.einsum("bhyxd,bhyxnd->bhyxn", q, kw) * scale                     # a padded key's logit is exactly 0
        o = torch.einsum("bhyxn,bhyxnd->bhyxd", _softmax_last(s), vw)
        out[:, :, :, g] = o.permute(0, 2, 3, 1, 4)
    return out.reshape(B, H, W, C)


def dilate_attention(x, qkv_weight, qkv_bias, proj_weight, proj_bias, num_heads, kernel_size=3, dilation=(1, 2, 3), scale=None):
    """MultiDilatelocalAttention.forward (dilateformer.py:85-97) on x [B, H, W, C]; qkv_weight [3C, C] or [3C, C, 1, 1]."""
    C = x.shape[-1]
    scale = scale or (C // num_heads) ** -0.5
    qkv = _lin(x, qkv_weight.reshape(3 * C, C), qkv_bias)
    return _lin(dilate_attention_core(qkv, num_heads, kernel_size, dilation, scale), proj_weight, proj_bias)


def dilate_block_attention_half(x, norm1_weight, norm1_bias, eps=1e-5, **attn_kw):
    """x + attn(norm1(x)) on channels-last x (dilateformer.py:130); attn_kw = dilate_attention's parameters."""
    return x + dilate_attention(_layer_norm_rows(x, norm1_weight, norm1_bias, eps), **attn_kw)


def dilate_block_forward(x, P, num_heads, kernel_size=3, dilation=(1, 2, 3), scale=None, eps=1e-5):
    """DilateBlock.forward (dilateformer.py:126-134) on NCHW x, eval mode, GELU MLP; P = the block's state_dict."""
    if "pos_embed.weight" in P:
        x = x + _dwconv_same(x, P["pos_embed.weight"], P["pos_embed.bias"], 3)
    h = x.permute(0, 2, 3, 1)
    h = dilate_block_attention_half(h, P["norm1.weight"], P["norm1.bias"], eps, qkv_weight=P["attn.qkv.weight"],
                                    qkv_bias=P.get("attn.qkv.bias"), proj_weight=P["attn.proj.weight"],
                                    proj_bias=P["attn.proj.bias"], num_heads=num_heads, kernel_size=kernel_size,
                                    dilation=dilation, scale=scale)
    m = _lin(F.gelu(_lin(_layer_norm_rows(h, P["norm2.weight"], P["norm2.bias"], eps), P["mlp.fc1.weight"], P["mlp.fc1.bias"])),
             P["mlp.fc2.weight"], P["mlp.fc2.bias"])
    return (h + m).permute(0, 3, 1, 2)


def run_case(spec, inputs, params, dtype=torch.float32):
    """Evaluate the restatement for a DILATE_CASES spec; params = the reference state_dict."""
    c = spec["ctor"]
    P = {k: t.to(dtype) for k, t in params.items()}
    x = inputs["x"].to(dtype)
    kw = dict(num_heads=c["num_heads"], kernel_size=c.get("kernel_size", 3), dilation=c.get("dilation", [1, 2, 3]),
              scale=c.get("qk_scale"))
    if spec["variant"] == "msda":
        return dilate_attention(x, P["qkv.weight"], P.get("qkv.bias"), P["proj.weight"], P["proj.bias"], **kw)
    if spec["variant"] == "dilate_block_half":
        return dilate_block_attention_half(x, P["norm1.weight"], P["norm1.bias"], qkv_weight=P["attn.qkv.weight"],
                                           qkv_bias=P.get("attn.qkv.bias"), proj_weight=P["attn.proj.weight"],
                                           proj_bias=P["attn.proj.bias"], **kw)
    if spec["variant"] == "dilate_block":
        return dilate_block_forward(x, P, **kw)
    raise KeyError(spec["variant"])


def reference_forward(spec, mod, x):
    """The reference module on a CLONE of x: MultiDilatelocalAttention.forward writes into a contiguous input
    (dilateformer.py:90-93), which would overwrite the stored input."""
    x = x.clone()
    with torch.no_grad():
        if spec["variant"] == "dilate_block_half":
            return x + mod.attn(mod.norm1(x))
        return mod(x)
