"""Case definitions shared by the golden generator and the tests (TEST ORACLE).

A *spec* is a plain dict: {"variant", "ctor": {...}, "x": shape tuple, extra}.
``params`` are always ``state_dict`` tensors keyed by the reference's own keys.
"""
from __future__ import annotations

import importlib
import math
import sys

import numpy as np
import torch

from . import attention as A

GOLDEN_CASES = {
    # ViT.Attention(dim, num_heads, qkv_bias)            ViT.py:67-89
    "vit_b2_n197_c128_h2": dict(variant="vit", ctor=dict(dim=128, num_heads=2), x=(2, 197, 128)),
    "vit_b3_n50_c192_h3_bias": dict(variant="vit", ctor=dict(dim=192, num_heads=3, qkv_bias=True), x=(3, 50, 192)),
    # 192-wide heads (the reference's default ViT.Attention(num_heads=4) at dim 768 has them; here at dim 384 to keep the file small)
    "vit_b2_n197_c384_h2_hd192": dict(variant="vit", ctor=dict(dim=384, num_heads=2), x=(2, 197, 384)),
    # ViT.TransformerEncoder, attention half: x + attn(layernorm1(x))      ViT.py:105-116
    "vitblock_b2_n197_c128_h2": dict(variant="vit_block", ctor=dict(dim=128, num_heads=2), x=(2, 197, 128)),
    # setr.Attention(dim, num_heads=8) setr.py:50-72 and moat.Attention(dim, num_heads=8) moat.py:62-84: ViT's math
    "setr_b2_n100_c256_default_heads": dict(variant="setr", ctor=dict(dim=256), x=(2, 100, 256)),
    "moat_b2_n196_c512_default_heads_bias": dict(variant="moat", ctor=dict(dim=512, qkv_bias=True), x=(2, 196, 512)),
    # bvit.Broad_Attention(dim, heads, dim_head): inner width != dim, (out, q, k, v) returned     bvit.py:49-76
    "bvit_b2_n65_c192_h3_hd64": dict(variant="bvit", ctor=dict(dim=192, heads=3, dim_head=64), x=(2, 65, 192)),
    "bvit_b2_n50_c96_h4_hd32": dict(variant="bvit", ctor=dict(dim=96, heads=4, dim_head=32), x=(2, 50, 96)),
    # dilateformer.GlobalAttention(dim, num_heads=8): ViT's math on [B, H, W, C]          dilateformer.py:136-164
    "dilateformer_b2_12x12_c128_h2": dict(variant="dilateformer", ctor=dict(dim=128, num_heads=2, qkv_bias=True), x=(2, 12, 12, 128)),
    # p2t.PoolingAttention(dim, num_heads, pool_ratios).forward(x, H, W, d_convs): keys / values from a pooling pyramid   p2t.py:46-94
    "p2t_b2_14x14_c128_h2": dict(variant="p2t", ctor=dict(dim=128, num_heads=2, qkv_bias=True, pool_ratios=[1, 2, 3, 6]), x=(2, 196, 128), hw=(14, 14)),
    "p2t_b2_12x20_c64_h1_ratios_3_4_5": dict(variant="p2t", ctor=dict(dim=64, num_heads=1, pool_ratios=[3, 4, 5]), x=(2, 240, 64), hw=(12, 20)),
    # kvt.KNNAttention(dim, num_heads, topk): only the topk largest scores of a row enter the softmax      kvt.py:67-94
    "kvt_b2_n197_c128_h2_top100": dict(variant="kvt", ctor=dict(dim=128, num_heads=2, qkv_bias=True, topk=100), x=(2, 197, 128)),
    "kvt_b2_n50_c64_h1_top7": dict(variant="kvt", ctor=dict(dim=64, num_heads=1, topk=7), x=(2, 50, 64)),
    # pvt.Attention(dim, num_heads, sr_ratio)            pvt.py:52-91
    "pvt_b2_16x16_c128_h2_sr4": dict(variant="pvt", ctor=dict(dim=128, num_heads=2, sr_ratio=4), x=(2, 256, 128), hw=(16, 16)),
    "pvt_b2_8x8_c128_h2_sr1_bias": dict(variant="pvt", ctor=dict(dim=128, num_heads=2, sr_ratio=1, qkv_bias=True), x=(2, 64, 128), hw=(8, 8)),
    # pvt.Block, attention half: x + attn(norm1(x), H, W)   pvt.py:93-106
    "pvtblock_b2_16x16_c128_h2_sr4": dict(variant="pvt_block", ctor=dict(dim=128, num_heads=2, sr_ratio=4), x=(2, 256, 128), hw=(16, 16),
                                         keep=("norm1.", "attn.")),
    # segformer.Attention(dim, num_heads, qkv_bias, ..., sr_ratio): dense reduction conv, fused kv    segformer.py:17-50
    "segformer_b2_16x16_c64_h2_sr4_bias": dict(variant="segformer", ctor=dict(dim=64, num_heads=2, qkv_bias=True, sr_ratio=4), x=(2, 256, 64), hw=(16, 16)),
    "segformer_b2_16x16_c160_h5_sr2": dict(variant="segformer", ctor=dict(dim=160, num_heads=5, sr_ratio=2), x=(2, 256, 160), hw=(16, 16)),
    "segformer_b2_8x8_c128_h2_sr1": dict(variant="segformer", ctor=dict(dim=128, num_heads=2, sr_ratio=1), x=(2, 64, 128), hw=(8, 8)),
    # cmt.Attention(dim, num_heads, sr_ratio).forward(x, H, W, relative_pos)          cmt.py:72-111
    "cmt_b2_14x14_c64_h1_sr2": dict(variant="cmt", ctor=dict(dim=64, num_heads=1, sr_ratio=2), x=(2, 196, 64), hw=(14, 14)),
    "cmt_b2_16x16_c128_h2_sr2_bias": dict(variant="cmt", ctor=dict(dim=128, num_heads=2, sr_ratio=2, qkv_bias=True), x=(2, 256, 128), hw=(16, 16)),
    # cvt.Attention(dim, num_heads, ks)                   cvt.py:48-76
    "cvt_b2_c128_h2_14x14": dict(variant="cvt", ctor=dict(dim=128, num_heads=2), x=(2, 128, 14, 14)),
    # cswin.LePEAttention(dim, resolution, idx, split_size, num_heads)   cswin.py:51-127
    "lepe_b2_c64_h2_r14_idx0": dict(variant="lepe", ctor=dict(dim=64, resolution=14, idx=0, split_size=7, num_heads=2), x=(3, 2, 196, 64)),
    "lepe_b2_c64_h2_r14_idx1": dict(variant="lepe", ctor=dict(dim=64, resolution=14, idx=1, split_size=7, num_heads=2), x=(3, 2, 196, 64)),
    "lepe_b2_c64_h2_r7_idxm1": dict(variant="lepe", ctor=dict(dim=64, resolution=7, idx=-1, split_size=7, num_heads=2), x=(3, 2, 49, 64)),
    # cswin.CSWinBlock attention half                      cswin.py:130-194
    "cswinblk_b2_c128_r14_h4": dict(variant="cswin_block", ctor=dict(dim=128, reso=14, num_heads=4, split_size=7, qkv_bias=True), x=(2, 196, 128)),
    "cswinblk_b2_c128_r7_h4_last": dict(variant="cswin_block", ctor=dict(dim=128, reso=7, num_heads=4, split_size=7, qkv_bias=True, last_stage=True), x=(2, 49, 128)),
    # xcit.XCA / xcit.ClassAttention                       xcit.py:233-265, 159-188
    "xca_b2_n196_c128_h2": dict(variant="xca", ctor=dict(dim=128, num_heads=2, qkv_bias=True), x=(2, 196, 128)),
    "classattn_b2_n197_c128_h2": dict(variant="class_attn", ctor=dict(dim=128, num_heads=2, qkv_bias=True), x=(2, 197, 128)),
    # dual_attention.PAM(dim): NCHW, one head as wide as the channel count, no scale, alpha * y + x   dual_attention.py:12-28
    "pam_b2_c64_16x16": dict(variant="pam", ctor=dict(dim=64), x=(2, 64, 16, 16)),
    "pam_b2_c96_12x20": dict(variant="pam", ctor=dict(dim=96), x=(2, 96, 12, 20)),
    # xcit.XCABlock, attention half: x + gamma1 * attn(norm1(x))          xcit.py:267-291
    "xcablock_b2_n196_c128_h2": dict(variant="xca_block", ctor=dict(dim=128, num_heads=2, qkv_bias=True, eta=1.0), x=(2, 196, 128),
                                     keep=("norm1.", "attn.", "gamma1")),
}

EXTRA_SPECS = {
    # configurations of the GPU oracle cases that have no golden file of their own: tests/golden/reference/fresh_seeds.npz holds the
    # reference's outputs for them, so those GPU cases are pinned through it
    "xca_nano_hd32": dict(variant="xca", ctor=dict(dim=128, num_heads=4), x=(3, 196, 128)),
    "classattn_nano_hd32": dict(variant="class_attn", ctor=dict(dim=128, num_heads=4), x=(3, 197, 128)),
    "vit_l_like": dict(variant="vit", ctor=dict(dim=256, num_heads=4), x=(2, 197, 256)),
}

# bvit.Broad_Attention configurations whose four outputs (out, q, k, v) are recorded: inner width != dim, and heads == 1 with
# dim_head == dim, where there is no output projection (bvit.py:52, 61-64)
BVIT_QKV_CTORS = [dict(dim=192, heads=3, dim_head=64), dict(dim=64, heads=1, dim_head=64)]

SAMPLE = 512        # elements of each recorded reference output kept in tests/golden/reference/fresh_seeds.npz

_REF_CLASS = {
    "vit": ("ViT", "Attention"),
    "vit_block": ("ViT", "TransformerEncoder"),
    "setr": ("setr", "Attention"),
    "moat": ("moat", "Attention"),
    "bvit": ("bvit", "Broad_Attention"),
    "dilateformer": ("dilateformer", "GlobalAttention"),
    "p2t": ("p2t", "PoolingAttention"),
    "kvt": ("kvt", "KNNAttention"),
    "pvt": ("pvt", "Attention"),
    "pvt_block": ("pvt", "Block"),
    "segformer": ("segformer", "Attention"),
    "cmt": ("cmt", "Attention"),
    "xca_block": ("xcit", "XCABlock"),
    "pam": ("dual_attention", "PAM"),
    "cvt": ("cvt", "Attention"),
    "lepe": ("cswin", "LePEAttention"),
    "cswin_block": ("cswin", "CSWinBlock"),
    "xca": ("xcit", "XCA"),
    "class_attn": ("xcit", "ClassAttention"),
}


def round_fp16_(t):
    """Round a float tensor in place to fp16-representable values."""
    if t.is_floating_point():
        t.copy_(t.half().float())
    return t


def randomise_module_(mod, seed):
    """Randomise BN stats/affine, LayerNorm affine and XCA temperature (SURVEY.md §8d):
    a freshly constructed BN is ~identity and would hide bugs."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, m in mod.named_modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g))
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) * 1.5 + 0.5)
                m.weight.copy_(torch.randn(m.weight.shape, generator=g))
                m.bias.copy_(torch.randn(m.bias.shape, generator=g))
            if isinstance(m, torch.nn.LayerNorm):
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
        for name, p in mod.named_parameters():
            if name.endswith("temperature"):
                p.copy_(torch.rand(p.shape, generator=g) * 1.5 + 0.5)
            if name.endswith("alpha"):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)       # PAM: alpha = 0 at init would hide the whole attention term
            if name.endswith("gamma1"):
                p.copy_((torch.rand(p.shape, generator=g) + 0.5) * p)   # LayerScale (xcit.py:285) = eta * ones: spread it so a dropped gamma shows
            if name.endswith(".bias") and "norm" not in name and "sr.1" not in name and "qkv.1" not in name:
                # default Linear/Conv biases are tiny; widen them a bit so a dropped bias is visible
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
        for p in mod.parameters():
            round_fp16_(p)
        for b in mod.buffers():
            round_fp16_(b)
    return mod


def make_inputs(spec, seed=0):
    g = torch.Generator().manual_seed(1000 + seed)
    x = torch.randn(spec["x"], generator=g)
    out = {"x": round_fp16_(x)}
    if spec["variant"] == "cmt":
        # the model's relative_pos parameter, [heads, N, N / sr^2] (cmt.py:169-180; zeros at init -- random here)
        c = spec["ctor"]
        N = spec["x"][1]
        M = N // (c.get("sr_ratio", 1) ** 2)
        out["relative_pos"] = round_fp16_(torch.randn(c["num_heads"], N, M, generator=g))
    if spec["variant"] == "p2t":
        # the model's d_convs (p2t.py: one depthwise 3x3 conv per pool ratio, owned by the stage and passed to every block)
        c = spec["ctor"]
        L_ = len(c["pool_ratios"])
        out["dconv_weight"] = round_fp16_(torch.randn(L_, c["dim"], 1, 3, 3, generator=g) / 3.0)
        out["dconv_bias"] = round_fp16_(torch.randn(L_, c["dim"], generator=g) * 0.05)
    return out


def shuffled_case(inputs, params, seed):
    """A fresh case drawn from a stored one: the elements of every floating tensor permuted by a seeded generator.  Each
    tensor keeps its values (BN variances stay positive, LayerNorm weights near one, all fp16-representable) at new places."""
    rng = np.random.default_rng(seed)

    def shuffle(group):
        out = {}
        for k in sorted(group):
            t = group[k]
            if t.is_floating_point():
                t = t.reshape(-1)[torch.from_numpy(rng.permutation(t.numel()))].reshape(t.shape)
            out[k] = t
        return out
    return shuffle(inputs), shuffle(params)


def synth_linear_params(shapes, seed):
    """Parameters for a module made of Linear layers (plus XCA's temperature), keyed and shaped like ``shapes``: weights
    uniform in +-1/sqrt(fan_in) as nn.Linear initialises them, biases N(0, 0.05^2), temperatures in [0.5, 2); fp16-rounded."""
    g = torch.Generator().manual_seed(2000 + seed)
    out = {}
    for k in sorted(shapes):
        shape = tuple(shapes[k])
        if k.endswith("temperature"):
            t = torch.rand(shape, generator=g) * 1.5 + 0.5
        elif len(shape) >= 2:
            t = (torch.rand(shape, generator=g) * 2 - 1) / math.sqrt(math.prod(shape[1:]))
        else:
            t = torch.randn(shape, generator=g) * 0.05
        out[k] = round_fp16_(t)
    return out


def sample_index(numel):
    """Flat indices of the elements of a recorded output that are stored: SAMPLE of them spread evenly over the tensor (all of
    them if it is smaller).  Plain integer arithmetic, so the same on every machine."""
    n = min(numel, SAMPLE)
    return np.arange(n, dtype=np.int64) * numel // n


def p2t_d_convs(inputs, device="cpu"):
    """nn.Conv2d(dim, dim, 3, 1, 1, groups=dim) modules holding a p2t case's d_conv tensors."""
    w, b = inputs["dconv_weight"].float(), inputs["dconv_bias"].float()
    convs = torch.nn.ModuleList()
    for i in range(w.shape[0]):
        m = torch.nn.Conv2d(w.shape[1], w.shape[1], 3, 1, 1, groups=w.shape[1])
        with torch.no_grad():
            m.weight.copy_(w[i]); m.bias.copy_(b[i])
        convs.append(m)
    return convs.to(device)


def load_reference(ref_path):
    if ref_path not in sys.path:
        sys.path.insert(0, ref_path)
    return {m: importlib.import_module(m) for m in ("ViT", "pvt", "cvt", "cswin", "xcit", "moat", "segformer", "cmt", "bvit", "p2t", "kvt")}


def load_reference_class(ref_path, module, cls):
    """The reference class object.  ``setr.py`` builds and runs a whole SETR model at import time (setr.py:131-134), so for
    that file only the module's imports and its own class definitions are executed -- still the reference's code, read
    from where it lies, just without the module-level demo."""
    if module == "dual_attention":           # the one class outside vision_transformers/: attention_mechanisms/dual_attention.py
        import os
        am = os.path.join(os.path.dirname(os.path.abspath(ref_path)), "attention_mechanisms")
        if am not in sys.path:
            sys.path.insert(0, am)
        return getattr(importlib.import_module(module), cls)
    if module not in ("setr", "dilateformer"):
        return getattr(load_reference(ref_path)[module], cls)
    # setr.py builds and runs a whole SETR model at import time (setr.py:131-134); dilateformer.py imports timm, which this
    # image does not have (dilateformer.py:19-20).  For those two files the module's imports (those that resolve) and its own
    # class / function definitions are executed one by one -- still the reference's code, read from where it lies.
    import ast
    import os
    src = open(os.path.join(ref_path, module + ".py")).read()
    tree = ast.parse(src)
    ns = {"__name__": "reference_" + module}
    for n in tree.body:
        if isinstance(n, (ast.Import, ast.ImportFrom, ast.ClassDef, ast.FunctionDef)):
            try:
                exec(compile(ast.Module(body=[n], type_ignores=[]), os.path.join(ref_path, module + ".py"), "exec"), ns)
            except (ImportError, NameError):
                if isinstance(n, ast.ClassDef) and n.name == cls:
                    raise
    return ns[cls]


def reference_forward(spec, mod, x, inputs=None):
    v = spec["variant"]
    with torch.no_grad():
        if v in ("pvt", "segformer"):
            return mod(x, *spec["hw"])
        if v == "cmt":
            return mod(x, *spec["hw"], inputs["relative_pos"])
        if v == "pvt_block":
            # attention half only (pvt.py:106), with the reference block's own sub-modules
            return x + mod.attn(mod.norm1(x), *spec["hw"])
        if v == "p2t":
            return mod(x, *spec["hw"], d_convs=p2t_d_convs(inputs))
        if v == "bvit":
            return mod(x)[0]           # (out, q, k, v): the golden file pins out; q/k/v are checked in tests/test_oracle_vs_reference.py
        if v == "xca_block":
            # first line of XCABlock.forward (xcit.py:291)
            return x + mod.gamma1 * mod.attn(mod.norm1(x))
        if v == "cswin_block":
            # attention half only (cswin.py:184-194): x + proj(attn(norm1(x)))
            return cswin_block_attention_half_reference(mod, x)
        if v == "vit_block":
            # attention half only (ViT.py:116), with the reference block's own sub-modules
            return x + mod.attn(mod.layernorm1(x))
        return mod(x)


def cswin_block_attention_half_reference(blk, x):
    """Runs the reference CSWinBlock's own sub-modules for lines cswin.py:181-194
    (everything before the MLP half)."""
    B, L, C = x.shape
    img = blk.norm1(x)
    qkv = blk.qkv(img).reshape(B, -1, 3, C).permute(2, 0, 1, 3)
    if blk.branch_num == 2:
        x1 = blk.attns[0](qkv[:, :, :, :C // 2])
        x2 = blk.attns[1](qkv[:, :, :, C // 2:])
        att = torch.cat([x1, x2], dim=2)
    else:
        att = blk.attns[0](qkv)
    return x + blk.proj(att)


def build_reference_case(spec, ref_path, seed=0):
    modname, clsname = _REF_CLASS[spec["variant"]]
    torch.manual_seed(seed)
    mod = load_reference_class(ref_path, modname, clsname)(**spec["ctor"]).eval()
    randomise_module_(mod, seed + 7)
    inputs = make_inputs(spec, seed)
    y = reference_forward(spec, mod, inputs["x"], inputs).float()
    keep = spec.get("keep")           # block cases: only the attention half's parameters are stored
    params = {k: v.detach().clone() for k, v in mod.state_dict().items() if keep is None or k.startswith(tuple(keep))}
    return {"inputs": inputs, "params": params, "y_ref": y, "module": mod}


def _kw(params, *keys):
    return {k.replace(".", "_"): params.get(k) for k in keys}


def run_oracle_case(spec, inputs, params, dtype=torch.float32):
    """Evaluate the oracle restatement for a spec.  params: reference state_dict."""
    v = spec["variant"]
    c = spec["ctor"]
    P = {k: (t.to(dtype) if t.is_floating_point() else t) for k, t in params.items()}
    x = inputs["x"].to(dtype)
    if v in ("vit", "setr", "moat"):
        # setr.py:62-72 and moat.py:74-84 restate ViT.py:79-89; their constructor default is 8 heads
        return A.vit_attention(x, P["qkv.weight"], P.get("qkv.bias"), P["proj.weight"], P["proj.bias"],
                               c.get("num_heads", 4 if v == "vit" else 8))
    if v == "vit_block":
        return A.vit_block_attention_half(x, P["layernorm1.weight"], P["layernorm1.bias"], P["attn.qkv.weight"],
                                          P.get("attn.qkv.bias"), P["attn.proj.weight"], P["attn.proj.bias"],
                                          c.get("num_heads", 4))
    if v == "pvt":
        kw = _kw(P, "q.weight", "q.bias", "k.weight", "k.bias", "v.weight", "v.bias", "proj.weight", "proj.bias",
                 "sr.0.weight", "sr.0.bias", "sr.1.weight", "sr.1.bias", "sr.1.running_mean", "sr.1.running_var")
        return A.pvt_attention(x, spec["hw"][0], spec["hw"][1], num_heads=c["num_heads"],
                               sr_ratio=c.get("sr_ratio", 1), **kw)
    if v == "p2t":
        L_ = len(c["pool_ratios"])
        dw, db = inputs["dconv_weight"].to(dtype), inputs["dconv_bias"].to(dtype)
        return A.p2t_pooling_attention(x, spec["hw"][0], spec["hw"][1], P["q.0.weight"], P.get("q.0.bias"), P["kv.0.weight"],
                                       P.get("kv.0.bias"), P["proj.weight"], P["proj.bias"], P["norm.weight"], P["norm.bias"],
                                       c["num_heads"], c["pool_ratios"], [dw[i] for i in range(L_)], [db[i] for i in range(L_)],
                                       c.get("qk_scale"))
    if v == "dilateformer":
        # dilateformer.py:151-162: ViT.Attention over the H * W positions of a channels-last image
        B_, H_, W_, C_ = x.shape
        scale = c.get("qk_scale") or None
        return A.vit_attention(x.reshape(B_, H_ * W_, C_), P["qkv.weight"], P.get("qkv.bias"), P["proj.weight"], P["proj.bias"],
                               c.get("num_heads", 8), scale).reshape(B_, H_, W_, C_)
    if v == "kvt":
        return A.kvt_knn_attention(x, P["qkv.weight"], P.get("qkv.bias"), P["proj.weight"], P["proj.bias"],
                                   c.get("num_heads", 4), c.get("topk", 100))
    if v == "pam":
        return A.pam_attention(x, P["b.weight"], P["b.bias"], P["c.weight"], P["c.bias"], P["d.weight"], P["d.bias"], P["alpha"])
    if v == "bvit":
        return A.bvit_broad_attention(x, P["to_qkv.weight"], P.get("to_out.0.weight"), P.get("to_out.0.bias"),
                                      c.get("heads", 8), c.get("dim_head", 64))[0]
    if v == "pvt_block":
        keys = ("q.weight", "q.bias", "k.weight", "k.bias", "v.weight", "v.bias", "proj.weight", "proj.bias",
                "sr.0.weight", "sr.0.bias", "sr.1.weight", "sr.1.bias", "sr.1.running_mean", "sr.1.running_var")
        kw = {k.replace(".", "_"): P.get("attn." + k) for k in keys}
        return A.pvt_block_attention_half(x, spec["hw"][0], spec["hw"][1], P["norm1.weight"], P["norm1.bias"],
                                          num_heads=c["num_heads"], sr_ratio=c.get("sr_ratio", 1), **kw)
    if v == "cmt":
        kw = _kw(P, "q.weight", "q.bias", "k.weight", "k.bias", "v.weight", "v.bias", "proj.weight", "proj.bias",
                 "sr.0.weight", "sr.0.bias", "sr.1.weight", "sr.1.bias", "sr.1.running_mean", "sr.1.running_var")
        return A.pvt_attention(x, spec["hw"][0], spec["hw"][1], num_heads=c["num_heads"], sr_ratio=c.get("sr_ratio", 1),
                               relative_pos=inputs["relative_pos"].to(dtype), **kw)
    if v == "segformer":
        return A.segformer_attention(x, spec["hw"][0], spec["hw"][1], P["q.weight"], P.get("q.bias"), P["kv.weight"], P.get("kv.bias"),
                                     P["proj.weight"], P["proj.bias"], c["num_heads"], c.get("sr_ratio", 1),
                                     P.get("sr.weight"), P.get("sr.bias"))
    if v == "xca_block":
        return A.xca_block_attention_half(x, P["norm1.weight"], P["norm1.bias"], P["gamma1"], P["attn.qkv.weight"],
                                          P.get("attn.qkv.bias"), P["attn.proj.weight"], P["attn.proj.bias"],
                                          P["attn.temperature"], c["num_heads"], eps=1e-5)
    if v == "cvt":
        kw = _kw(P, "conv_proj_qkv.0.weight", "conv_proj_qkv.0.bias", "conv_proj_qkv.1.weight",
                 "conv_proj_qkv.1.bias", "conv_proj_qkv.1.running_mean", "conv_proj_qkv.1.running_var",
                 "conv_proj_qkv.2.weight", "conv_proj_qkv.2.bias", "proj.weight", "proj.bias")
        return A.cvt_attention(x, num_heads=c["num_heads"], ks=c.get("ks", 3), **kw)
    if v == "lepe":
        return A.cswin_lepe_attention(x, P["get_v.weight"], P["get_v.bias"], c["resolution"], c["idx"],
                                      c.get("split_size", 7), c["num_heads"], c.get("qk_scale"))
    if v == "cswin_block":
        nb = 1 if (c.get("last_stage", False) or c["reso"] == c.get("split_size", 7)) else 2
        return A.cswin_block_attention(
            x, P["norm1.weight"], P["norm1.bias"], P["qkv.weight"], P.get("qkv.bias"),
            P["proj.weight"], P["proj.bias"],
            [P[f"attns.{i}.get_v.weight"] for i in range(nb)], [P[f"attns.{i}.get_v.bias"] for i in range(nb)],
            c["reso"], c["num_heads"], c.get("split_size", 7), c.get("last_stage", False), c.get("qk_scale"))
    if v == "xca":
        return A.xca_attention(x, P["qkv.weight"], P.get("qkv.bias"), P["proj.weight"], P["proj.bias"],
                               P["temperature"], c["num_heads"])
    if v == "class_attn":
        return A.class_attention(x, P["qkv.weight"], P.get("qkv.bias"), P["proj.weight"], P["proj.bias"],
                                 c["num_heads"], c.get("qk_scale"))
    raise KeyError(v)
