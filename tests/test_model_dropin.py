"""The drop-in attention inside a WHOLE reference model (SURVEY.md §8b "what calls it").

tests/golden/models/vit_tiny.npz holds the parameters, an input batch and the logits of the real reference
`ViT.VisionTransformer` (oracle/make_golden_model.py).  The model glue around the attention modules is restated in
oracle/model_glue.py, so the same model can be evaluated where /root/reference is absent:
  * CPU: glue + oracle attention reproduces the reference logits (pins the glue);
  * CPU: the drop-in class, built with the constructor arguments the reference's own model passes to the class it
    replaces (recorded in tests/golden/reference/reference_contract.json by oracle/record_reference.py), loads the reference
    state_dict strictly (constructor signature + keys), and refuses to run on CPU;
  * GPU: glue + B200 drop-in attention (fp16 I/O) against the reference logits.
"""
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from _util import GOLDEN_DIR, rel_fro

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import vit_attention  # noqa: E402
from oracle.model_glue import attention_state, vit_model_forward  # noqa: E402

CFG = dict(image_size=64, patch_size=16, in_channels=3, depths=2, num_heads=2, embedding_dim=128, num_classes=10)
with open(os.path.join(GOLDEN_DIR, "reference", "reference_contract.json")) as _f:
    MODELS = json.load(_f)["models"]


def _decode(v):
    """Constructor arguments as recorded (oracle/record_reference.py:_encode): classes and partials by qualified name."""
    if isinstance(v, list):
        return [_decode(a) for a in v]
    if isinstance(v, dict) and "class" in v:
        mod, _, name = v["class"].rpartition(".")
        return getattr(importlib.import_module(mod), name)
    if isinstance(v, dict) and "partial" in v:
        import functools
        return functools.partial(_decode(v["partial"]), **{k: _decode(a) for k, a in v["kwargs"].items()})
    return v


def _swap_in(record, swaps):
    """Build the drop-in for every recorded outermost constructor call the reference model made to a class in `swaps`, with
    the same arguments.  Checks that it replaces as many reference modules as the call built and that its state_dict has the
    reference sub-module's keys and shapes; returns [(path, drop-in)]."""
    built = []
    for call in record["calls"]:
        m = swaps[call["cls"]](*_decode(call["args"]), **{k: _decode(v) for k, v in call["kwargs"].items()})
        assert sum(isinstance(x, tuple(swaps.values())) for x in m.modules()) == call["replaced"] > 0
        assert {k: list(v.shape) for k, v in m.state_dict().items()} == {k: s for k, (s, _) in call["state_dict"].items()}
        built.append((call["path"], m))
    return built


def _sub_state(sd, path):
    return {k[len(path) + 1:]: v for k, v in sd.items() if k.startswith(path + ".")}


def _load():
    z = np.load(os.path.join(GOLDEN_DIR, "models", "vit_tiny.npz"))
    sd = {k[2:]: torch.from_numpy(z[k].astype(np.float32)) for k in z.files if k.startswith("p.")}
    return sd, torch.from_numpy(z["in.x"].astype(np.float32)), torch.from_numpy(z["y_ref"])


def test_glue_with_oracle_attention_reproduces_reference_model_logits():
    sd, x, y_ref = _load()

    def attn(i, t):
        a = attention_state(sd, i)
        return vit_attention(t, a["qkv.weight"], a.get("qkv.bias"), a["proj.weight"], a["proj.bias"], CFG["num_heads"])

    y = vit_model_forward(sd, x, attn, CFG["patch_size"], CFG["depths"])
    assert (y - y_ref).abs().max().item() <= 2e-5 * y_ref.abs().max().item()


@pytest.mark.parametrize("level", ["attention", "block"])
def test_class_swap_inside_the_reference_model_constructs_and_loads(level):
    import pytorch_attention_b200 as pa
    if level == "attention":
        swaps = {"Attention": pa.vit.Attention}                    # the substitution INTEGRATION.md describes
    else:
        swaps = {"TransformerEncoder": pa.vit.TransformerEncoder}  # whole block: LN + attention + residual fused
    # ViT.py:98 constructs the drop-in with the reference's arguments
    built = _swap_in(MODELS["ViT.VisionTransformer(tiny):" + next(iter(swaps))], swaps)
    assert [p for p, _ in built] == [f"blocks.{i}" + (".attn" if level == "attention" else "") for i in range(CFG["depths"])]
    sd, x, _ = _load()
    for path, m in built:
        assert isinstance(m if level == "attention" else m.attn, pa.vit.Attention)
        m.eval().load_state_dict(_sub_state(sd, path), strict=True)   # identical keys and shapes
        with pytest.raises(RuntimeError, match="CPU"):             # product path: no CPU fallback
            with torch.no_grad():
                m(torch.randn(2, 17, CFG["embedding_dim"]).half())


@pytest.mark.gpu
def test_dropin_attention_inside_the_whole_model_matches_reference_logits():
    import pytorch_attention_b200 as pa
    sd, x, y_ref = _load()
    dev = torch.device("cuda", 0)
    sdg = {k: v.to(dev) for k, v in sd.items()}
    mods = []
    for i in range(CFG["depths"]):
        m = pa.vit.Attention(CFG["embedding_dim"], CFG["num_heads"]).eval()
        m.load_state_dict(attention_state(sd, i), strict=True)
        mods.append(m.to(dev))

    def attn(i, t):
        return mods[i](t.half()).float()                           # LayerNorm output rounded once to the kernel's fp16 input

    with torch.no_grad():
        y = vit_model_forward(sdg, x.to(dev), attn, CFG["patch_size"], CFG["depths"]).cpu()
    # the path's own tolerance is 1e-3 per attention; two blocks, fp16-rounded attention inputs and the MLP/head amplify it
    assert rel_fro(y, y_ref) < 3e-3, rel_fro(y, y_ref)


def _swap_targets():
    import pytorch_attention_b200 as pa
    return {
        "pvt": ("pvt_t", {"Attention": pa.pvt.Attention}),
        "cvt": ("cvt_13", {"Attention": pa.cvt.Attention}),
        "cswin": ("CSWin_64_12211_tiny_224", {"LePEAttention": pa.cswin.LePEAttention, "CSWinBlock": pa.cswin.CSWinBlock}),
        "xcit": ("xcit_nano_12_p16", {"XCA": pa.xcit.XCA, "ClassAttention": pa.xcit.ClassAttention}),
        "moat": ("moat_0", {"Attention": pa.moat.Attention}),      # 48- and 96-wide heads (dims 384 / 768, 8 heads)
    }


@pytest.mark.parametrize("modname", ["pvt", "cvt", "cswin", "xcit", "moat"])
def test_class_swap_in_the_reference_zoo_models(modname):
    """The drop-ins accept the arguments the reference's own model constructors pass, replace as many modules as the stock
    model has, and hold the same state_dict keys and shapes -- for every model family on the path."""
    factory, swaps = _swap_targets()[modname]
    record = MODELS[f"{modname}.{factory}()"]
    assert {c["cls"] for c in record["calls"]} <= set(swaps)
    for call, (_, m) in zip(record["calls"], _swap_in(record, swaps)):
        m.load_state_dict({k: torch.zeros(s, dtype=getattr(torch, dt)) for k, (s, dt) in call["state_dict"].items()}, strict=True)


# ---------------------------------------------------------------- the reference's DEFAULT model: VisionTransformer()
def _load_default():
    from oracle.model_glue import vit_state_shapes, synth_state_dict
    z = np.load(os.path.join(GOLDEN_DIR, "models", "vit_default.npz"))
    seed = int(z["seed"])
    sd = synth_state_dict(vit_state_shapes(), seed)              # 86 M parameters rebuilt from the seed (only logits are stored)
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(seed)).half().float()
    return sd, x, torch.from_numpy(z["y_ref"])


def test_default_model_glue_with_oracle_attention_reproduces_reference_logits():
    """`VisionTransformer()` with every constructor default (12 blocks, dim 768, 4 heads of 192: README.md:331-334)."""
    sd, x, y_ref = _load_default()

    def attn(i, t):
        a = attention_state(sd, i)
        return vit_attention(t, a["qkv.weight"], a.get("qkv.bias"), a["proj.weight"], a["proj.bias"], 4)

    with torch.no_grad():
        y = vit_model_forward(sd, x, attn, 16, 12)
    assert (y - y_ref).abs().max().item() <= 5e-5 * y_ref.abs().max().item()


def test_default_reference_model_accepts_the_dropin_and_the_synthetic_state():
    import pytorch_attention_b200 as pa
    from oracle.model_glue import vit_state_shapes, synth_state_dict
    record = MODELS["ViT.VisionTransformer():Attention"]           # every default: 4 heads of 192
    shapes = vit_state_shapes()
    assert {k: list(s) for k, s in shapes.items()} == {k: s for k, (s, _) in record["state_dict"].items()}
    built = _swap_in(record, {"Attention": pa.vit.Attention})
    assert len(built) == 12 and all(m.num_heads == 4 for _, m in built)
    sd = synth_state_dict(shapes, 77)
    for path, m in built:
        m.load_state_dict(_sub_state(sd, path), strict=True)


@pytest.mark.gpu
def test_default_model_with_dropin_attention_matches_reference_logits():
    """The INTEGRATION.md §1 example at full size: the reference's default ViT (192-wide heads -> the panelled attention
    core) with the B200 drop-in in all 12 blocks, against the logits of the real reference model."""
    import pytorch_attention_b200 as pa
    sd, x, y_ref = _load_default()
    dev = torch.device("cuda", 0)
    sdg = {k: v.to(dev) for k, v in sd.items()}
    mods = []
    for i in range(12):
        m = pa.vit.Attention(768).eval()                            # constructor defaults, as ViT.py:111 builds it
        m.load_state_dict(attention_state(sd, i), strict=True)
        m = m.to(dev)
        m.fp32_input = torch.float16                                # fp32 model: opt-in cast, fp32 result
        mods.append(m)
    with torch.no_grad():
        y = vit_model_forward(sdg, x.to(dev), lambda i, t: mods[i](t), 16, 12).cpu()
    # 12 blocks of a 1e-3 path with fp16-rounded attention inputs, amplified by the MLPs and the head
    assert rel_fro(y, y_ref) < 1e-2, rel_fro(y, y_ref)
    assert (y.argmax(-1) == y_ref.argmax(-1)).all()
