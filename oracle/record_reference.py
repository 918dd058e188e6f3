#!/usr/bin/env python
"""Record, from the LIVE reference, what the reference-comparison tests check against, so that they run anywhere.

Run:  python oracle/record_reference.py        (needs the reference checkout, PA_REFERENCE=<path>/vision_transformers)
Writes three fixtures under tests/golden/reference/:
  * fresh_seeds.npz       -- reference outputs on cases other than the seed-0 golden files: every golden case re-drawn
                             with seeds 1 and 2 (oracle.cases.shuffled_case), three configurations without a golden file
                             and Broad_Attention's four outputs (parameters from oracle.cases.synth_linear_params).  Each
                             output is stored as SAMPLE evenly spread elements (oracle.cases.sample_index) plus max|y|;
  * cswin_windows.npz     -- the reference's img2windows / windows2img applied to index images;
  * reference_contract.json -- constructor / forward signatures and state_dict shapes of the reference classes, and the
                             constructor calls the reference's model factories make to the classes the drop-ins replace.
The oracle is checked against every recorded output here before anything is written.
"""
from __future__ import annotations

import functools
import importlib
import inspect
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
REF = os.environ.get("PA_REFERENCE", "")

from oracle.cases import (GOLDEN_CASES, EXTRA_SPECS, BVIT_QKV_CTORS, SAMPLE, load_reference, load_reference_class,  # noqa: E402
                          make_inputs, reference_forward, round_fp16_, run_oracle_case, sample_index, shuffled_case,
                          synth_linear_params, _REF_CLASS)
from oracle import attention as A  # noqa: E402
from _util import load_golden  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference")


def _check(name, y_or, y_ref):
    tol = 5e-6 * max(1.0, y_ref.abs().max().item())
    err = (y_or - y_ref).abs().max().item()
    print(f"{name:44s} out{tuple(y_ref.shape)} oracle-vs-reference max-abs={err:.3e}")
    assert err <= tol, name


def _store(blob, key, y):
    idx = sample_index(y.numel())
    blob[key + ".y"] = y.reshape(-1)[torch.from_numpy(idx)].numpy().astype(np.float32)
    blob[key + ".shape"] = np.array(y.shape, dtype=np.int64)
    blob[key + ".ymax"] = np.float32(y.abs().max().item())


def _reference_module(spec, params):
    modname, clsname = _REF_CLASS[spec["variant"]]
    mod = load_reference_class(REF, modname, clsname)(**spec["ctor"]).eval()
    res = mod.load_state_dict(params, strict=spec.get("keep") is None)
    assert not res.unexpected_keys and not [k for k in res.missing_keys if k.startswith(tuple(spec.get("keep", ())))]
    return mod


def _shapes(mod):
    return {k: list(v.shape) for k, v in mod.state_dict().items()}


def fresh_seeds():
    blob = {}
    for name, spec in sorted(GOLDEN_CASES.items()):
        inputs0, params0, _ = load_golden(name)
        for seed in (1, 2):
            inputs, params = shuffled_case(inputs0, params0, seed)
            y = reference_forward(spec, _reference_module(spec, params), inputs["x"], inputs).float()
            _check(f"{name} seed {seed}", run_oracle_case(spec, inputs, params), y)
            _store(blob, f"{name}.s{seed}", y)
    for name, spec in sorted(EXTRA_SPECS.items()):
        modname, clsname = _REF_CLASS[spec["variant"]]
        shapes = _shapes(load_reference_class(REF, modname, clsname)(**spec["ctor"]))
        params, inputs = synth_linear_params(shapes, 7), make_inputs(spec, 7)
        y = reference_forward(spec, _reference_module(spec, params), inputs["x"], inputs).float()
        _check(name, run_oracle_case(spec, inputs, params), y)
        _store(blob, name, y)
        blob[name + ".params"] = np.array(json.dumps(shapes))
    ref_cls = load_reference(REF)["bvit"].Broad_Attention
    for i, ctor in enumerate(BVIT_QKV_CTORS):
        mod = ref_cls(**ctor).eval()
        shapes = _shapes(mod)
        params = synth_linear_params(shapes, 3)
        mod.load_state_dict(params)
        x = round_fp16_(torch.randn(2, 37, ctor["dim"], generator=torch.Generator().manual_seed(3)))
        with torch.no_grad():
            ref = mod(x)
        got = A.bvit_broad_attention(x, params["to_qkv.weight"], params.get("to_out.0.weight"), params.get("to_out.0.bias"),
                                     ctor["heads"], ctor["dim_head"])
        key = f"bvit_qkv{i}"
        for j, (r, g) in enumerate(zip(ref, got)):
            _check(f"{key} output {j}", g, r)
            _store(blob, f"{key}.out{j}", r)
        blob[key + ".params"] = np.array(json.dumps(shapes))
    np.savez_compressed(os.path.join(OUT, "fresh_seeds.npz"), **blob)


WINDOW_CASES = [(14, 0, 7), (14, 1, 7), (7, -1, 7), (28, 0, 2)]


def cswin_windows():
    cswin = load_reference(REF)["cswin"]
    blob = {}
    for reso, idx, split in WINDOW_CASES:
        H_sp, W_sp = {(-1): (reso, reso), 0: (reso, split), 1: (split, reso)}[idx]
        img = torch.arange(reso * reso, dtype=torch.float32).reshape(1, 1, reso, reso)
        win = cswin.img2windows(img, H_sp, W_sp)[..., 0]
        back = cswin.windows2img(win.reshape(-1, H_sp, W_sp, 1), H_sp, W_sp, reso, reso)
        key = f"r{reso}_i{idx}_s{split}"
        blob[key + ".img2windows"] = win.long().numpy().astype(np.int32)
        blob[key + ".windows2img"] = back.reshape(-1).long().numpy().astype(np.int32)
    np.savez_compressed(os.path.join(OUT, "cswin_windows.npz"), **blob)


# ------------------------------------------------------------------------------------------------ reference_contract.json
def _encode(v):
    """Constructor arguments as JSON: classes (norm / activation layers) and functools.partial by qualified name."""
    if isinstance(v, functools.partial):
        return {"partial": _encode(v.func), "kwargs": {k: _encode(a) for k, a in v.keywords.items()}}
    if inspect.isclass(v):
        return {"class": v.__module__ + "." + v.__qualname__}
    if isinstance(v, (torch.Tensor, np.generic)):
        return v.item()
    if isinstance(v, (list, tuple)):
        return [_encode(a) for a in v]
    assert v is None or isinstance(v, (bool, int, float, str)), type(v)
    return v


def _sd(mod):
    return {k: [list(t.shape), str(t.dtype).replace("torch.", "")] for k, t in mod.state_dict().items()}


CONTRACT_CLASSES = [
    # (module, class, constructor kwargs whose state_dict is recorded)
    ("ViT", "Attention", dict(dim=192, num_heads=3, qkv_bias=True)),
    ("setr", "Attention", dict(dim=256, qkv_bias=True)),
    ("moat", "Attention", dict(dim=256, qkv_bias=True)),
    ("segformer", "Attention", dict(dim=64, num_heads=2, qkv_bias=True, sr_ratio=4)),
    ("cmt", "Attention", dict(dim=128, num_heads=2, sr_ratio=2, qkv_bias=True)),
    ("pvt", "Block", dict(dim=128, num_heads=2, sr_ratio=4)),
    ("xcit", "XCABlock", dict(dim=128, num_heads=4, qkv_bias=True, eta=1.0)),
    ("bvit", "Broad_Attention", dict(dim=192, heads=3, dim_head=64)),
    ("bvit", "Broad_Attention", dict(dim=64, heads=1, dim_head=64)),
    ("dual_attention", "PAM", dict(dim=64)),
    ("dilateformer", "GlobalAttention", dict(dim=128, num_heads=2, qkv_bias=True)),
    ("p2t", "PoolingAttention", dict(dim=128, num_heads=2, qkv_bias=True)),
    ("kvt", "KNNAttention", dict(dim=128, num_heads=2, qkv_bias=True, topk=50)),
]


def contract_key(module, cls, kw):
    return f"{module}.{cls}(" + ", ".join(f"{k}={v!r}" for k, v in kw.items()) + ")"


def _record_calls(mod, names, monkey):
    """Swap classes `names` of reference module `mod` for subclasses that log their outermost constructor calls."""
    calls, depth = [], [0]
    for n in names:
        base = getattr(mod, n)

        def init(self, *a, __base=base, __n=n, **kw):
            depth[0] += 1
            try:
                __base.__init__(self, *a, **kw)
            finally:
                depth[0] -= 1
            if depth[0] == 0:
                calls.append((self, __n, a, kw))
        monkey.append((mod, n, base))
        setattr(mod, n, type(base.__name__, (base,), {"__init__": init}))
    return calls


def _model_record(modname, factory, names, ctor_kw=None):
    mod = importlib.import_module(modname)
    monkey = []
    calls = _record_calls(mod, names, monkey)
    try:
        torch.manual_seed(0)
        model = getattr(mod, factory)(**(ctor_kw or {}))
    finally:
        for m, n, base in monkey:
            setattr(m, n, base)
    path = {id(m): p for p, m in model.named_modules()}
    out = []
    for inst, n, a, kw in calls:
        out.append(dict(path=path[id(inst)], cls=n, args=_encode(list(a)), kwargs={k: _encode(v) for k, v in kw.items()},
                        replaced=sum(type(m).__name__ in names for m in inst.modules()), state_dict=_sd(inst)))
    assert out
    return dict(calls=out, state_dict=_sd(model))


def contract():
    load_reference(REF)
    doc = {"classes": {}, "models": {}}
    for module, cls, kw in CONTRACT_CLASSES:
        ref = load_reference_class(REF, module, cls)
        entry = doc["classes"].setdefault(f"{module}.{cls}", {
            "init": str(inspect.signature(ref.__init__)), "forward": str(inspect.signature(ref.forward)), "instances": {}})
        r = ref(**kw)
        inst = {"state_dict": _sd(r)}
        for attr in ("scale", "num_elements", "topk"):
            if hasattr(r, attr):
                inst[attr] = _encode(getattr(r, attr))
        if hasattr(r, "to_out"):
            inst["to_out_is_identity"] = isinstance(r.to_out, torch.nn.Identity)
        entry["instances"][contract_key(module, cls, kw)] = inst
    doc["classes"]["dilateformer.GlobalAttention"]["qk_scale_0.25"] = load_reference_class(
        REF, "dilateformer", "GlobalAttention")(128, 2, qk_scale=0.25).scale
    tiny = dict(image_size=64, patch_size=16, in_channels=3, depths=2, num_heads=2, embedding_dim=128, num_classes=10)
    doc["models"]["ViT.VisionTransformer(tiny):Attention"] = _model_record("ViT", "VisionTransformer", ["Attention"], tiny)
    doc["models"]["ViT.VisionTransformer(tiny):TransformerEncoder"] = _model_record("ViT", "VisionTransformer",
                                                                                   ["TransformerEncoder"], tiny)
    doc["models"]["ViT.VisionTransformer():Attention"] = _model_record("ViT", "VisionTransformer", ["Attention"])
    for modname, factory, names in [("pvt", "pvt_t", ["Attention"]), ("cvt", "cvt_13", ["Attention"]),
                                    ("cswin", "CSWin_64_12211_tiny_224", ["LePEAttention", "CSWinBlock"]),
                                    ("xcit", "xcit_nano_12_p16", ["XCA", "ClassAttention"]), ("moat", "moat_0", ["Attention"])]:
        rec = _model_record(modname, factory, names)
        del rec["state_dict"]               # only the replaced sub-modules matter for the zoo models
        doc["models"][f"{modname}.{factory}()"] = rec
    del doc["models"]["ViT.VisionTransformer(tiny):Attention"]["state_dict"]
    del doc["models"]["ViT.VisionTransformer(tiny):TransformerEncoder"]["state_dict"]
    with open(os.path.join(OUT, "reference_contract.json"), "w") as f:
        json.dump(doc, f, indent=None, separators=(",", ":"), sort_keys=True)
        f.write("\n")


def main():
    if not os.path.isdir(REF):
        raise SystemExit("set PA_REFERENCE to the reference checkout's vision_transformers directory")
    fresh_seeds()
    cswin_windows()
    contract()
    print("wrote fresh_seeds.npz, cswin_windows.npz, reference_contract.json to", OUT)


if __name__ == "__main__":
    main()
