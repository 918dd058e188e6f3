#!/usr/bin/env python
"""Generate tests/golden/dilate/ from the LIVE reference (vision_transformers/dilateformer.py).

Run:  PA_REFERENCE=<reference checkout>/vision_transformers python oracle/make_golden_dilate.py
dilateformer.py imports timm at the top, so its classes are loaded with ``load_reference_class`` (the module's own class and
function definitions executed one by one).  For every case of ``oracle.dilate.DILATE_CASES`` it
  1. builds the reference module, eval() mode, LayerNorm affine / biases randomised, everything rounded to fp16 values,
  2. runs the reference forward in fp32 on CPU on a clone of x (the reference writes into a contiguous x) -> ``y_ref``,
  3. checks the restatement of oracle/dilate.py against it (max-abs <= 5e-6 * max|y|),
  4. stores inputs (fp16), parameters (fp16) and y_ref (fp32) as <case>.npz.
It also writes contract.json: constructor / forward signatures, state_dict shapes and attributes of a few instances, and the
constructor's assertion message for a head count the groups do not divide.
"""
from __future__ import annotations

import inspect
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.environ.get("PA_REFERENCE", "/root/reference/vision_transformers")
OUT = os.path.join(ROOT, "tests", "golden", "dilate")

from oracle.cases import load_reference_class, make_inputs, randomise_module_  # noqa: E402
from oracle.dilate import DILATE_CASES, REF_CLASS, reference_forward, run_case  # noqa: E402

CONTRACT_INSTANCES = [
    ("MultiDilatelocalAttention", dict(dim=72, num_heads=3, qkv_bias=True)),
    ("MultiDilatelocalAttention", dict(dim=96, num_heads=6, qk_scale=0.25, kernel_size=5, dilation=[1, 3])),
    ("MultiDilatelocalAttention", dict(dim=64, num_heads=8, dilation=[1, 2])),
    ("DilateBlock", dict(dim=72, num_heads=3, qkv_bias=True, cpe_per_block=True)),
    ("DilateBlock", dict(dim=144, num_heads=6, mlp_ratio=2.0)),
]


def _sd(mod):
    return {k: [list(t.shape), str(t.dtype).replace("torch.", "")] for k, t in mod.state_dict().items()}


def goldens():
    for name, spec in DILATE_CASES.items():
        torch.manual_seed(0)
        mod = load_reference_class(REF, "dilateformer", REF_CLASS[spec["variant"]])(**spec["ctor"]).eval()
        randomise_module_(mod, 7)
        inputs = make_inputs(spec, 0)
        x_before = inputs["x"].clone()
        y_ref = reference_forward(spec, mod, inputs["x"]).float()
        assert torch.equal(inputs["x"], x_before)
        keep = spec.get("keep")
        params = {k: v.detach().clone() for k, v in mod.state_dict().items() if keep is None or k.startswith(tuple(keep))}
        y_or = run_case(spec, inputs, params)
        err = (y_or - y_ref).abs().max().item()
        mag = y_ref.abs().max().item()
        print(f"{name:36s} out{tuple(y_ref.shape)} max|y|={mag:.4f} oracle-vs-reference max-abs={err:.3e}")
        assert err <= 5e-6 * max(1.0, mag), f"oracle restatement disagrees with reference on {name}"
        blob = {"in." + k: v.numpy().astype(np.float16) for k, v in inputs.items()}
        blob.update({"p." + k: v.numpy().astype(np.float16) for k, v in params.items()})
        blob["y_ref"] = y_ref.numpy().astype(np.float32)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **blob)


def contract():
    doc = {"classes": {}, "instances": []}
    for cls in ("MultiDilatelocalAttention", "DilateBlock"):
        ref = load_reference_class(REF, "dilateformer", cls)
        doc["classes"][cls] = {"init": str(inspect.signature(ref.__init__)), "forward": str(inspect.signature(ref.forward))}
    for cls, kw in CONTRACT_INSTANCES:
        r = load_reference_class(REF, "dilateformer", cls)(**kw)
        a = r if cls == "MultiDilatelocalAttention" else r.attn
        doc["instances"].append(dict(cls=cls, kwargs=kw, state_dict=_sd(r), scale=a.scale, dilation=list(a.dilation),
                                     kernel_size=a.kernel_size, num_dilation=a.num_dilation,
                                     n_dilate_attention=len(a.dilate_attention)))
    bad = dict(dim=64, num_heads=4, dilation=[1, 2, 3])
    try:
        load_reference_class(REF, "dilateformer", "MultiDilatelocalAttention")(**bad)
    except AssertionError as e:
        doc["ctor_assert"] = dict(kwargs=bad, message=str(e))
    assert "ctor_assert" in doc, "expected the constructor to reject 4 heads over 3 dilation groups"
    with open(os.path.join(OUT, "contract.json"), "w") as f:
        json.dump(doc, f, indent=1, sort_keys=True)
        f.write("\n")


def main():
    if not os.path.isdir(REF):
        raise SystemExit(f"reference not found at {REF}; set PA_REFERENCE")
    os.makedirs(OUT, exist_ok=True)
    goldens()
    contract()
    print("wrote", len(DILATE_CASES), "golden files and contract.json to", OUT)


if __name__ == "__main__":
    main()
