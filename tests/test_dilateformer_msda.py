"""DilateFormer's multi-scale dilated attention: ``dilateformer.MultiDilatelocalAttention`` and ``DilateBlock``
(dilateformer.py:64-134).  CPU: the oracle against the reference's golden outputs, the module contract against the recorded
reference contract, C-ABI argument validation.  GPU: the drop-ins against the goldens and the oracle at the zoo's stage shapes,
the index path of the kernel alone, batch properties and CUDA-graph replay."""
import ctypes as C
import inspect
import json
import math
import os

import pytest
import torch

import pytorch_attention_b200 as pa
from oracle.cases import randomise_module_, round_fp16_
from oracle.dilate import DILATE_CASES, dilate_attention_core, dilate_block_forward, gather_windows, run_case
from pytorch_attention_b200 import _lib as L
from pytorch_attention_b200 import ops

from _util import GOLDEN_DIR, load_golden, rel_fro, rel_max

DILATE_DIR = os.path.join(GOLDEN_DIR, "dilate")
with open(os.path.join(DILATE_DIR, "contract.json")) as _f:
    CONTRACT = json.load(_f)
TOL = 1e-3
gpu = pytest.mark.gpu
CLASSES = {"MultiDilatelocalAttention": pa.dilateformer.MultiDilatelocalAttention, "DilateBlock": pa.dilateformer.DilateBlock}


def _dropin(spec):
    cls = pa.dilateformer.MultiDilatelocalAttention if spec["variant"] == "msda" else pa.dilateformer.DilateBlock
    return cls(**spec["ctor"]).eval()


def _load(m, spec, params):
    if spec.get("keep"):
        res = m.load_state_dict(params, strict=False)
        assert not res.unexpected_keys, res.unexpected_keys
        assert not [k for k in res.missing_keys if k.startswith(tuple(spec["keep"]))], res.missing_keys
    else:
        m.load_state_dict(params)                      # strict: keys and shapes must match the reference's
    return m


# ================================================================ CPU
def test_all_dilate_golden_cases_present():
    names = sorted(os.path.splitext(f)[0] for f in os.listdir(DILATE_DIR) if f.endswith(".npz"))
    assert names == sorted(DILATE_CASES)


@pytest.mark.parametrize("name", sorted(DILATE_CASES))
def test_oracle_vs_reference_golden(name):
    inputs, params, y_ref = load_golden(os.path.join("dilate", name))
    y = run_case(DILATE_CASES[name], inputs, params)
    assert y.shape == y_ref.shape
    assert (y - y_ref).abs().max().item() <= 5e-6 * max(1.0, y_ref.abs().max().item())


def test_oracle_padding_is_a_zero_key_not_a_masked_one():
    """One query on a 1 x 1 map with k = 3: its own key plus eight padded keys of logit 0 and value 0 (nn.Unfold's zeros)."""
    qkv = torch.tensor([[[[2.0, 1.0, 3.0]]]])                # C = 1: q = 2, k = 1, v = 3
    o = dilate_attention_core(qkv, 1, 3, [1], 1.0)
    e = math.exp(2.0)
    assert abs(o.item() - 3.0 * e / (e + 8.0)) < 1e-6


def test_module_contract_matches_reference():
    for cls, rec in CONTRACT["classes"].items():
        ours = CLASSES[cls]
        assert rec["init"] == str(inspect.signature(ours.__init__)), cls
        assert rec["forward"] == str(inspect.signature(ours.forward)), cls
    for inst in CONTRACT["instances"]:
        m = CLASSES[inst["cls"]](**inst["kwargs"])
        sd = {k: [list(t.shape), str(t.dtype).replace("torch.", "")] for k, t in m.state_dict().items()}
        assert sd == inst["state_dict"], inst["kwargs"]
        a = m if inst["cls"] == "MultiDilatelocalAttention" else m.attn
        assert a.scale == inst["scale"] and list(a.dilation) == inst["dilation"] and a.kernel_size == inst["kernel_size"]
        assert a.num_dilation == inst["num_dilation"] and len(a.dilate_attention) == inst["n_dilate_attention"]
        assert not list(a.dilate_attention.parameters())
        g = torch.Generator().manual_seed(0)
        ref_sd = {k: torch.randn(shape, generator=g) for k, (shape, _) in inst["state_dict"].items()}
        m.load_state_dict(ref_sd)                      # strict
    bad = CONTRACT["ctor_assert"]
    with pytest.raises(AssertionError, match=bad["message"].replace("!", r"\!")):
        pa.dilateformer.MultiDilatelocalAttention(**bad["kwargs"])


def _args(**kw):
    a = L.DilateArgs()
    a.B, a.Himg, a.Wimg, a.C, a.H, a.kernel_size, a.n_dilation, a.scale = 2, 56, 56, 72, 3, 3, 3, 24 ** -0.5
    a.dilation[0], a.dilation[1], a.dilation[2] = 1, 2, 3
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_abi_argument_validation_without_gpu():
    lib = L.load()
    ok = _args()
    assert lib.pa_dilate_workspace_bytes(C.byref(ok)) >= 2 * 56 * 56 * 72 * 2 * 4
    assert lib.pa_dilate_fwd(C.byref(ok), None, 0, None) == L.PA_ERR_NULL            # x / weights NULL
    assert lib.pa_dilate_fwd(None, None, 0, None) == L.PA_ERR_NULL
    assert lib.pa_dilate_core(C.byref(ok), None, None, None) == L.PA_ERR_NULL
    cases = [(dict(H=4), L.PA_ERR_BAD_SHAPE, b"num_dilation"),                        # dilateformer.py:77
             (dict(C=70), L.PA_ERR_BAD_SHAPE, b"divisible"),
             (dict(kernel_size=4), L.PA_ERR_BAD_SHAPE, b"odd"),                       # unfold output does not reshape
             (dict(kernel_size=9), L.PA_ERR_UNSUPPORTED, b"kernel_size"),
             (dict(C=36), L.PA_ERR_UNSUPPORTED, b"head_dim 12"),                      # not a multiple of 8
             (dict(C=216), L.PA_ERR_UNSUPPORTED, b"head_dim 72"),                     # above 64
             (dict(n_dilation=9, H=9, C=72 * 3), L.PA_ERR_UNSUPPORTED, b"groups"),
             (dict(n_dilation=0), L.PA_ERR_UNSUPPORTED, b"groups"),
             (dict(scale=0.0), L.PA_ERR_UNSUPPORTED, b"scale"),
             (dict(B=0), L.PA_ERR_BAD_SHAPE, b"positive")]
    for kw, code, msg in cases:
        a = _args(**kw)
        assert lib.pa_dilate_workspace_bytes(C.byref(a)) == 0, kw
        assert lib.pa_dilate_fwd(C.byref(a), None, 0, None) == code, kw
        assert msg in lib.pa_last_error(), (kw, lib.pa_last_error())
        assert lib.pa_dilate_core(C.byref(a), C.c_void_p(16), C.c_void_p(16), None) == code, kw
    a = _args()
    a.dilation[1] = 0
    assert lib.pa_dilate_fwd(C.byref(a), None, 0, None) == L.PA_ERR_BAD_SHAPE
    blk = L.DilateBlockArgs()
    assert lib.pa_dilate_block_attn_workspace_bytes(C.byref(blk)) == 0
    assert lib.pa_dilate_block_attn_fwd(None, None, 0, None) == L.PA_ERR_NULL
    blk.attn = _args()
    assert lib.pa_dilate_block_attn_workspace_bytes(C.byref(blk)) == \
        lib.pa_dilate_workspace_bytes(C.byref(ok)) + 2 * 56 * 56 * 72 * 2
    assert lib.pa_dilate_block_attn_fwd(C.byref(blk), None, 0, None) == L.PA_ERR_NULL


def _planned(a):
    """pa_dilate_fwd with non-NULL tensors and no workspace: PA_ERR_WORKSPACE means the shared-memory plan accepted the shape
    (it runs before the workspace check), PA_ERR_UNSUPPORTED that it did not.  Nothing is launched either way."""
    a.x = a.qkv_weight = a.proj_weight = a.y = 16
    return L.load().pa_dilate_fwd(C.byref(a), None, 0, None)


@pytest.mark.parametrize("kw,dil", [(dict(), [1, 2, 3]),
                                    (dict(), [1, 30, 56]),                              # tiny stage 1, dilations up to the map
                                    (dict(), [1, 22, 1 << 30]),                         # far beyond the map: all padding but the centre
                                    (dict(C=120, H=3), [13, 40, 100]),                  # Cg 40 (pitch 40)
                                    (dict(C=144, H=6, Himg=28, Wimg=28), [1, 2, 3]),    # tiny stage 2
                                    (dict(C=96, H=3, kernel_size=7), [5, 9, 56]),       # base stage 1 width, k = 7
                                    (dict(C=72, H=3, Wimg=807), [1, 2, 300]),           # the documented width bound at Cg 24
                                    (dict(C=96, H=3, Wimg=484), [2, 9, 500])])                  # ... and at Cg 32
def test_any_dilation_fits_the_plan_without_gpu(kw, dil):
    a = _args(**kw)
    for i, d in enumerate(dil):
        a.dilation[i] = d
    assert _planned(a) == L.PA_ERR_WORKSPACE, L.load().pa_last_error()


@pytest.mark.parametrize("kw", [dict(Wimg=808), dict(C=96, H=3, Wimg=485), dict(C=144, H=6, Wimg=346),
                                dict(Wimg=2000, C=512, H=8, n_dilation=1)])
def test_map_wider_than_the_documented_bound_is_unsupported_without_gpu(kw):
    a = _args(**kw)
    assert _planned(a) == L.PA_ERR_UNSUPPORTED
    assert b"map too wide" in L.load().pa_last_error()
    a.Wimg -= 1
    assert _planned(a) == (L.PA_ERR_WORKSPACE if kw.get("C") != 512 else L.PA_ERR_UNSUPPORTED)


def test_error_mapping_without_gpu():
    lib = L.load()
    with pytest.raises(AssertionError, match="odd"):
        L.check(lib.pa_dilate_fwd(C.byref(_args(kernel_size=2)), None, 0, None))
    with pytest.raises(ValueError, match="head_dim"):
        L.check(lib.pa_dilate_fwd(C.byref(_args(C=36)), None, 0, None))
    m = pa.dilateformer.MultiDilatelocalAttention(72, 3).eval()
    with pytest.raises(RuntimeError, match="CPU tensor"):
        m(torch.randn(1, 4, 4, 72).half())
    blk = pa.dilateformer.DilateBlock(72, 3, drop_path=0.1)
    with pytest.raises(RuntimeError, match="CPU tensor"):
        blk.eval()(torch.randn(1, 72, 4, 4).half())
    with pytest.raises(NotImplementedError):
        blk.train().drop_path(torch.zeros(2))
    assert torch.equal(blk.eval().drop_path(torch.ones(2)), torch.ones(2))


# ================================================================ GPU
def _seeded(spec, seed):
    torch.manual_seed(seed)
    m = _dropin(spec)
    randomise_module_(m, seed + 7)
    g = torch.Generator().manual_seed(1000 + seed)
    x = round_fp16_(torch.randn(spec["x"], generator=g))
    sd = {k: v.detach().float().clone() for k, v in m.state_dict().items()}
    return m, x, sd


@gpu
@pytest.mark.parametrize("name", sorted(DILATE_CASES))
def test_dropin_vs_reference_golden(name):
    spec = DILATE_CASES[name]
    inputs, params, y_ref = load_golden(os.path.join("dilate", name))
    m = _load(_dropin(spec), spec, params).cuda()
    x = inputs["x"].cuda()
    with torch.no_grad():
        if spec["variant"] == "dilate_block":
            m.fp32_input = torch.float16          # cpe conv and MLP half in fp32, attention half on fp16 activations
            y = m(x)
        elif spec["variant"] == "dilate_block_half":
            y = m.attention_half(x.half())
        else:
            m.out_dtype = torch.float32
            y = m(x.half())
    y = y.float().cpu()
    assert rel_fro(y, y_ref) < TOL and rel_max(y, y_ref) < TOL, (rel_fro(y, y_ref), rel_max(y, y_ref))


ZOO = {
    "tiny_stage1_56x56_c72_h3": dict(variant="msda", ctor=dict(dim=72, num_heads=3, qkv_bias=True), x=(2, 56, 56, 72)),
    "tiny_stage2_28x28_c144_h6": dict(variant="msda", ctor=dict(dim=144, num_heads=6, qkv_bias=True), x=(2, 28, 28, 144)),
    "base_stage1_56x56_c96_h3": dict(variant="msda", ctor=dict(dim=96, num_heads=3, qkv_bias=True), x=(2, 56, 56, 96)),
    "dil3_on_4x4_c48_h3": dict(variant="msda", ctor=dict(dim=48, num_heads=3), x=(3, 4, 4, 48)),
    # dilations beyond the contiguous halo: per-tap-row staging (dilation > band rows), one of them larger than the map
    "tiny_stage1_dil_1_30_64": dict(variant="msda", ctor=dict(dim=72, num_heads=3, qkv_bias=True, dilation=[1, 30, 64]),
                                    x=(2, 56, 56, 72)),
    "base_stage1_k7_dil_5_9_56": dict(variant="msda", ctor=dict(dim=96, num_heads=3, kernel_size=7, dilation=[5, 9, 56]),
                                      x=(1, 56, 56, 96)),
    "k7_d2_hd64_9x13": dict(variant="msda", ctor=dict(dim=128, num_heads=2, kernel_size=7, dilation=[2, 1], qk_scale=0.1),
                            x=(2, 9, 13, 128)),
    "block_half_tiny_stage2": dict(variant="dilate_block_half", ctor=dict(dim=144, num_heads=6, qkv_bias=True), x=(2, 28, 28, 144)),
}


@gpu
@pytest.mark.parametrize("name", sorted(ZOO))
def test_dropin_vs_oracle_at_stage_shapes(name):
    spec = ZOO[name]
    m, x, sd = _seeded(spec, 3)
    ref = run_case(spec, {"x": x}, sd)
    with torch.no_grad():
        m = m.cuda()
        y = m.attention_half(x.half().cuda()) if spec["variant"] == "dilate_block_half" else m(x.half().cuda())
    y = y.float().cpu()
    assert rel_fro(y, ref) < TOL and rel_max(y, ref) < TOL, (rel_fro(y, ref), rel_max(y, ref))


@gpu
def test_block_full_forward_in_an_fp32_model_and_a_16bit_model():
    """DilateBlock.forward = cpe conv + B200 attention half + the block's own PyTorch MLP half (dilateformer.py:126-134), against
    the oracle in fp32: works in a .half() model and, with fp32_input set, in an fp32 model; NCHW in and out."""
    spec = dict(variant="dilate_block", ctor=dict(dim=72, num_heads=3, qkv_bias=True, cpe_per_block=True), x=(2, 72, 28, 28))
    m, x, sd = _seeded(spec, 5)
    ref = dilate_block_forward(x, sd, 3)
    with torch.no_grad():
        m = m.cuda()
        m.fp32_input = torch.float16
        y32 = m(x.cuda())
        assert y32.dtype == torch.float32 and y32.shape == x.shape
        y16 = m.half()(x.half().cuda())
        assert y16.dtype == torch.float16
    assert rel_fro(y32.cpu(), ref) < 2e-3 and rel_fro(y16.float().cpu(), ref) < 3e-3


def _core(qkv, B, Hh, Ww, Cc, heads, k, dil, scale):
    a = _args(B=B, Himg=Hh, Wimg=Ww, C=Cc, H=heads, kernel_size=k, n_dilation=len(dil), scale=scale)
    for i, d in enumerate(dil):
        a.dilation[i] = d
    o = torch.empty(B * Hh * Ww, Cc, dtype=torch.float16, device=qkv.device)
    L.check(L.load().pa_dilate_core(C.byref(a), ops._ptr(qkv), ops._ptr(o), ops.stream_ptr(qkv.device)))
    return o


@gpu
@pytest.mark.parametrize("B,Hh,Ww,Cc,heads,k,dil", [(2, 9, 11, 72, 3, 3, [1, 2, 3]),
                                                   (1, 5, 6, 64, 4, 5, [1, 3]),
                                                   (2, 6, 7, 64, 1, 7, [4]),
                                                   (1, 30, 17, 192, 8, 3, [1, 2, 3, 5]),
                                                   (2, 40, 12, 48, 3, 3, [1, 9, 30]),
                                                   (1, 23, 9, 64, 2, 7, [12, 100]),
                                                   (1, 4, 4, 24, 3, 1, [1, 2, 3])])
def test_core_with_zero_queries_averages_the_gathered_values(B, Hh, Ww, Cc, heads, k, dil):
    """q = 0: every weight is 1 / k^2, so each output is the mean of the k^2 gathered values with zeros outside the map.  A wrong
    neighbour, a wrong group / head column or a masked border is a gross error."""
    g = torch.Generator().manual_seed(11)
    qkv = torch.randn(B, Hh, Ww, 3 * Cc, generator=g).half()
    qkv[..., :Cc] = 0
    o = _core(qkv.reshape(-1, 3 * Cc).cuda(), B, Hh, Ww, Cc, heads, k, dil, 0.3)
    torch.cuda.synchronize()
    nd = len(dil)
    Cg = Cc // nd
    v = qkv[..., 2 * Cc:].float()
    ref = torch.cat([gather_windows(v[..., gi * Cg:(gi + 1) * Cg], k, dil[gi]).mean(dim=-2) for gi in range(nd)], dim=-1)
    y = o.float().cpu().reshape(B, Hh, Ww, Cc)
    assert (y - ref).abs().max().item() < 2e-3 * max(1.0, ref.abs().max().item())


@gpu
def test_forward_leaves_x_untouched():
    spec = dict(variant="msda", ctor=dict(dim=72, num_heads=3), x=(2, 12, 12, 72))
    m, x, _ = _seeded(spec, 1)
    xg = x.half().cuda()
    x0 = xg.clone()
    with torch.no_grad():
        m.cuda()(xg)
        blk = pa.dilateformer.DilateBlock(72, 3).eval().cuda()
        blk.attention_half(xg)
        xn = xg.permute(0, 3, 1, 2)
        xn0 = xn.clone()
        blk.half()(xn)
    torch.cuda.synchronize()
    assert torch.equal(xg, x0) and torch.equal(xn, xn0)


@gpu
def test_full_batch_properties_and_oracle_slice():
    """Images are independent in eval mode: at B = 64 (tiny stage 1) a batch permutation permutes the output bit-exactly, and the
    first k images of the batch equal, bit for bit, the same k images run alone -- the small run the oracle pins."""
    spec = dict(variant="msda", ctor=dict(dim=72, num_heads=3, qkv_bias=True), x=(2, 56, 56, 72))
    m, x2, sd = _seeded(spec, 9)
    ref2 = run_case(spec, {"x": x2}, sd)
    m = m.cuda()
    gen = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(64, 56, 56, 72, device="cuda", generator=gen).half()
    x[:2] = x2.half().cuda()
    with torch.no_grad():
        y = m(x)
        perm = torch.randperm(64, device=x.device)
        assert torch.equal(m(x[perm]), y[perm])
        assert torch.equal(m(x[:2].contiguous()), y[:2])
    assert rel_fro(y[:2].float().cpu(), ref2) < TOL


@gpu
def test_capture_and_replay_in_a_cuda_graph():
    spec = dict(variant="dilate_block_half", ctor=dict(dim=72, num_heads=3, qkv_bias=True), x=(4, 28, 28, 72))
    m, x, _ = _seeded(spec, 2)
    m = m.cuda()
    xg = x.half().cuda()
    with torch.no_grad():
        y0 = m.attention_half(xg)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            m.attention_half(xg)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                yg = m.attention_half(xg)
        torch.cuda.current_stream().wait_stream(s)
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
    assert torch.equal(yg, y0)


@gpu
def test_error_mapping_on_the_device():
    x = torch.randn(1, 6, 6, 72, device="cuda").half()
    m = pa.dilateformer.MultiDilatelocalAttention(72, 3, attn_drop=0.1).cuda().train()
    with pytest.raises(NotImplementedError):
        m(x)
    blk = pa.dilateformer.DilateBlock(72, 3, drop_path=0.1).cuda().train()
    with pytest.raises(NotImplementedError):
        blk(x.permute(0, 3, 1, 2))
    assert blk.eval()(x.permute(0, 3, 1, 2)).shape == (1, 72, 6, 6)
    with pytest.raises(ValueError, match="head_dim 12"):
        pa.dilateformer.MultiDilatelocalAttention(36, 3).cuda().eval()(torch.randn(1, 6, 6, 36, device="cuda").half())
    with pytest.raises(AssertionError, match="odd"):
        pa.dilateformer.MultiDilatelocalAttention(72, 3, kernel_size=4).cuda().eval()(x)
