"""Host-side contract of the drop-in modules (no GPU): constructor signatures, state_dict keys/shapes,
error behaviour, and no silent CPU fallback."""
import inspect
import json
import os

import pytest
import torch

import pytorch_attention_b200 as pa
from _util import GOLDEN_DIR

# signatures and state_dict shapes of the reference classes, recorded by oracle/record_reference.py
with open(os.path.join(GOLDEN_DIR, "reference", "reference_contract.json")) as _f:
    CONTRACT = json.load(_f)["classes"]


class _Ref:
    """What was recorded of one reference class: its signatures and, per constructor call, its state_dict and attributes."""

    def __init__(self, name):
        self.name, self.entry = name, CONTRACT[name]
        self.init, self.forward = self.entry["init"], self.entry["forward"]

    def __call__(self, **kw):
        key = f"{self.name}(" + ", ".join(f"{k}={v!r}" for k, v in kw.items()) + ")"
        return self.entry["instances"][key]


def _ref_state_dict(inst):
    """Zero tensors with the recorded keys, shapes and dtypes of a reference module's state_dict."""
    return {k: torch.zeros(shape, dtype=getattr(torch, dt)) for k, (shape, dt) in inst["state_dict"].items()}


def _shapes(inst):
    return {k: torch.Size(shape) for k, (shape, _) in inst["state_dict"].items()}


def test_vit_state_dict_keys_and_shapes():
    m = pa.ViTAttention(768, 12)
    sd = m.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {
        "qkv.weight": (2304, 768), "proj.weight": (768, 768), "proj.bias": (768,)}
    m = pa.ViTAttention(128, 2, qkv_bias=True)
    assert "qkv.bias" in m.state_dict()
    assert m.scale == 64 ** -0.5


def test_vit_constructor_asserts_like_reference():
    with pytest.raises(AssertionError):       # ViT.py:70
        pa.ViTAttention(100, 3)


def test_cpu_tensor_is_an_error_not_a_fallback():
    m = pa.ViTAttention(128, 2).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 8, 128).half())


def test_unsupported_modes_raise():
    from pytorch_attention_b200._common import check_forward_mode

    class Fake:  # a CUDA-looking tensor stand-in is not constructible here; exercise the dtype / mode checks
        is_cuda, dtype, requires_grad, device = True, torch.float32, False, torch.device("cpu")
    m = pa.ViTAttention(128, 2, attn_drop=0.1)
    with pytest.raises(ValueError):
        check_forward_mode(m.eval(), Fake(), (0.1,))
    Fake.dtype = torch.float16
    with pytest.raises(NotImplementedError):
        check_forward_mode(m.train(), Fake(), (0.1,))
    check_forward_mode(m.eval(), Fake(), (0.1,))
    Fake.device = torch.device("cuda", 0)          # parameters elsewhere than the input: a clean error, not a bad pointer in a kernel
    with pytest.raises(RuntimeError, match="move the module"):
        check_forward_mode(m.eval(), Fake(), (0.1,))


def test_vit_matches_live_reference_contract():
    ref = _Ref("ViT.Attention")
    assert ref.init == str(inspect.signature(pa.ViTAttention.__init__))
    r = ref(dim=192, num_heads=3, qkv_bias=True)
    m = pa.ViTAttention(192, 3, qkv_bias=True)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))          # reference weights load unchanged


def test_setr_moat_defaults_and_keys():
    """setr.Attention / moat.Attention: ViT's parameters with the constructor default num_heads=8 (setr.py:51, moat.py:63)."""
    for cls in (pa.setr.Attention, pa.moat.Attention):
        m = cls(256)
        assert m.num_heads == 8 and m.scale == 32 ** -0.5
        assert sorted(m.state_dict()) == ["proj.bias", "proj.weight", "qkv.weight"]
        with pytest.raises(AssertionError):       # setr.py:53 / moat.py:65
            cls(100, 3)


@pytest.mark.parametrize("modname", ["setr", "moat"])
def test_setr_moat_match_live_reference_contract(modname):
    ref = _Ref(f"{modname}.Attention")
    ours = getattr(pa, modname).Attention
    assert ref.init == str(inspect.signature(ours.__init__))
    r = ref(dim=256, qkv_bias=True)
    m = ours(256, qkv_bias=True)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))


def test_param_stage_is_dropped_when_parameters_may_have_changed():
    """load_state_dict and every _apply (.to / .half / .float ...) clear the staged 16-bit copies; refresh() does it on demand
    (in-place edits through .data do not bump a tensor's version counter)."""
    m = pa.ViTAttention(128, 2).eval()
    m._stage.get("k", (m.qkv.weight,), lambda: "staged")
    assert m._stage._entries
    m.load_state_dict(m.state_dict())
    assert not m._stage._entries
    m._stage.get("k", (m.qkv.weight,), lambda: "staged")
    m.half()
    assert not m._stage._entries
    m._stage.get("k", (m.qkv.weight,), lambda: "staged")
    m.refresh()
    assert not m._stage._entries
    blk = pa.CSWinBlock(64, 14, 2)
    blk.attns[0]._stage.get("k", (), lambda: 1)
    blk.refresh()
    assert not blk.attns[0]._stage._entries


def test_build_is_atomic_and_locked(tmp_path, monkeypatch):
    """build_lib compiles to a temporary name and renames it into place under a file lock; a second caller that finds the
    library fresh after taking the lock does not compile again."""
    from pytorch_attention_b200 import build as b
    calls = []

    def fake_run(cmd, capture_output, text):
        out = cmd[cmd.index("-o") + 1]
        assert out != b.LIB_PATH and out.startswith(b.LIB_PATH + ".tmp.")
        open(out, "wb").write(b"x")
        calls.append(out)

        class R:
            returncode, stdout, stderr = 0, "", ""
        return R()
    monkeypatch.setattr(b, "LIB_DIR", str(tmp_path))
    monkeypatch.setattr(b, "LIB_PATH", str(tmp_path / "libpa_b200.so"))
    monkeypatch.setattr(b.subprocess, "run", fake_run)
    b.build_lib(force=True)
    assert len(calls) == 1 and (tmp_path / "libpa_b200.so").read_bytes() == b"x"
    assert not list(tmp_path.glob("*.tmp.*"))
    b.build_lib()                       # fresh: no second compile
    assert len(calls) == 1


def test_segformer_cmt_keys_and_defaults():
    """segformer.Attention (segformer.py:18-31): q, fused kv, dense sr conv with bias; cmt.Attention (cmt.py:73-91): pvt's keys."""
    m = pa.segformer.Attention(64, 2, qkv_bias=True, sr_ratio=4)
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == {
        "q.weight": (64, 64), "q.bias": (64,), "kv.weight": (128, 64), "kv.bias": (128,), "sr.weight": (64, 64, 4, 4),
        "sr.bias": (64,), "proj.weight": (64, 64), "proj.bias": (64,)}
    assert "sr.weight" not in pa.segformer.Attention(64, 2).state_dict()       # sr_ratio=1: no reduction conv (segformer.py:26)
    c = pa.cmt.Attention(128, 2, sr_ratio=2)
    assert sorted(c.state_dict()) == sorted(pa.pvt.Attention(128, 2, sr_ratio=2).state_dict())
    with pytest.raises(AssertionError):       # segformer.py:20 / cmt.py:76
        pa.segformer.Attention(100, 3)
    with pytest.raises(AssertionError):
        pa.cmt.Attention(100, 3)


@pytest.mark.parametrize("modname,cls,kw", [
    ("segformer", "Attention", dict(dim=64, num_heads=2, qkv_bias=True, sr_ratio=4)),
    ("cmt", "Attention", dict(dim=128, num_heads=2, sr_ratio=2, qkv_bias=True)),
    ("pvt", "Block", dict(dim=128, num_heads=2, sr_ratio=4)),
])
def test_siblings_match_live_reference_contract(modname, cls, kw):
    ref = _Ref(f"{modname}.{cls}")
    ours = getattr(getattr(pa, modname), cls)
    assert ref.init == str(inspect.signature(ours.__init__))
    if cls == "Attention":
        assert ref.forward == str(inspect.signature(ours.forward))
    r, m = ref(**kw), ours(**kw)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))          # reference weights load unchanged


def test_xca_block_attention_half_loads_a_reference_block():
    """XCABlockAttentionHalf holds the attention half's parameters under XCABlock's own keys (xcit.py:267-291)."""
    blk = _Ref("xcit.XCABlock")(dim=128, num_heads=4, qkv_bias=True, eta=1.0)
    m = pa.xcit.XCABlockAttentionHalf(128, 4, qkv_bias=True, eta=1.0)
    res = m.load_state_dict(_ref_state_dict(blk), strict=False)
    assert not res.missing_keys
    assert all(k.split(".")[0] in ("norm2", "norm3", "mlp", "local_mp", "gamma2", "gamma3") for k in res.unexpected_keys)


@pytest.mark.parametrize("kw", [dict(dim=192, heads=3, dim_head=64), dict(dim=64, heads=1, dim_head=64)])
def test_bvit_broad_attention_matches_live_reference_contract(kw):
    ref = _Ref("bvit.Broad_Attention")
    assert ref.init == str(inspect.signature(pa.bvit.Broad_Attention.__init__))
    r, m = ref(**kw), pa.bvit.Broad_Attention(**kw)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))
    assert isinstance(m.to_out, torch.nn.Identity) == r["to_out_is_identity"]


def test_pam_matches_live_reference_contract():
    ref = _Ref("dual_attention.PAM")
    assert ref.init == str(inspect.signature(pa.dual_attention.PAM.__init__))
    r, m = ref(dim=64), pa.dual_attention.PAM(64)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))


def test_dilateformer_global_attention_matches_live_reference_contract():
    ref = _Ref("dilateformer.GlobalAttention")
    ours = pa.dilateformer.GlobalAttention
    assert ref.init == str(inspect.signature(ours.__init__))
    r, m = ref(dim=128, num_heads=2, qkv_bias=True), ours(128, 2, qkv_bias=True)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))
    assert ours(128, 2, qk_scale=0.25).scale == ref.entry["qk_scale_0.25"] == 0.25


def test_p2t_pooling_attention_matches_live_reference_contract():
    ref = _Ref("p2t.PoolingAttention")
    ours = pa.p2t.PoolingAttention
    assert ref.init == str(inspect.signature(ours.__init__))
    assert ref.forward == str(inspect.signature(ours.forward))
    r, m = ref(dim=128, num_heads=2, qkv_bias=True), ours(128, 2, qkv_bias=True)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))
    assert m.num_elements == r["num_elements"]


def test_kvt_knn_attention_matches_live_reference_contract():
    ref = _Ref("kvt.KNNAttention")
    ours = pa.kvt.KNNAttention
    assert ref.init == str(inspect.signature(ours.__init__))
    r, m = ref(dim=128, num_heads=2, qkv_bias=True, topk=50), ours(128, 2, qkv_bias=True, topk=50)
    assert _shapes(r) == {k: v.shape for k, v in m.state_dict().items()}
    m.load_state_dict(_ref_state_dict(r))
    assert m.topk == r["topk"] == 50
