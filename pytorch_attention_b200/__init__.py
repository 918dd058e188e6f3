"""pytorch_attention_b200 — B200-native (sm_100a) attention forward, drop-in for the attention modules of
changzy00/pytorch-attention's vision_transformers/ (ViT, PVT, CvT, CSWin, XCiT, the ViT-identical SETR / MOAT attention and
the PVT siblings SegFormer / CMT, BViT's Broad_Attention, DilateFormer's multi-scale dilated attention) and of attention_mechanisms/dual_attention.py (PAM).

Python here is plumbing only (module state, device memory, streams); all arithmetic runs in the hand-written
CUDA library ``lib/libpa_b200.so`` behind the C ABI declared in ``include/pa_b200.h``.  The sub-modules mirror
the reference's file names so that ``from pytorch_attention_b200.pvt import Attention`` replaces
``from pvt import Attention``.
"""
from . import _lib, ops  # noqa: F401
from . import vit, pvt, cvt, cswin, xcit, setr, moat, segformer, cmt, bvit, dual_attention, dilateformer, p2t, kvt  # noqa: F401
from .vit import Attention as ViTAttention  # noqa: F401
from .vit import TransformerEncoder as ViTTransformerEncoder  # noqa: F401
from .pvt import Attention as PVTAttention  # noqa: F401
from .cvt import Attention as CvTAttention  # noqa: F401
from .cswin import LePEAttention, CSWinBlock  # noqa: F401
from .xcit import XCA, ClassAttention  # noqa: F401
from .dilateformer import MultiDilatelocalAttention, DilateBlock  # noqa: F401

__all__ = ["ops", "vit", "pvt", "cvt", "cswin", "xcit", "setr", "moat", "segformer", "cmt", "bvit", "dual_attention", "dilateformer", "p2t", "kvt", "ViTAttention", "ViTTransformerEncoder", "PVTAttention", "CvTAttention",
           "LePEAttention", "CSWinBlock", "XCA", "ClassAttention", "MultiDilatelocalAttention", "DilateBlock"]
