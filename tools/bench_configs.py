#!/usr/bin/env python
"""Throughput of the drop-ins on the other BASELINE.json configurations (parity-test cases, not the bench line):
C3 PVT-SR8, C4 CSWin block (attention half), C4' CSWin last stage, C5 ViT-L per-GPU shard, plus XCA and CvT shapes.
Each forward is captured in a CUDA graph and replayed; device time by CUDA events.  JSON lines -> gpurun_out/configs.jsonl"""
from __future__ import annotations

import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import pytorch_attention_b200 as pa  # noqa: E402
from pytorch_attention_b200 import _lib  # noqa: E402

OUT = os.path.join(ROOT, "gpurun_out")
PEAK = 1704.0
try:
    PEAK = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]
except Exception:
    pass


def graph_time(fn, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e3


_collected = None     # collect(): lines are gathered instead of printed


def emit(**kw):
    if _collected is not None:
        _collected.append(kw)
        return
    line = json.dumps(kw)
    print(line, flush=True)
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "configs.jsonl"), "a") as f:
        f.write(line + "\n")


REPS = 20


def collect(reps=20):
    """All configurations as a list of dicts (bench.py's `other_configs` key)."""
    global _collected, REPS
    _collected, REPS = [], reps
    try:
        main()
        return _collected
    finally:
        _collected = None


def run(name, mod, x, call, tokens, flops, launches_expected=None):
    mod = mod.eval().half().cuda()
    with torch.no_grad():
        n0 = _lib.launch_count()
        y = call(mod, x)
        torch.cuda.synchronize()
        n1 = _lib.launch_count()
        us = graph_time(lambda: call(mod, x), REPS)
    emit(config=name, us=round(us, 2), tokens_per_s=round(tokens / us * 1e6), tflops=round(flops / us / 1e6, 1),
         frac_of_measured_peak=round(flops / us / 1e6 / PEAK, 3), launches=n1 - n0, out_shape=list(y.shape))


def main():
    torch.manual_seed(0)
    dev = "cuda"
    # C5 per-GPU shard: ViT-L/16 attention, 64 images, dim 1024, 16 heads
    B, N, C = 64, 197, 1024
    run("C5 shard: ViT-L Attention B=64 N=197 C=1024 H=16", pa.vit.Attention(C, 16), torch.randn(B, N, C, device=dev).half(),
        lambda m, x: m(x), B * N, B * (8 * N * C * C + 4 * N * N * C))
    # C2 for reference
    B, N, C = 64, 197, 768
    run("C2: ViT-B Attention B=64 N=197 C=768 H=12", pa.vit.Attention(C, 12), torch.randn(B, N, C, device=dev).half(),
        lambda m, x: m(x), B * N, B * (8 * N * C * C + 4 * N * N * C))
    # C3: PVT SR-attention sr=8, B=32, 64x64 tokens, dim 512, 8 heads
    B, Hh, Ww, C, sr = 32, 64, 64, 512, 8
    N, M = Hh * Ww, (Hh // sr) * (Ww // sr)
    m = pa.pvt.Attention(C, 8, sr_ratio=sr)
    run("C3: PVT SR-Attention sr=8 B=32 64x64 C=512 H=8", m, torch.randn(B, N, C, device=dev).half(),
        lambda mod, x: mod(x, Hh, Ww), B * N, B * (4 * N * C * C + 4 * M * C * C + 4 * N * M * C + 2 * M * C * sr * sr))
    # C4: CSWin block attention half, reso 56, dim 512, 16 heads, split 7, B=128
    B, R, C = 128, 56, 512
    L = R * R
    m = pa.cswin.CSWinBlock(C, R, 16, split_size=7, qkv_bias=True)
    Nw = R * 7
    run("C4: CSWinBlock attention half B=128 reso=56 C=512 H=16 split=7", m, torch.randn(B, L, C, device=dev).half(),
        lambda mod, x: mod.attention_half(x), B * L, B * (8 * L * C * C + 2 * 4 * L * Nw * (C // 2) + 18 * L * C))
    # C4': last stage, reso 7
    B, R, C = 128, 7, 512
    L = R * R
    m = pa.cswin.CSWinBlock(C, R, 16, split_size=7, qkv_bias=True, last_stage=True)
    run("C4': CSWinBlock last stage B=128 reso=7 C=512 H=16", m, torch.randn(B, L, C, device=dev).half(),
        lambda mod, x: mod.attention_half(x), B * L, B * (8 * L * C * C + 4 * L * L * C + 18 * L * C))
    # XCA and CvT zoo-like shapes
    B, N, C = 64, 196, 768
    run("XCA B=64 N=196 C=768 H=12", pa.xcit.XCA(C, 12), torch.randn(B, N, C, device=dev).half(), lambda m, x: m(x), B * N,
        B * (8 * N * C * C + 4 * N * C * 64))
    B, C, Hh = 64, 384, 14
    run("CvT B=64 C=384 14x14 H=6", pa.cvt.Attention(C, 6), torch.randn(B, C, Hh, Hh, device=dev).half(), lambda m, x: m(x),
        B * Hh * Hh, B * (8 * Hh * Hh * C * C + 4 * (Hh * Hh) ** 2 * C + 18 * Hh * Hh * C))
    B, N, C = 64, 197, 768
    run("ClassAttention B=64 N=197 C=768 H=12", pa.xcit.ClassAttention(C, 12), torch.randn(B, N, C, device=dev).half(), lambda m, x: m(x),
        B * N, B * (6 * N * C * C + 2 * C * C + 4 * N * C))
    # round-2 siblings / block halves (rows f-1, f-2, f-4): same geometry as C3 / XCA / C2 so the lines compare
    B, Hh, Ww, C, sr = 32, 64, 64, 512, 8
    N, M = Hh * Ww, (Hh // sr) * (Ww // sr)
    pvt_flops = B * (4 * N * C * C + 4 * M * C * C + 4 * N * M * C)
    run("SegFormer Attention sr=8 B=32 64x64 C=512 H=8 (dense reduction conv)", pa.segformer.Attention(C, 8, sr_ratio=sr),
        torch.randn(B, N, C, device=dev).half(), lambda mod, x: mod(x, Hh, Ww), B * N, pvt_flops + B * 2 * M * C * C * sr * sr)
    rel = torch.randn(8, N, M, device=dev)
    run("CMT Attention sr=8 B=32 64x64 C=512 H=8 (+ relative_pos)", pa.cmt.Attention(C, 8, sr_ratio=sr),
        torch.randn(B, N, C, device=dev).half(), lambda mod, x: mod(x, Hh, Ww, rel), B * N, pvt_flops + B * 2 * M * C * sr * sr)
    run("pvt.Block attention half sr=8 B=32 64x64 C=512 H=8 (LN + residual)", pa.pvt.Block(C, 8, sr_ratio=sr),
        torch.randn(B, N, C, device=dev).half(), lambda mod, x: mod.attention_half(x, Hh, Ww), B * N, pvt_flops + B * 2 * M * C * sr * sr)
    B, N, C = 64, 196, 768
    run("XCABlock attention half B=64 N=196 C=768 H=12 (LN + LayerScale + residual)", pa.xcit.XCABlockAttentionHalf(C, 12, eta=1.0),
        torch.randn(B, N, C, device=dev).half(), lambda m, x: m(x), B * N, B * (8 * N * C * C + 4 * N * C * 64))
    B, N, C = 64, 197, 768
    run("ViT TransformerEncoder attention half B=64 N=197 C=768 H=12 (LN + residual)", pa.vit.TransformerEncoder(C, 12),
        torch.randn(B, N, C, device=dev).half(), lambda m, x: m.attention_half(x), B * N, B * (8 * N * C * C + 4 * N * N * C))
    run("bvit.Broad_Attention B=64 N=197 dim=768 heads=12 dim_head=64", pa.bvit.Broad_Attention(C, 12, 64),
        torch.randn(B, N, C, device=dev).half(), lambda m, x: m(x)[0], B * N, B * (8 * N * C * C + 4 * N * N * C))


if __name__ == "__main__":
    main()
