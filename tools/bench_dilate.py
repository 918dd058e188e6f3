#!/usr/bin/env python
"""Device time of DilateFormer's multi-scale dilated attention (MultiDilatelocalAttention, dilateformer.py:64-97) on the B200.

For each shape: the whole forward (GEMM(qkv) -> dilated-attention kernel -> GEMM(proj)) and the dilated-attention kernel alone
(pa_dilate_core), each captured once in a CUDA graph and replayed between CUDA events -- --repeats windows of --iters replays
each, the median reported with the spread (min / max) of the windows; and the same math in eager PyTorch fp16
(the reference's unfold / matmul / softmax formulation) on the same GPU.  Batches are chosen so that the qkv buffer (the
kernel's input) is larger than the 126 MB L2, so the kernel reads it from HBM; every line says whether it fits.  Achieved GB/s
counts the bytes the algorithm needs (kernel: qkv read once, O written once = 8 C bytes per token; forward: x, qkv written and
read, O written and read, y = 20 C bytes per token) over device time, against 7.7 TB/s of HBM3e.  The card's name and power
limit are read in the same run.  One JSON line per shape on stdout (and in --out DIR/bench_dilate.jsonl)."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pytorch_attention_b200 as pa  # noqa: E402
from pytorch_attention_b200 import _lib as L  # noqa: E402
from pytorch_attention_b200 import ops  # noqa: E402

HBM_TBPS = 7.7
L2_BYTES = 126e6
# name -> (B, H, W, C, heads): DilateFormer stage shapes at 224 x 224 (dilateformer.py:446-461), kernel 3, dilation [1, 2, 3]
SHAPES = {
    "tiny_stage1": (128, 56, 56, 72, 3),
    "tiny_stage2": (256, 28, 28, 144, 6),
    "base_stage1": (128, 56, 56, 96, 3),
}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        idx = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0] or "0"
        out = subprocess.run(["nvidia-smi", "-i", idx, "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return name, float(out[0]), float(out[1])
    except Exception:                  # noqa: BLE001 -- the fields are reported as unknown
        return name, None, None


def graph_time_us(fn, iters, warmup, repeats):
    """Per-call device time of `fn` in each of `repeats` windows of `iters` graph replays."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(warmup):
        g.replay()
    return windows_us(g.replay, iters, repeats)


def windows_us(fn, iters, repeats):
    out = []
    for _ in range(repeats):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(iters):
            fn()
        t1.record()
        torch.cuda.synchronize()
        out.append(t0.elapsed_time(t1) * 1e3 / iters)
    return out


def event_time_us(fn, iters, warmup, repeats):
    for _ in range(warmup):
        fn()
    return windows_us(fn, iters, repeats)


def stats(ts):
    ts = sorted(ts)
    return ts[len(ts) // 2], ts[0], ts[-1]


def eager_forward(m, x):
    """dilateformer.py:85-97 in eager PyTorch on fp16 tensors (without writing into x)."""
    B, H, W, C = x.shape
    nd, k = m.num_dilation, m.kernel_size
    Cg, hd = C // nd, C // m.num_heads
    qkv = F.conv2d(x.permute(0, 3, 1, 2), m.qkv.weight, m.qkv.bias).reshape(B, 3, nd, Cg, H, W).permute(2, 1, 0, 3, 4, 5)
    out = torch.empty(nd, B, H, W, Cg, dtype=x.dtype, device=x.device)
    for i, d in enumerate(m.dilation):
        q, kk, v = qkv[i][0], qkv[i][1], qkv[i][2]
        q = q.reshape(B, Cg // hd, hd, 1, H * W).permute(0, 1, 4, 3, 2)
        kk = F.unfold(kk, k, d, d * (k - 1) // 2, 1).reshape(B, Cg // hd, hd, k * k, H * W).permute(0, 1, 4, 2, 3)
        a = ((q @ kk) * m.scale).softmax(dim=-1)
        v = F.unfold(v, k, d, d * (k - 1) // 2, 1).reshape(B, Cg // hd, hd, k * k, H * W).permute(0, 1, 4, 3, 2)
        out[i] = (a @ v).transpose(1, 2).reshape(B, H, W, Cg)
    return m.proj(out.permute(1, 2, 3, 0, 4).reshape(B, H, W, C))


def run_shape(name, B, H, W, C, heads, iters, warmup, repeats, dev):
    torch.manual_seed(0)
    m = pa.dilateformer.MultiDilatelocalAttention(C, heads, qkv_bias=True).half().cuda().eval()
    x = torch.randn(B, H, W, C, device="cuda", dtype=torch.float16)
    tokens = B * H * W
    qkv = torch.randn(tokens, 3 * C, device="cuda", dtype=torch.float16)
    o = torch.empty(tokens, C, device="cuda", dtype=torch.float16)
    a = L.DilateArgs()
    a.B, a.Himg, a.Wimg, a.C, a.H, a.kernel_size, a.n_dilation, a.scale = B, H, W, C, heads, 3, 3, float(m.scale)
    for i, d in enumerate(m.dilation):
        a.dilation[i] = d
    lib = L.load()

    def core():
        L.check(lib.pa_dilate_core(ctypes.byref(a), ops._ptr(qkv), ops._ptr(o), ops.stream_ptr(x.device)))

    with torch.no_grad():
        y = m(x)
        ye = eager_forward(m, x)
        torch.cuda.synchronize()
        err = ((y.float() - ye.float()).abs().max() / ye.float().abs().max()).item()
        fwd_us, fwd_min, fwd_max = stats(graph_time_us(lambda: m(x), iters, warmup, repeats))
        core_us, core_min, core_max = stats(graph_time_us(core, iters, warmup, repeats))
        eager_us, eager_min, eager_max = stats(event_time_us(lambda: eager_forward(m, x), max(3, iters // 20), 2, repeats))
    core_bytes = tokens * 8 * C
    fwd_bytes = tokens * 20 * C
    qkv_bytes = tokens * 3 * C * 2
    name_, plimit, clk = dev
    return dict(shape=name, B=B, H=H, W=W, C=C, heads=heads, kernel_size=3, dilation=list(m.dilation),
                qkv_bytes=qkv_bytes, qkv_fits_l2=qkv_bytes <= L2_BYTES,
                core_us=round(core_us, 2), core_us_min=round(core_min, 2), core_us_max=round(core_max, 2), core_bytes=core_bytes, core_GBps=round(core_bytes / core_us / 1e3, 1),
                core_share_of_hbm=round(core_bytes / core_us / 1e6 / HBM_TBPS, 3),
                fwd_us=round(fwd_us, 2), fwd_us_min=round(fwd_min, 2), fwd_us_max=round(fwd_max, 2), fwd_bytes=fwd_bytes, fwd_GBps=round(fwd_bytes / fwd_us / 1e3, 1),
                eager_fp16_fwd_us=round(eager_us, 2), eager_fp16_fwd_us_min=round(eager_min, 2),
                eager_fp16_fwd_us_max=round(eager_max, 2), speedup_vs_eager=round(eager_us / fwd_us, 2),
                max_rel_diff_vs_eager=err, iters=iters, repeats=repeats, device=name_, power_limit_W=plimit, clocks_max_sm_MHz=clk)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--shapes", nargs="*", default=list(SHAPES), choices=list(SHAPES))
    ap.add_argument("--iters", type=int, default=500, help="graph replays per timed window (>= 60 ms of work per window)")
    ap.add_argument("--repeats", type=int, default=5, help="timed windows per measurement")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for bench_dilate.jsonl (created when given)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dilate.py measures on a CUDA device; none is available")
    dev = card()
    lines = []
    for s in args.shapes:
        r = run_shape(s, *SHAPES[s], args.iters, args.warmup, args.repeats, dev)
        print(json.dumps(r), flush=True)
        lines.append(r)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_dilate.jsonl"), "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
