#!/usr/bin/env python
"""bench.py — attention-forward throughput of the B200 path on BASELINE.json's headline configuration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W      (N > 1)

A "step" is one forward of the drop-in ``ViT.Attention(768, 12)`` over one batch of synthetic tokens
(BASELINE.json configs[1]: B=64 per GPU, N=197, d=768, heads=12; weak scaling: each rank has its own batch,
no collective on the data path).  Rank 0 prints ONE JSON line; see DESIGN.md §Measurement for every field.

--dump-outputs DIR: after the timed steps, rank 0 writes the output of the last timed step, y [B, N, C], as DIR/y.npy
(float32).  Inputs and parameters are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOAD = dict(name="ViT-B/16 Attention fwd", B=64, N=197, C=768, H=12)
RING = 8   # distinct input/output buffers cycled through: 8 x 19.4 MB x 2 > 126 MB L2


def algorithmic_flops(B, N, C):
    return B * (8 * N * C * C + 4 * N * N * C)       # SURVEY.md §8(d): 5.3238 MFLOP/token for ViT-B


def algorithmic_bytes(B, N, C, elt=2):
    return elt * (2 * B * N * C + 4 * C * C + C)      # read x + params once, write y once


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return dict(bf16_tflops=pk["bf16_tflops"], bf16_tflops_sustained=pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                    hbm_gbs=pk["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.sm_max = index, [], set(), False, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def result(self):
        s = sorted(self.samples)
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.sm_max, reasons=sorted(self.reasons),
                    samples=len(s))


_ORIG_AFFINITY = None


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs NVML reports as local to GPU `index` BEFORE any pinned host buffer is allocated, so that
    the end-to-end leg's staging memory and the copy-issuing thread sit on the GPU's NUMA node (round-1 SCALE: GPU0-3 hang
    off NUMA node 0, GPU4-7 off node 1; unbound ranks lost 15 % of the PCIe rate).  Returns the number of CPUs bound to."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = nv.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [i for i in range(ncpu) if (int(mask[i // 64]) >> (i % 64)) & 1]
        allowed = os.sched_getaffinity(0)
        global _ORIG_AFFINITY
        _ORIG_AFFINITY = allowed
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        backend = "nccl" if torch.cuda.is_available() else "gloo"
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
        dist.init_process_group(backend=backend, device_id=torch.device("cuda", local) if backend == "nccl" else None)
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(val, world, device):
    if world == 1:
        return val
    import torch.distributed as dist
    t = torch.tensor([val], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def make_cpu_model(seed=0):
    """Reference-shaped parameters (nn.Linear default init), rounded once to fp16 so CPU and GPU see equal values."""
    g = torch.Generator().manual_seed(seed)
    C = WORKLOAD["C"]
    bound = 1.0 / C ** 0.5
    sd = {
        "qkv.weight": (torch.rand(3 * C, C, generator=g) * 2 - 1) * bound,
        "proj.weight": (torch.rand(C, C, generator=g) * 2 - 1) * bound,
        "proj.bias": (torch.rand(C, generator=g) * 2 - 1) * bound,
    }
    return {k: v.half().float() for k, v in sd.items()}


def cpu_forward_timer(sd, batch, runs):
    """Times the CPU port of the reference forward (oracle/aten_port.py: the reference's own ATen op sequence,
    fp32, all host threads) on a batch of `batch` images."""
    from oracle.aten_port import vit_attention_aten as vit_attention
    N, C, H = WORKLOAD["N"], WORKLOAD["C"], WORKLOAD["H"]
    x = torch.randn(batch, N, C).half().float()
    times = []
    with torch.no_grad():
        for i in range(runs + 1):
            t0 = time.perf_counter()
            vit_attention(x, sd["qkv.weight"], None, sd["proj.weight"], sd["proj.bias"], H)
            if i:                      # first run is the warm-up
                times.append(time.perf_counter() - t0)
    times.sort()
    return times[len(times) // 2]


def best_cpu_threads(sd):
    """The reference's forward is small for a many-core host: oversubscribing threads slows ATen down by >10x.
    Time a short probe at a few thread counts and keep the fastest (that count is what `cores` reports)."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        t = cpu_forward_timer(sd, 8, 2)
        if best_t is None or t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU forward (oracle port of ViT.py:79-89) on the host cores."""
    if rank != 0:
        return
    sd = make_cpu_model()
    best_cpu_threads(sd)
    N = WORKLOAD["N"]
    t8 = cpu_forward_timer(sd, 8, 1)
    budget = 120.0
    per_step_batch = int(max(1, min(WORKLOAD["B"], budget / max(1, args.steps + args.warmup) / (t8 / 8))))
    from oracle.aten_port import vit_attention_aten as vit_attention
    x = torch.randn(per_step_batch, N, WORKLOAD["C"]).half().float()
    with torch.no_grad():
        for _ in range(args.warmup):
            vit_attention(x, sd["qkv.weight"], None, sd["proj.weight"], sd["proj.bias"], WORKLOAD["H"])
        t0 = time.perf_counter()
        for _ in range(args.steps):
            vit_attention(x, sd["qkv.weight"], None, sd["proj.weight"], sd["proj.bias"], WORKLOAD["H"])
        dt = time.perf_counter() - t0
    val = per_step_batch * N * args.steps / dt
    sample = f"{per_step_batch} of {WORKLOAD['B']} images per step (fp32 torch CPU, ATen-op port of ViT.py:79-89)"
    out = dict(impl="reference", metric="attn-fwd tokens/sec (ViT-B N=197 d=768)", value=val, unit="tokens/s", n_gpus=args.gpus,
               steps=args.steps, warmup=args.warmup, ms_per_step=dt / args.steps * 1e3, higher_is_better=True,
               scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
               config=dict(workload="ViT.Attention(768,12) fwd, N=197, host CPU", batch_per_step=per_step_batch),
               cpu_baseline=dict(value=val, unit="tokens/s", cores=torch.get_num_threads(), threads=torch.get_num_threads(),
                                 host_cpus=os.cpu_count(), kind="port", sample=sample),
               e2e=dict(value=val, unit="tokens/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out), flush=True)


def run_ours(args, rank, world, local):
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    import pytorch_attention_b200 as pa
    from pytorch_attention_b200 import _lib, ops
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    numa_cpus = bind_to_gpu_numa(local)
    B, N, C, H = WORKLOAD["B"], WORKLOAD["N"], WORKLOAD["C"], WORKLOAD["H"]
    dt = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    sd = make_cpu_model()
    mod = pa.ViTAttention(C, H).eval()
    mod.load_state_dict(sd)
    mod = mod.to(dev)
    mod.out_dtype = torch.float16      # y in fp16: the only 16-bit output type that can meet the 1e-3 parity bar
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    xs = [torch.randn(B, N, C, device=dev, generator=gen).to(dt) for _ in range(RING)]
    peaks = load_peaks()

    with torch.no_grad():
        for i in range(3):
            mod(xs[i % RING])
        torch.cuda.synchronize()
        # one CUDA graph per ring slot: the three launches of a step replay without host work
        graphs, outs = [], []
        if not args.no_graph:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                mod(xs[0])
            torch.cuda.current_stream().wait_stream(side)
            for i in range(RING):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    y = mod(xs[i])
                graphs.append(g)
                outs.append(y)

        l_before = _lib.launch_count()
        mod(xs[0])                                   # eager: count this library's kernel launches per forward
        launches_per_forward = _lib.launch_count() - l_before
        fused = launches_per_forward == 1
        vit_path = {1: "three launches", 2: "vit_fused_kernel (sequenced phases)", 3: "vit_cosched_kernel (GEMMs under the softmax chain)"}.get(
            int(_lib.load().pa_last_vit_path()), "?")

        def step(i):
            if graphs:
                graphs[i % RING].replay()
                return outs[i % RING]
            return mod(xs[i % RING])

        for i in range(max(args.warmup, 3)):
            step(i)
        torch.cuda.synchronize()
        barrier(world)
        sampler = ClockSampler(local)
        sampler.start()
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(args.steps):
            y_last = step(i)
        e1.record()
        torch.cuda.synchronize()
        sampler.stop_flag = True
        sampler.join()
        if args.dump_outputs and rank == 0:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "y.npy"), y_last.float().cpu().numpy())
        barrier(world)
        launches = (_lib.launch_count() - l0) if not graphs else launches_per_forward * args.steps
        elapsed_ms = max_over_ranks(e0.elapsed_time(e1), world, dev)

        # ---- end-to-end leg: host (pinned) x -> H2D -> forward -> D2H y, every step, copies inside the timed region
        hx = [torch.randn(B, N, C).to(dt).pin_memory() for _ in range(2)]
        hy = [torch.empty(B, N, C, dtype=torch.float16).pin_memory() for _ in range(2)]
        dx = [torch.empty(B, N, C, dtype=dt, device=dev) for _ in range(2)]
        s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_cmp = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]
        dys = [None, None]

        def e2e_steps(n):
            for i in range(n):
                b = i & 1
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_cmp[b])        # dx[b] free once the forward that read it is done
                    dx[b].copy_(hx[b], non_blocking=True)
                    ev_in[b].record(s_in)
                with torch.cuda.stream(s_cmp):
                    s_cmp.wait_event(ev_in[b])
                    s_cmp.wait_event(ev_out[b])       # previous D2H of this slot's y finished
                    dys[b] = mod(dx[b])
                    ev_cmp[b].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[b])
                    hy[b].copy_(dys[b], non_blocking=True)
                    ev_out[b].record(s_out)
            torch.cuda.synchronize()

        e2e_n = 200                    # fixed: independent of --steps (a 20-step sample was noise-dominated in round 1)
        e2e_steps(20)
        barrier(world)
        t0 = time.perf_counter()
        e2e_steps(e2e_n)
        e2e_dt = max_over_ranks(time.perf_counter() - t0, world, dev)
        barrier(world)

        # ---- per-kernel durations (CUDA events on the launching stream), rank 0 only
        kern = {}
        if rank == 0:
            rows = B * N
            wq = mod.qkv.weight.detach().to(dt)
            wp = mod.proj.weight.detach().half()
            bp = mod.proj.bias.detach().float()
            qkv = torch.empty(RING, rows, 3 * C, dtype=torch.float16, device=dev)   # ring > L2
            obuf = torch.empty(RING, rows, C, dtype=torch.float16, device=dev)
            ybuf = torch.empty(RING, rows, C, dtype=torch.float16, device=dev)
            xf = [x.view(rows, C) for x in xs]

            def timed(fn, reps=6):
                """One CUDA graph holding RING launches (one per ring slot), replayed `reps` times: device time only."""
                for i in range(RING):
                    fn(i)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for i in range(RING):
                        fn(i)
                g.replay()
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(reps):
                    g.replay()
                b.record()
                torch.cuda.synchronize()
                return a.elapsed_time(b) / (reps * RING) * 1e3

            kern["qkv_gemm_us"] = timed(lambda i: ops.gemm_tn(xf[i % RING], wq, out=qkv[i % RING]))
            kern["attn_core_us"] = timed(lambda i: ops.attn_core(qkv[i % RING].view(B, N, 3 * C), qkv[i % RING].view(B, N, 3 * C), H,
                                                                 mod.scale, 0, C, 2 * C, out=obuf[i % RING].view(B, N, C)))
            kern["proj_gemm_us"] = timed(lambda i: ops.gemm_tn(obuf[i % RING], wp, bias=bp, out=ybuf[i % RING]))

    if rank != 0:
        return
    tokens = B * N * world
    ms_per_step = elapsed_ms / args.steps
    value = tokens / (ms_per_step * 1e-3)
    flops_step = algorithmic_flops(B, N, C)
    qkv_flops = 2.0 * B * N * C * 3 * C
    roof_peak = peaks["bf16_tflops"]
    if fused:
        # one kernel IS the step: algorithmic flops of the whole forward / its average duration in the timed region.
        # Denominator: the BURST cuBLAS figure -- the timed region is K launches of < 0.1 ms at full clock (milliseconds in
        # total), not a seconds-long power-capped loop; the sustained figure is printed beside it for reference.
        roof_kernel = vit_path
        achieved = flops_step / (ms_per_step * 1e-3) / 1e12
        roof_peak, peak_kind = peaks["bf16_tflops"], "burst"
        traffic_key = "vit_cosched_dram_bytes_per_launch" if "cosched" in vit_path else "vit_fused_dram_bytes_per_launch"
    else:
        roof_kernel = "gemm_tn_kernel (qkv projection)"
        achieved = qkv_flops / (kern["qkv_gemm_us"] * 1e-6) / 1e12
        peak_kind, traffic_key = "burst (kernel timed alone)", "qkv_gemm_dram_bytes_per_launch"
    traffic = None
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            with open(prof) as f:
                traffic = json.load(f).get(traffic_key)
        except Exception:
            traffic = None
    # CPU baseline: oracle port on the host cores, bounded sample (a few forwards of 16 images)
    cpu_batch = 64
    cpu_line = None                              # timed on rank 0 at N=1 only (the scaling runs do not repeat it)
    if world == 1:
        if _ORIG_AFFINITY:
            os.sched_setaffinity(0, _ORIG_AFFINITY)      # the CPU arm may use every host core again
        best_cpu_threads(sd)
        t_cpu = cpu_forward_timer(sd, cpu_batch, 5)
        cpu_line = dict(value=cpu_batch * N / t_cpu, unit="tokens/s", cores=torch.get_num_threads(), threads=torch.get_num_threads(),
                        host_cpus=os.cpu_count(), kind="port",
                        sample=f"median of 5 forwards of {cpu_batch} images (fp32 torch CPU, ATen-op port of ViT.py:79-89); "
                               f"threads = fastest of a short probe over {{8,16,32,64,all}} of the host's {os.cpu_count()} CPUs")
    other = None
    if world == 1 and not args.no_other_configs:
        # the other BASELINE.json configurations (parity-test cases, NOT the bench line): one device-timed number each
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_configs
            other = bench_configs.collect(reps=20)
        except Exception as e:      # never lose the headline line to a side measurement
            other = [dict(error=repr(e))]
    out = dict(
        metric="attn-fwd tokens/sec (ViT-B N=197 d=768)", value=value, unit="tokens/s", n_gpus=world, steps=args.steps,
        warmup=args.warmup, ms_per_step=ms_per_step, higher_is_better=True, scaling="weak", vs_baseline=None,
        dtype=args.dtype, data="synthetic",
        config=dict(workload="ViT-B/16 Attention fwd, B=64 per GPU, N=197, dim=768, heads=12 (BASELINE.json configs[1])",
                    global_batch=B * world, per_gpu_batch=B, tokens_per_step=tokens, io_dtype=args.dtype, out_dtype="fp16",
                    accumulate="fp32", parallelism=f"dp{world} (batch-sharded, no collective)",
                    l2="inputs/outputs rotate over a ring of %d buffers (%.0f MB) > 126 MB L2" % (RING, RING * 2 * B * N * C * 2 / 1e6),
                    cuda_graph=not args.no_graph, fused_single_launch=bool(fused), path=vit_path,
                    numa_bound_cpus=numa_cpus),
        step_tflops=flops_step * world / (ms_per_step * 1e-3) / 1e12,
        step_frac_of_peak=flops_step / (ms_per_step * 1e-3) / 1e12 / peaks["bf16_tflops"],
        step_frac_of_sustained_peak=flops_step / (ms_per_step * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
        roofline=dict(bound="tensor", kernel=roof_kernel, achieved=achieved, peak=roof_peak, unit="TFLOP/s",
                      frac=achieved / roof_peak, traffic=traffic, peak_source=peaks["source"] + ", " + peak_kind),
        phase_kernels_alone_us=kern,
        qkv_gemm_alone=dict(tflops=qkv_flops / (kern["qkv_gemm_us"] * 1e-6) / 1e12,
                            frac_of_burst_peak=qkv_flops / (kern["qkv_gemm_us"] * 1e-6) / 1e12 / peaks["bf16_tflops"]),
        cpu_baseline=cpu_line,
        e2e=dict(value=tokens * e2e_n / e2e_dt, unit="tokens/s", h2d_bytes_per_step=B * N * C * 2, d2h_bytes_per_step=B * N * C * 2,
                 steps=e2e_n, warmup=20,
                 note="pinned host x -> H2D -> forward -> D2H y each step; 3 streams, 2 slots in flight; process bound to the GPU's NUMA node"),
        gpu_launches=int(launches),
        clocks=sampler.result(),
        other_configs=other,
    )
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-fused", action="store_true", help="three launches (qkv GEMM, attention, proj GEMM) instead of a single-launch kernel")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the side measurements of the other BASELINE configurations")
    ap.add_argument("--no-cosched", action="store_true", help="sequenced single-launch kernel instead of the co-scheduled one")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output to DIR/y.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the output of the B200 path (--impl ours)")
    if args.no_fused:
        os.environ["PA_VIT_FUSED"] = "0"
    if args.no_cosched:
        os.environ["PA_VIT_COSCHED"] = "0"
    rank, world, local = dist_setup(args.gpus)
    try:
        if args.impl == "reference":
            run_reference(args, rank, world)
        else:
            run_ours(args, rank, world, local)
    finally:
        if world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
