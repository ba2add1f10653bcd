#!/usr/bin/env python
"""Fused SSIM (deblurgs_b200.loss.ssim, dgs_ssim.cu) against the torch statement of the reference's `ssim`
(oracle/ssim_torch.py: 5 depthwise 11x11 conv2d through cuDNN in fp32 plus the elementwise map), both arms in one
process on one GPU, and the cost of the D-SSIM term in the graph-replayed c2 training step.

Per shape, each arm is timed with CUDA events in two ways after a warm-up:
  device  : GRAPH_CALLS calls captured in one CUDA graph, replayed; per-call time = GPU time without host overhead
  eager   : the Python call in a loop, as a training script issues it (host overhead included where it dominates)
for the forward alone (metric call, no gradient maps), the forward that writes the gradient maps, and forward +
backward (torch.autograd.grad; the backward alone is the difference of the last two).  Achieved bytes/s are over the
least traffic each fused call needs: forward = read 2 images + write 3 maps, backward = read 3 maps + 2 images + write
1 image.  The c2 working set (~14 MB) stays in the 126 MB L2 between calls,
the [16,3,400,600] stack (5 planes = 230 MB) does not; c3 (5 planes = 124 MB) is at the edge.

Step cost: BlurryViewGraph at c2 (300k Gaussians, 600x400, 16 sub-frames) with lambda_dssim = 0.2 and 0, replays
alternated in ROUNDS rounds of STEP_ITERS; the median per-step difference is the added cost.

  python tools/bench_ssim.py [--iters 200] [--out profiles/ssim_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deblurgs_b200.loss import ssim  # noqa: E402
from oracle import ssim_torch as ot  # noqa: E402

SHAPES = {"c2": (3, 400, 600), "stack16": (16, 3, 400, 600), "c3": (3, 1080, 1920)}
GRAPH_CALLS = 20
ROUNDS, STEP_ITERS = 5, 50


def gpu_identity():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": r.stdout.strip()}


def events_ms(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def time_arm(fn, iters, warmup):
    """(device ms per call from graph replays, eager ms per call)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    eager = events_ms(fn, iters)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(GRAPH_CALLS):
            fn()
    for _ in range(3):
        graph.replay()
    device = events_ms(graph.replay, max(iters // GRAPH_CALLS, 10)) / GRAPH_CALLS
    return device, eager


def bench_shape(name, shape, iters, warmup):
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(shape, generator=g, device="cuda")
    y = (x + 0.1 * torch.randn(shape, generator=g, device="cuda")).clamp(0, 1)
    xr = x.clone().requires_grad_(True)
    # the torch arm with its window already on the device (the reference copies it from the host on every call)
    window = ot.create_window(11, shape[-3]).cuda()
    ref = lambda a, b: ot._ssim(a, b, window, 11, shape[-3], True)   # noqa: E731
    arms = {}
    for arm, f in (("fused", ssim), ("torch", ref)):
        res = {
            "fwd": time_arm(lambda: f(x, y), iters, warmup),
            "fwd_grad_maps": time_arm(lambda: f(xr, y), iters, warmup),
            "fwd_bwd": time_arm(lambda: torch.autograd.grad(f(xr, y), xr), iters, warmup),
        }
        arms[arm] = {k: {"device_ms": round(v[0], 5), "eager_ms": round(v[1], 5)} for k, v in res.items()}
    n = x.numel()
    fwd_bytes, bwd_bytes = 5 * 4 * n, 6 * 4 * n
    fu, to = arms["fused"], arms["torch"]
    bwd_ms = fu["fwd_bwd"]["device_ms"] - fu["fwd_grad_maps"]["device_ms"]
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    with torch.no_grad():
        diff = abs(ssim(x, y).item() - ref(x, y).item())
    torch.backends.cudnn.allow_tf32 = prev
    return {
        "shape": list(shape), **arms,
        "speedup_device": {k: round(to[k]["device_ms"] / fu[k]["device_ms"], 2) for k in fu},
        "speedup_eager": {k: round(to[k]["eager_ms"] / fu[k]["eager_ms"], 2) for k in fu},
        "min_bytes": {"fwd_grad_maps": fwd_bytes, "bwd": bwd_bytes},
        # backward device time = (forward + backward) - (forward writing the maps); includes the upstream-gradient fill
        "fused_bwd_device_ms": round(bwd_ms, 5),
        "fused_achieved_GBps": {"fwd_grad_maps": round(fwd_bytes / fu["fwd_grad_maps"]["device_ms"] / 1e6, 1),
                                "bwd": round(bwd_bytes / bwd_ms / 1e6, 1) if bwd_ms > 0 else None},
        "abs_diff_vs_torch_fp32": diff,
    }


def step_cost(warmup):
    sys.path.insert(0, ROOT)
    import bench
    from deblurgs_b200.graph import BlurryViewGraph
    dev = torch.device("cuda", torch.cuda.current_device())
    w = bench.build_workload("c2", 0, dev)
    gt = w["gt_host"].to(dev)
    steps = {lam: BlurryViewGraph(w["cmm"], 0, w["bg"], (3, w["H"], w["W"]), 0.0, lambda_dssim=lam)
             for lam in (0.0, 0.2)}
    for s in steps.values():
        s.step(gt)
        for _ in range(warmup):
            s.replay()
    torch.cuda.synchronize()
    per = {0.0: [], 0.2: []}
    for _ in range(ROUNDS):
        for lam, s in steps.items():
            per[lam].append(events_ms(s.replay, STEP_ITERS))
            s.check()
    base, with_ssim = statistics.median(per[0.0]), statistics.median(per[0.2])
    return {"config": "c2", "step_ms_lambda_dssim_0": round(base, 4), "step_ms_lambda_dssim_0.2": round(with_ssim, 4),
            "added_ms": round(with_ssim - base, 4), "rounds_ms": {str(k): [round(v, 4) for v in vs] for k, vs in per.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--no-step", action="store_true", help="skip the c2 training-step cost")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ssim needs a CUDA device")
    result = {"tool": "bench_ssim", **gpu_identity(), "iters": args.iters, "graph_calls": GRAPH_CALLS,
              "shapes": {name: bench_shape(name, shape, args.iters, args.warmup) for name, shape in SHAPES.items()}}
    if not args.no_step:
        result["step_cost"] = step_cost(args.warmup)
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
