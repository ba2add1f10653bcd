#!/usr/bin/env python
"""Cost of Mip-Splatting's 3-D smoothing filter (DESIGN.md section 3): the sampling-depth sweep and the training step.

Sweep: k_filter3d_depth over 32 views of F sub-frames each at c2 scale (300k Gaussians, F = 16) and c4 scale (3M,
F = 32), the synthetic scene seen from 32 trajectories around the base pose.  `sweep_kernel_ms` times the kernel alone
on precomputed poses (CUDA events, mean of SWEEP_ITERS sweeps of all 32 * F cameras); `compute_3D_filter_ms` the
whole `CameraMotionModule.compute_3D_filter` (32 pose launches, the sweep and the finalisation with its one host
synchronisation), host clock around a synchronised call.

Step: BlurryViewGraph at c2 (300k, 600x400, 16 sub-frames) and c3 (1M, 1920x1080, 16), one graph captured with the
filter off and one with it on (computed from the workload's own view); replays alternated in ROUNDS rounds of
STEP_ITERS, the median per-step time of each and their ratio, and the duplicate count D (list entries) of each.  The
activations read 4 more bytes per Gaussian; the larger cost is that filtered Gaussians are wider, touch more tiles and
blend more entries.  Per-stage times (library stage profiler) separate the two at c2.

  python tools/bench_filter3d.py [--out profiles/bench_filter3d_b200.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_antialias import events_ms, gpu_identity, read_stages  # noqa: E402
from deblurgs_b200 import _lib, synthetic  # noqa: E402
from deblurgs_b200.filter3d import SamplingDepth  # noqa: E402
from deblurgs_b200.graph import BlurryViewGraph  # noqa: E402
from deblurgs_b200.loss import training_loss  # noqa: E402
from deblurgs_b200.motion import CameraMotionModule, GaussianParams  # noqa: E402

ROUNDS, STEP_ITERS, PROFILE_ITERS, SWEEP_ITERS, VIEWS = 5, 50, 20, 20, 32
STAGES = ("activate_fwd", "preprocess_fwd", "render_fwd", "render_bwd", "preprocess_bwd", "activate_bwd")


def sweep_cost(P, F, dev):
    _, W, H, _, order = synthetic.CONFIGS["c2"]
    cam = synthetic.make_camera(W, H)
    scene = synthetic.make_scene(P, cam, seed=0).to(dev)
    store = GaussianParams.from_scene(scene)
    base = torch.tensor([synthetic.BASE_SE3], dtype=torch.float32, device=dev).repeat(VIEWS, 1)
    ref = bench.RefCamera(cam, dev)
    cmm = CameraMotionModule([ref] * VIEWS, base, curve_order=order, num_subframes=F)
    with torch.no_grad():
        for i in range(VIEWS):
            t = synthetic.make_trajectory(F, order, seed=100 + i).to(dev)
            cmm._trans._control_points[i].copy_(t.ctrl_trans)
            cmm._rot._control_points[i].copy_(t.ctrl_rot)
    cmm.link_gaussian(store)
    with torch.no_grad():
        views = torch.cat([cmm.get_trajectory_tensors(i)[0] for i in range(VIEWS)])
    depth = SamplingDepth(P, dev)

    def sweep():
        depth.add(store._xyz, views, W, H, cam.fovx, cam.fovy, store.z_near)

    for _ in range(3):
        sweep()
    kernel_ms = events_ms(sweep, SWEEP_ITERS)
    times = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        f = cmm.compute_3D_filter()
        torch.cuda.synchronize()
        times.append(1e3 * (time.perf_counter() - t0))
    seen = int(torch.isfinite(depth.min_depth).sum())
    return {"P": P, "F": F, "views": VIEWS, "cameras": VIEWS * F, "sweep_kernel_ms": round(kernel_ms, 4),
            "compute_3D_filter_ms": round(statistics.median(times[1:]), 4), "gaussians_seen": seen,
            "filter_median": float(f.median()), "ns_per_pair": round(1e6 * kernel_ms / (P * VIEWS * F), 5)}


def kernel_profile(w, gt, filt, warmup):
    """Per-stage device ms of one eager step, filter off and on, alternated."""
    lib = _lib.load()
    store, cmm = w["gaussians"], w["cmm"]
    params = store.parameters() + cmm.parameters()

    def step():
        for p in params:
            p.grad = None
        out = cmm.query(0, "all", background=w["bg"])
        training_loss(out["blurred"], out["subframes"], gt).backward()

    per = {False: {s: [] for s in STAGES}, True: {s: [] for s in STAGES}}
    for on in (False, True):
        store.filter_3D = filt if on else None
        for _ in range(warmup):
            step()
    torch.cuda.synchronize()
    for _ in range(ROUNDS):
        for on in (False, True):
            store.filter_3D = filt if on else None
            lib.dgs_profile_read(None, None, 0, 1)
            lib.dgs_profile_enable(1)
            for _ in range(PROFILE_ITERS):
                step()
            torch.cuda.synchronize()
            st = read_stages(lib)
            lib.dgs_profile_enable(0)
            for s in STAGES:
                per[on][s].append(st[s] / PROFILE_ITERS)
    return {("filter_on" if on else "filter_off"): {s: round(statistics.median(v), 4) for s, v in d.items()}
            for on, d in per.items()}


def step_cost(config, warmup):
    dev = torch.device("cuda", torch.cuda.current_device())
    w = bench.build_workload(config, 0, dev)
    gt = w["gt_host"].to(dev)
    store, cmm = w["gaussians"], w["cmm"]
    filt = cmm.compute_3D_filter()
    graphs = {}
    for on in (False, True):
        store.filter_3D = filt if on else None      # read when the step is captured
        graphs[on] = BlurryViewGraph(cmm, 0, w["bg"], (3, w["H"], w["W"]), 0.0)
    losses, dup = {}, {}
    for on, g in graphs.items():
        store.filter_3D = filt if on else None      # a captured step replays only with the filter it was captured with
        losses[on] = g.step(gt)
        dup[on] = g.num_rendered()
        for _ in range(warmup):
            g.replay()
    torch.cuda.synchronize()
    per = {False: [], True: []}
    for _ in range(ROUNDS):
        for on, g in graphs.items():
            store.filter_3D = filt if on else None
            per[on].append(events_ms(g.replay, STEP_ITERS))
            g.check()
    off, on = statistics.median(per[False]), statistics.median(per[True])
    res = {"config": config, "P": w["P"], "W": w["W"], "H": w["H"], "F": w["F"],
           "step_ms_filter_off": round(off, 4), "step_ms_filter_on": round(on, 4), "ratio_on_off": round(on / off, 4),
           "D_filter_off": dup[False], "D_filter_on": dup[True], "D_ratio": round(dup[True] / dup[False], 4),
           "loss_filter_off": losses[False], "loss_filter_on": losses[True],
           "filter_median": float(filt.median()), "scale_min_median": float(store.get_scaling.min(1).values.median()),
           "rounds_ms": {"filter_off": [round(v, 4) for v in per[False]],
                         "filter_on": [round(v, 4) for v in per[True]]}}
    del graphs
    if config == "c2":
        res["kernels_ms_per_step"] = kernel_profile(w, gt, filt, warmup)
    store.filter_3D = None
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_filter3d needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    result = {"tool": "bench_filter3d", **gpu_identity(), "rounds": ROUNDS, "step_iters": STEP_ITERS,
              "sweep": [sweep_cost(300_000, 16, dev), sweep_cost(3_000_000, 32, dev)],
              "steps": [step_cost(c, args.warmup) for c in args.configs.split(",")]}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
