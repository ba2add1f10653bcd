#!/usr/bin/env python
"""Cost of the antialiasing option (Mip-Splatting's screen-space filter, DESIGN.md section 3) on the training step.

Step time: BlurryViewGraph at c2 (300k Gaussians, 600x400, 16 sub-frames) and c3 (1M, 1920x1080, 16), one graph
captured with the store's antialiasing off and one with it on; replays alternated in ROUNDS rounds of STEP_ITERS, the
median per-step time of each and their ratio.  Antialiasing changes the code of the two per-Gaussian kernels only (one
4-byte load and ~20 flops per visible pair); the blend kernels run the same code on the same lists, but with the
lower opacities fewer pixels reach the transmittance cut-off early, so they blend more list entries.  The per-stage
times below separate the two effects.

Kernels: the eager step with the library's stage profiler on (dgs_profile_*: CUDA events around each stage), per
stage mean ms over PROFILE_ITERS steps, both settings alternated.  preprocess_fwd is k_preprocess_fwd; preprocess_bwd
is the per-Gaussian backward (k_preprocess_bwd + k_sh_bwd) plus the view / projection-gradient finish; render_fwd and
render_bwd are the two blend kernels.

  python tools/bench_antialias.py [--out profiles/bench_antialias_b200.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from deblurgs_b200 import _lib  # noqa: E402
from deblurgs_b200.graph import BlurryViewGraph  # noqa: E402
from deblurgs_b200.loss import training_loss  # noqa: E402

ROUNDS, STEP_ITERS, PROFILE_ITERS = 5, 50, 20
STAGES = ("preprocess_fwd", "render_fwd", "render_bwd", "preprocess_bwd")


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


def read_stages(lib):
    n = lib.dgs_profile_num_stages()
    ms, calls = (C.c_double * n)(), (C.c_int64 * n)()
    _lib.check(lib.dgs_profile_read(ms, calls, n, 1), "dgs_profile_read")
    return {lib.dgs_profile_stage_name(i).decode(): ms[i] for i in range(n)}


def kernel_profile(w, gt, warmup):
    """Per-stage device ms of one eager step, antialiasing off and on, alternated."""
    lib = _lib.load()
    store, cmm = w["gaussians"], w["cmm"]
    params = store.parameters() + cmm.parameters()

    def step():
        for p in params:
            p.grad = None
        out = cmm.query(0, "all", background=w["bg"])
        training_loss(out["blurred"], out["subframes"], gt).backward()

    per = {False: {s: [] for s in STAGES}, True: {s: [] for s in STAGES}}
    for aa in (False, True):
        store.antialiasing = aa
        for _ in range(warmup):
            step()
    torch.cuda.synchronize()
    for _ in range(ROUNDS):
        for aa in (False, True):
            store.antialiasing = aa
            lib.dgs_profile_read(None, None, 0, 1)
            lib.dgs_profile_enable(1)
            for _ in range(PROFILE_ITERS):
                step()
            torch.cuda.synchronize()
            st = read_stages(lib)
            lib.dgs_profile_enable(0)
            for s in STAGES:
                per[aa][s].append(st[s] / PROFILE_ITERS)
    return {("aa_on" if aa else "aa_off"): {s: round(statistics.median(v), 4) for s, v in d.items()}
            for aa, d in per.items()}


def step_cost(config, warmup):
    dev = torch.device("cuda", torch.cuda.current_device())
    w = bench.build_workload(config, 0, dev)
    gt = w["gt_host"].to(dev)
    store = w["gaussians"]
    graphs = {}
    for aa in (False, True):
        store.antialiasing = aa            # read when the step is captured
        graphs[aa] = BlurryViewGraph(w["cmm"], 0, w["bg"], (3, w["H"], w["W"]), 0.0)
    losses = {}
    for aa, g in graphs.items():
        store.antialiasing = aa            # a captured step replays only with the flag it was captured with
        losses[aa] = g.step(gt)
        for _ in range(warmup):
            g.replay()
    torch.cuda.synchronize()
    per = {False: [], True: []}
    for _ in range(ROUNDS):
        for aa, g in graphs.items():
            store.antialiasing = aa
            per[aa].append(events_ms(g.replay, STEP_ITERS))
            g.check()
    off, on = statistics.median(per[False]), statistics.median(per[True])
    res = {"config": config, "P": w["P"], "W": w["W"], "H": w["H"], "F": w["F"],
           "step_ms_aa_off": round(off, 4), "step_ms_aa_on": round(on, 4), "ratio_on_off": round(on / off, 4),
           "loss_aa_off": losses[False], "loss_aa_on": losses[True],
           "rounds_ms": {"aa_off": [round(v, 4) for v in per[False]], "aa_on": [round(v, 4) for v in per[True]]}}
    del graphs
    if config == "c2":
        res["kernels_ms_per_step"] = kernel_profile(w, gt, warmup)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_antialias needs a CUDA device")
    result = {"tool": "bench_antialias", **gpu_identity(), "rounds": ROUNDS, "step_iters": STEP_ITERS,
              "steps": [step_cost(c, args.warmup) for c in args.configs.split(",")]}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
