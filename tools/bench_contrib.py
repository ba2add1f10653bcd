#!/usr/bin/env python
"""Cost of the contribution scores (DESIGN.md section 3) and what pruning by them buys per training step.

Blend kernel: at c2 (300k Gaussians, 600x400, 16 sub-frames) and c3 (1M, 1920x1080, 16), the eager no-grad forward of
one blurry view with the library's stage profiler on (dgs_profile_*: CUDA events around each stage); render_fwd is
k_render_fwd without scores and k_render_fwd_contrib with them.  Both settings alternated in ROUNDS rounds of
PROFILE_ITERS forwards; per-forward median ms of each and their ratio.

Sweep: one CameraMotionModule.accumulate_contribution over the view (all its sub-frames, scores included), CUDA events,
mean of SWEEP_ITERS.

Pruning: the c2 store scored over its view, then 0 %, 30 % and 60 % of it removed by weight sum
(prune_by_contribution); for each, the graph-replayed training step (BlurryViewGraph), median of ROUNDS rounds of
STEP_ITERS replays.

  python tools/bench_contrib.py [--out profiles/bench_contrib_b200.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_antialias import events_ms, gpu_identity, read_stages  # noqa: E402
from deblurgs_b200 import _lib, renderer  # noqa: E402
from deblurgs_b200.graph import BlurryViewGraph  # noqa: E402
from deblurgs_b200.motion import GaussianParams  # noqa: E402
from deblurgs_b200.rasterizer import ContributionScores  # noqa: E402

ROUNDS, PROFILE_ITERS, SWEEP_ITERS, STEP_ITERS = 5, 20, 20, 50


def blend_cost(config, warmup):
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    w = bench.build_workload(config, 0, dev)
    cmm, store, bg = w["cmm"], w["gaussians"], w["bg"]
    scores = ContributionScores(w["P"], dev)
    with torch.no_grad():
        view, proj, campos = cmm.get_trajectory_tensors(0)

    def forward(score):
        with torch.no_grad():
            renderer.render_blurry(view, proj, campos, cmm.original_cam[0], store, bg,
                                   contrib=scores if score else None)

    for score in (False, True):
        for _ in range(warmup):
            forward(score)
    torch.cuda.synchronize()
    per = {False: [], True: []}
    for _ in range(ROUNDS):
        for score in (False, True):
            lib.dgs_profile_read(None, None, 0, 1)
            lib.dgs_profile_enable(1)
            for _ in range(PROFILE_ITERS):
                forward(score)
            torch.cuda.synchronize()
            st = read_stages(lib)
            lib.dgs_profile_enable(0)
            per[score].append(st["render_fwd"] / PROFILE_ITERS)
    off, on = statistics.median(per[False]), statistics.median(per[True])
    sweep = events_ms(lambda: cmm.accumulate_contribution(bg, scores=scores), SWEEP_ITERS)
    return {"config": config, "P": w["P"], "W": w["W"], "H": w["H"], "F": w["F"],
            "render_fwd_ms_plain": round(off, 4), "render_fwd_ms_scoring": round(on, 4),
            "ratio_scoring_plain": round(on / off, 4), "sweep_ms_one_view": round(sweep, 4),
            "rounds_ms": {"plain": [round(v, 4) for v in per[False]], "scoring": [round(v, 4) for v in per[True]]}}


def pruned_step_cost(config, fractions, warmup):
    dev = torch.device("cuda", torch.cuda.current_device())
    w = bench.build_workload(config, 0, dev)
    gt = w["gt_host"].to(dev)
    cmm = w["cmm"]
    scores = cmm.accumulate_contribution(w["bg"])
    out = []
    for frac in fractions:
        store = GaussianParams.from_scene(w["scene"])
        store.training_setup()
        store.prune_by_contribution(scores, fraction=frac)
        store.optimizer = None
        cmm.link_gaussian(store)
        g = BlurryViewGraph(cmm, 0, w["bg"], (3, w["H"], w["W"]), 0.0)
        loss = g.step(gt)
        for _ in range(warmup):
            g.replay()
        torch.cuda.synchronize()
        per = []
        for _ in range(ROUNDS):
            per.append(events_ms(g.replay, STEP_ITERS))
            g.check()
        out.append({"fraction": frac, "P": store.get_xyz.shape[0], "step_ms": round(statistics.median(per), 4),
                    "loss": loss, "rounds_ms": [round(v, 4) for v in per]})
        del g
    return {"config": config, "steps": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--prune-config", default="c2")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_contrib needs a CUDA device")
    result = {"tool": "bench_contrib", **gpu_identity(), "rounds": ROUNDS, "profile_iters": PROFILE_ITERS,
              "blend": [blend_cost(c, args.warmup) for c in args.configs.split(",")],
              "pruning": pruned_step_cost(args.prune_config, (0.0, 0.3, 0.6), args.warmup)}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
