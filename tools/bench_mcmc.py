#!/usr/bin/env python
"""Cost of 3DGS-MCMC densification (DESIGN.md section 3, csrc/dgs_mcmc.cu) and what it does to training.

noise       k_mcmc_noise at 300k, 1M and 3M Gaussians (56 B each: 17 MB at 300k fits the 126 MB L2 and is read from there
            after the first launch; 3M = 168 MB does not), CUDA events around NOISE_ITERS launches, against the torch
            statement of the original (build_scaling_rotation, L L^T, randn, bmm, add) on the same store.
relocation  one `relocate_gs` round (5 % of the rows dead; sampling, ratio and the two-kernel launch) and one
            `add_new_gs` round (5 % growth: sampling, the row-gather rebuild and the relocation), host clock around a
            synchronised call, median of ROUNDS, at the same sizes.  Store: synthetic scene, SH degree 3, Adam moments on.
regularise  loss.mcmc_regularization forward + backward at 300k (two torch reductions), CUDA events.
graph       the graph-replayed c2 step (bench.py's workload) before and after an in-place relocation of 5 % of the rows,
            replays alternated in ROUNDS rounds of STEP_ITERS; the duplicate count D of each.
example     examples/train_blurry_views.py with the default densification and with --mcmc: PSNR / SSIM before -> after
            of the sharp mid-exposure views and the final Gaussian count.

  python tools/bench_mcmc.py [--out profiles/bench_mcmc_b200.json]
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_antialias import events_ms, gpu_identity  # noqa: E402
from deblurgs_b200 import mcmc, synthetic  # noqa: E402
from deblurgs_b200.densify import build_rotation  # noqa: E402
from deblurgs_b200.graph import BlurryViewGraph  # noqa: E402
from deblurgs_b200.loss import mcmc_regularization  # noqa: E402
from deblurgs_b200.motion import GaussianParams  # noqa: E402

ROUNDS, STEP_ITERS, NOISE_ITERS = 5, 50, 200
SIZES = (300_000, 1_000_000, 3_000_000)
LR, NOISE_LR = 1.6e-4, 5e5


def make_store(P, dev):
    cam = synthetic.make_camera(600, 400)
    store = GaussianParams.from_scene(synthetic.make_scene(P, cam, seed=0).to(dev))
    opt = store.training_setup()
    for grp in opt.param_groups:
        p = grp["params"][0]
        opt.state[p] = {"step": 1, "exp_avg": torch.zeros_like(p), "exp_avg_sq": torch.zeros_like(p)}
    store._ensure_stats()
    return store


def torch_noise(store, step_scale):
    """The original's statement (3DGS-MCMC train.py): L = R S, cov = L L^T, noise = randn * gate * lr scale, bmm, add."""
    with torch.no_grad():
        L = build_rotation(store.get_rotation) * store.get_scaling[:, None, :]
        cov = L @ L.transpose(1, 2)
        gate = 1.0 / (1.0 + torch.exp(-mcmc.NOISE_K * ((1.0 - store.get_opacity) - mcmc.NOISE_X0)))
        noise = torch.randn_like(store._xyz) * gate * step_scale
        store._xyz.add_(torch.bmm(cov, noise[:, :, None])[:, :, 0])


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), out


def store_cost(P, dev):
    store = make_store(P, dev)
    step = [0]

    def kernel():
        step[0] += 1
        mcmc.add_sgld_noise(store, LR, step[0], NOISE_LR)

    for _ in range(5):
        kernel()
        torch_noise(store, NOISE_LR * LR)
    kernel_ms = events_ms(kernel, NOISE_ITERS)
    torch_ms = events_ms(lambda: torch_noise(store, NOISE_LR * LR), max(NOISE_ITERS // 10, 5))
    gen = torch.Generator().manual_seed(0)
    reloc, n_dead = [], P // 20
    for _ in range(ROUNDS + 1):
        with torch.no_grad():
            store._opacity[torch.randperm(P, generator=gen)[:n_dead].to(dev)] = 0.0
        ms, n = timed(lambda: store.relocate_gs(generator=gen))
        assert n == n_dead
        reloc.append(ms)
    grow = []
    for _ in range(3):
        ms, n = timed(lambda: store.add_new_gs(10 ** 12, generator=gen))
        grow.append((ms, n))
    res = {"P": P, "noise_kernel_ms": round(kernel_ms, 5), "noise_torch_ms": round(torch_ms, 4),
           "noise_speedup": round(torch_ms / kernel_ms, 2),
           "noise_GBps": round(56 * P / (kernel_ms * 1e-3) / 1e9, 1),
           "relocate_rows": n_dead, "relocate_round_ms": round(statistics.median(reloc[1:]), 3),
           "grow_rows": grow[-1][1], "grow_round_ms": round(statistics.median([g[0] for g in grow[1:]]), 3)}
    if P == SIZES[0]:
        def reg():
            for p in (store._opacity, store._scaling):
                p.grad = None
            mcmc_regularization(store).backward()
        for _ in range(5):
            reg()
        res["regularization_fwd_bwd_ms"] = round(events_ms(reg, 100), 4)
    return res


def graph_cost(warmup):
    dev = torch.device("cuda", torch.cuda.current_device())
    w = bench.build_workload("c2", 0, dev)
    store = w["gaussians"]
    store.training_setup()
    gt = w["gt_host"].to(dev)
    g = BlurryViewGraph(w["cmm"], 0, w["bg"], (3, w["H"], w["W"]), 0.0)
    res = {"config": "c2", "P": w["P"], "W": w["W"], "H": w["H"], "F": w["F"]}
    res["loss_before"] = g.step(gt)
    res["D_before"] = g.num_rendered()
    for _ in range(warmup):
        g.replay()
    before = [events_ms(g.replay, STEP_ITERS) for _ in range(ROUNDS)]
    g.check()
    dead = torch.zeros(w["P"], dtype=torch.bool, device=dev)
    dead[torch.randperm(w["P"], generator=torch.Generator().manual_seed(0))[: w["P"] // 20].to(dev)] = True
    res["relocated"] = store.relocate_gs(dead_mask=dead, generator=torch.Generator().manual_seed(1))
    res["loss_after"] = g.step(gt)
    res["D_after"] = g.num_rendered()
    for _ in range(warmup):
        g.replay()
    after = [events_ms(g.replay, STEP_ITERS) for _ in range(ROUNDS)]
    g.check()
    res.update(step_ms_before=round(statistics.median(before), 4), step_ms_after=round(statistics.median(after), 4),
               recaptures=g.recaptures, rounds_ms={"before": [round(v, 4) for v in before],
                                                   "after": [round(v, 4) for v in after]})
    return res


def example_run(extra):
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train_blurry_views.py")] + extra
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("%s failed:\n%s\n%s" % (" ".join(cmd), r.stdout[-3000:], r.stderr[-3000:]))
    out = {"args": extra, "wall_s": round(time.perf_counter() - t0, 1)}
    for line in r.stdout.splitlines():
        m = re.search(r"(full|half|double) size .*PSNR ([\d.]+) -> ([\d.]+) dB, SSIM ([\d.]+) -> ([\d.]+)", line)
        if m:
            out[m.group(1)] = {"psnr": [float(m.group(2)), float(m.group(3))],
                               "ssim": [float(m.group(4)), float(m.group(5))]}
        m = re.search(r"-> (\d+) Gaussians", line)
        if m:
            out["final_gaussians"] = int(m.group(1))
        m = re.search(r"loss ([\d.]+) -> ([\d.]+)", line)
        if m:
            out["loss"] = [float(m.group(1)), float(m.group(2))]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mcmc needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    result = {"tool": "bench_mcmc", **gpu_identity(), "rounds": ROUNDS, "noise_iters": NOISE_ITERS,
              "noise_lr": NOISE_LR, "lr": LR, "stores": [store_cost(P, dev) for P in SIZES],
              "graph": graph_cost(args.warmup),
              "example": {"default": example_run([]), "mcmc": example_run(["--mcmc"])}}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
