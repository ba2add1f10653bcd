#!/usr/bin/env python
"""The blend backward (k_render_bwd, DESIGN.md section 3): how many (warp, list entry) pairs it replays, and its time.

Pairs: one forward of the view at each config; over every list entry inside the tile ranges, its hand-over byte b
(bit 2 * band + column half: which 8x4 rectangles of the tile blended the entry) counts
  popc(b)                      (8x4 rectangle, entry) pairs  -- a warp per 8x4 rectangle
  popc((b | b >> 2) & 0x33)    (8x8 block, entry) pairs      -- a warp per 8x8 block: bits 4 strip + c and 4 strip + 2 + c
and their ratio.  Every such pair is one gathered and replayed entry of the warp that owns the rectangle or block.

Time: the eager training step (photometric loss, so the DEPTH = false instantiation) with the library's stage profiler
on (dgs_profile_*: CUDA events around each launch); render_bwd is k_render_bwd alone, mean ms per launch over
PROFILE_ITERS steps, median of ROUNDS rounds.  The geometry records the kernel gathers are 3 x 16 B x F x P (230 MB at
c2, 768 MB at c3), larger than the 126 MB L2, and the forward between two launches evicts what was left.

  python tools/bench_blend_bwd.py [--configs c2,c3] [--out profiles/bench_blend_bwd_b200.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_antialias import gpu_identity, read_stages  # noqa: E402
from deblurgs_b200 import _lib, rasterizer  # noqa: E402
from deblurgs_b200.loss import training_loss  # noqa: E402

ROUNDS, PROFILE_ITERS = 5, 20
TILE = 16


def _aligned(t):
    """The library places its buffers at the first 128-byte boundary of the tensor it is given."""
    return t[(-t.data_ptr()) % 128:]


def pair_counts(w):
    """(8x4 pairs, 8x8 pairs, list entries) over all sub-frames of one forward of the view."""
    captured = []
    fwd = rasterizer._forward_batched

    def capture(*a, **k):
        out = fwd(*a, **k)
        captured.append(out)
        return out

    rasterizer._forward_batched = capture
    try:
        with torch.no_grad():
            w["cmm"].query(0, "all", background=w["bg"])
    finally:
        rasterizer._forward_batched = fwd
    torch.cuda.synchronize()
    W, H = w["W"], w["H"]
    tiles = ((W + TILE - 1) // TILE) * ((H + TILE - 1) // TILE)
    n4 = n8 = entries = 0
    for (color, _d, _r, _b, _D, _geom, binning, img) in captured:
        F = color.shape[0]
        bin_u8, img_u8 = _aligned(binning), _aligned(img)
        wmask_off = int(bin_u8[:8].view(torch.int64).item())        # BinHeader.wmask_offset
        wmask = bin_u8[wmask_off:]
        ranges = img_u8[:F * tiles * 8].view(torch.int32).view(F * tiles, 2).long() & 0xFFFFFFFF
        live = ranges[:, 1] != 0                                      # (~start, end); (0, 0) = empty tile
        start = (~ranges[live, 0]) & 0xFFFFFFFF
        length = ranges[live, 1] - start
        total = int(length.sum().item())
        first = torch.repeat_interleave(start - (torch.cumsum(length, 0) - length), length)
        b = wmask[first + torch.arange(total, device=first.device)].long()
        n4 += int(sum(((b >> i) & 1).sum().item() for i in range(8)))
        m = (b | (b >> 2)) & 0x33
        n8 += int(sum(((m >> i) & 1).sum().item() for i in (0, 1, 4, 5)))
        entries += total
    return n4, n8, entries


def render_bwd_ms(w, warmup):
    lib = _lib.load()
    dev = w["bg"].device
    gt = w["gt_host"].to(dev)
    store, cmm = w["gaussians"], w["cmm"]
    params = store.parameters() + cmm.parameters()

    def step():
        for p in params:
            p.grad = None
        out = cmm.query(0, "all", background=w["bg"])
        training_loss(out["blurred"], out["subframes"], gt).backward()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    per = []
    for _ in range(ROUNDS):
        lib.dgs_profile_read(None, None, 0, 1)
        lib.dgs_profile_enable(1)
        for _ in range(PROFILE_ITERS):
            step()
        torch.cuda.synchronize()
        st = read_stages(lib)
        lib.dgs_profile_enable(0)
        per.append(st["render_bwd"] / PROFILE_ITERS)
    return statistics.median(per), per


def measure(config, warmup):
    dev = torch.device("cuda", torch.cuda.current_device())
    w = bench.build_workload(config, 0, dev)
    n4, n8, entries = pair_counts(w)
    ms, per = render_bwd_ms(w, warmup)
    return {"config": config, "P": w["P"], "W": w["W"], "H": w["H"], "F": w["F"], "list_entries": entries,
            "pairs_8x4": n4, "pairs_8x8": n8, "ratio_8x8_8x4": round(n8 / max(n4, 1), 4),
            "render_bwd_ms": round(ms, 4), "rounds_ms": [round(v, 4) for v in per]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_blend_bwd needs a CUDA device")
    result = {"tool": "bench_blend_bwd", **gpu_identity(), "rounds": ROUNDS, "profile_iters": PROFILE_ITERS,
              "configs": [measure(c, args.warmup) for c in args.configs.split(",")]}
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
