"""Torch restatement of the contribution scores (include/dgs_b200.h, dgs_blur_forward_contrib): per Gaussian, the sum
and the maximum of its blending weights w = alpha * T over every pixel where it blended.

The compositing is raster_torch_cpu.composite's, line for line; where that function forms the per-(entry, pixel)
weight tensor `wgt` for the colour sum, this one scatters it onto the Gaussian ids instead.  The working precision is
that of the projection dict (float64 for the tests)."""
import torch

from . import raster_aa_torch as ra
from . import raster_torch_cpu as rt


@torch.no_grad()
def contribution(pre, point_list, bounds, W, H, chunk_pairs=6_000_000):
    """(weight_sum [P], weight_max [P], blended pixel count [P]) of one view."""
    P = pre["px"].shape[0]
    dtype = pre["px"].dtype
    wsum = torch.zeros(P, dtype=dtype)
    wmax = torch.zeros(P, dtype=dtype)
    nblend = torch.zeros(P, dtype=torch.int64)
    tiles_x, tiles_y = pre["tiles"]
    n_tiles = tiles_x * tiles_y
    lens = bounds[1:] - bounds[:-1]
    TILE = rt.TILE
    lx = torch.arange(TILE).repeat(TILE).to(dtype)
    ly = torch.arange(TILE).repeat_interleave(TILE).to(dtype)
    t0 = 0
    while t0 < n_tiles:
        t1 = t0 + 1
        kmax = int(lens[t0])
        while t1 < n_tiles and max(kmax, int(lens[t1])) * (t1 + 1 - t0) * 256 <= chunk_pairs:
            kmax = max(kmax, int(lens[t1]))
            t1 += 1
        K = max(kmax, 1)
        pos = bounds[t0:t1, None] + torch.arange(K)[None]
        valid = torch.arange(K)[None] < lens[t0:t1, None]
        if point_list.numel() == 0:
            t0 = t1
            continue
        gid = point_list[torch.where(valid, pos, torch.zeros_like(pos)).clamp(max=point_list.numel() - 1)]
        tiles = torch.arange(t0, t1)
        pixx = ((tiles % tiles_x) * TILE)[:, None].to(dtype) + lx[None]
        pixy = ((tiles // tiles_x) * TILE)[:, None].to(dtype) + ly[None]
        dx = pre["px"][gid][:, :, None] - pixx[:, None, :]
        dy = pre["py"][gid][:, :, None] - pixy[:, None, :]
        con = pre["conic"][gid]
        power = -0.5 * (con[:, :, 0:1] * dx * dx + con[:, :, 2:3] * dy * dy) - con[:, :, 1:2] * dx * dy
        alpha = torch.clamp_max(pre["opac"][gid][:, :, None] * torch.exp(power), 0.99)
        ok = valid[:, :, None] & (power <= 0) & (alpha >= 1.0 / 255.0)
        inside = ((pixx < W) & (pixy < H))[:, None, :]
        a = torch.where(ok & inside, alpha, torch.zeros_like(alpha))
        T_incl = torch.cumprod(1 - a, dim=1)
        stopped = torch.cummax(((T_incl < 1e-4) & ok).to(torch.uint8), dim=1).values.bool()
        a = torch.where(stopped, torch.zeros_like(a), a)
        T_incl = torch.cumprod(1 - a, dim=1)
        T_excl = T_incl / (1 - a)
        wgt = a * T_excl                                                          # [nt,K,256]
        g = gid.reshape(-1)
        keep = valid.reshape(-1)
        wgt2 = wgt.reshape(-1, 256)[keep]
        g = g[keep]
        wsum.index_add_(0, g, wgt2.sum(1))
        wmax.scatter_reduce_(0, g, wgt2.amax(1), reduce="amax")
        nblend.index_add_(0, g, (wgt2 > 0).sum(1))
        t0 = t1
    return wsum, wmax, nblend


@torch.no_grad()
def contribution_view(means, opac, view, proj, W, H, tanx, tany, antialiasing=False, **inputs):
    """Scores of one sub-frame from the raw inputs (those of raster_aa_torch.render_view).  The tile lists sort on
    float32 depth bits, as the library does."""
    pre = ra.project(means, opac, view, proj, W, H, tanx, tany, antialiasing=antialiasing, **inputs)
    point_list, bounds = rt.bin_tiles(dict(pre, depth=pre["depth"].float()))
    return contribution(pre, point_list, bounds, W, H)
