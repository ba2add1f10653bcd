"""The blend backward's pixel geometry (k_render_bwd: a warp per 8x8 block, two rows per lane) against the float64
evaluation of the same backward (oracle/truth_bwd.cu), on scenes chosen for the cases that geometry has to get right:
images whose width and height are not multiples of 8, an image smaller than one tile, entries blended in only one
8x4 half of a block, blocks whose two rows per lane stop at different entries, tile lists that span several 32-entry
steps, and the instantiation with a depth-image gradient.  Each case checks that its scene really contains what it is
meant to exercise, then compares the per-(sub-frame, Gaussian) screen-space gradients the blend backward writes."""
import pytest
import torch

from tests import parity_utils as pu
from deblurgs_b200 import rasterizer as rz, synthetic
from oracle import ref_cuda

pytestmark = pytest.mark.gpu

# name: W, H, P, Gaussian size (sigma in pixels), sub-frames, depth-image gradient
CASES = {
    "below_one_tile": (13, 7, 40, 3.0, 2, False),
    "odd_size_long_lists": (93, 61, 3000, 2.0, 2, False),
    "small_gaussians": (64, 40, 4000, 0.5, 2, False),
    "depth_gradient": (93, 61, 3000, 2.0, 2, True),
}


def _inputs(W, H, P, sigma, F, seed):
    cam = synthetic.make_camera(W, H)
    scene = synthetic.make_scene(P, cam, seed=seed, sigma_px=sigma).to("cuda")
    traj = synthetic.make_trajectory(F, 9, seed=seed + 1).to("cuda")
    bg = synthetic.make_background().to("cuda")
    view, proj, campos = pu.bezier_se3_poses(traj.ctrl_trans, traj.ctrl_rot, traj.nu,
                                             cam.projection_matrix_t().to("cuda"))
    return cam, scene, bg, view.contiguous(), proj.contiguous(), campos.contiguous()


def _aligned(t):
    return t[(-t.data_ptr()) % 128:]          # the library places its buffers at the first 128-byte boundary


def _handover_bytes(fw, s, tiles):
    """Hand-over bytes of sub-frame s's list entries (one per entry, written by the forward for the backward)."""
    b, img = _aligned(fw["binning"]), _aligned(fw["img"])
    off = int(b[:8].view(torch.int64).item())            # BinHeader.wmask_offset
    r = img[:fw["color"].shape[0] * tiles * 8].view(torch.int32).view(-1, tiles, 2)[s].long() & 0xFFFFFFFF
    r = r[r[:, 1] != 0]                                   # (~start, end); (0, 0) = empty tile
    pos = torch.cat([torch.arange(int(~a & 0xFFFFFFFF), int(e), device=b.device) for a, e in r.tolist()])
    return b[off:][pos].long()


@pytest.mark.parametrize("name", list(CASES))
def test_blend_backward_blocks_against_float64(name, capsys):
    W, H, P, sigma, F, with_depth = CASES[name]
    cam, scene, bg, view, proj, campos = _inputs(W, H, P, sigma, F, seed=11)
    fw = pu.ours_forward(cam, scene, bg, view, proj, campos)
    g = torch.Generator().manual_seed(5)
    gt = torch.rand(3, H, W, generator=g).cuda()
    dpix = (torch.sign(fw["blur"] - gt) / (3 * H * W * F))[None].expand(F, 3, H, W).contiguous()
    ddep = (torch.randn(F, 1, H, W, generator=g) / (H * W)).cuda() if with_depth else None
    rz._KEEP_SCRATCH = True
    try:
        pu.ours_backward(cam, scene, bg, view, proj, campos, fw, dpix, ddep)
        off = (-rz._last_scratch.data_ptr()) % 128
        planes = rz._last_scratch[off:off + P * F * 48].view(torch.float32).view(3, F, P, 4)     # g0 | g1 | g2
        mine2d = torch.cat((planes[0], planes[1], planes[2]), dim=-1)
    finally:
        rz._KEEP_SCRATCH = False
    dec = pu.ours_decode(fw, P, F, W, H)
    zeros = torch.zeros(F, 1, H, W, device="cuda")
    errs, seen = {}, {"one_half_only": 0, "rows_differ": 0, "max_list": 0}
    base = 0
    for s in range(F):
        R = int(dec["tiles_touched"][s].sum())
        ranges = dec["ranges"][s].clone()
        ranges[ranges[:, 1] > ranges[:, 0]] -= base
        t2d = ref_cuda.truth_blend_backward(W, H, ranges, dec["point_list"][base:base + R], dec["means2D"][s],
                                            dec["conic_opacity"][s], dec["rgb"][s], dec["depths"][s],
                                            dec["n_contrib"][s], bg, dpix[s], (ddep if with_depth else zeros)[s])
        # what the scene exercises: entries one 8x8 block blended in only one of its 8x4 halves, lanes whose two
        # rows stop at different entries, lists over several 32-entry steps of the backward
        b = _handover_bytes(fw, s, dec["ranges"].shape[1])
        for k in (0, 1, 4, 5):
            half = b & (5 << k)
            seen["one_half_only"] += int(((half == (1 << k)) | (half == (4 << k))).sum())
        nc = dec["n_contrib"][s]
        Hp = (H + 7) // 8 * 8
        ncp = torch.zeros(Hp, W, dtype=nc.dtype, device=nc.device)
        ncp[:H] = nc
        blocks = ncp.view(Hp // 8, 2, 4, W)                         # [block row][upper / lower half][row][x]
        seen["rows_differ"] += int((blocks[:, 0] != blocks[:, 1]).sum())
        seen["max_list"] = max(seen["max_list"], int((dec["ranges"][s][:, 1] - dec["ranges"][s][:, 0]).max()))
        base += R
        vis = fw["radii"][s] > 0
        comp = {"dmean2D": (mine2d[s][:, 0:2], t2d[0]), "dconic": (mine2d[s][:, 2:5], t2d[1]),
                "dopacity": (mine2d[s][:, 5], t2d[2]), "dcolor": (mine2d[s][:, 8:11], t2d[3])}
        if with_depth:
            comp["ddepth"] = (mine2d[s][:, 6], t2d[4])
        for k, (mo, to) in comp.items():
            errs[k] = max(errs.get(k, 0.0), pu.rel_err(mo[vis], to[vis]))
    with capsys.disabled():
        print("\n%s (%dx%d, P=%d): %s  per-element error against float64 (floor 1e-3 of the max): %s"
              % (name, W, H, P, seen, " ".join("%s %.2e" % kv for kv in errs.items())))
    assert seen["rows_differ"] > 0
    if name == "small_gaussians":
        assert seen["one_half_only"] > 0
    if name in ("odd_size_long_lists", "depth_gradient"):
        assert seen["max_list"] > 96
    bad = {k: e for k, e in errs.items() if not e <= 1e-3}
    assert not bad, (bad, errs)
