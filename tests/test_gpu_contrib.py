"""GPU: per-Gaussian contribution scores (include/dgs_b200.h, dgs_blur_forward_contrib).

The scoring forward changes nothing else the forward produces; the weight sums conserve the rendered opacity; they
follow a float64 torch oracle (oracle/contrib_torch.py); they are exact and order-independent across calls, batchings
and the speculative forward's re-run; removing the Gaussians that scored zero leaves every scored view unchanged; and
pruning by score damages the image far less than pruning at random."""
import types

import numpy as np
import pytest
import torch

from tests import parity_utils as pu
from deblurgs_b200 import rasterizer as rz, renderer
from deblurgs_b200.motion import GaussianParams
from oracle import contrib_torch as ct

pytestmark = pytest.mark.gpu


def _fwd(cam, scene, bg, view, proj, campos, aa=False, contrib=None, colors=None, exact=True):
    shs = None if colors is not None else scene.shs
    color, depth, radii, blur, D, geom, binning, img = rz._forward_batched(
        scene.means3D, shs, colors, scene.opacities, scene.scales, scene.rotations, None, view, proj, campos, bg, cam.height,
        cam.width, cam.tanfovx, cam.tanfovy, 1.0, 0.2, 100.0, scene.sh_degree, False, False, True,
        float(view.shape[0]), exact=exact, antialiasing=aa, contrib=contrib)
    return dict(color=color, depth=depth, radii=radii, blur=blur, num_rendered=D, geom=geom, binning=binning, img=img)


def _scores(P):
    return rz.ContributionScores(P, "cuda")


def _handover_bytes(fw, n_contrib, W, H):
    """(positions, bytes) of the hand-over bytes the backward reads: those of every tile's list entries up to the
    deepest contributor of its pixels (n_contrib: last blended 1-based list position per pixel, [F,H,W]).  Bytes past
    it may never be written: the forward stops staging a tile once all its pixels are done.  The tile ranges are the
    first array of the image buffer, stored as (~start, end); the byte array's offset is the binning buffer's 64-bit
    header."""
    F = n_contrib.shape[0]
    tx, ty = (W + 15) // 16, (H + 15) // 16
    nc = torch.zeros(F, ty * 16, tx * 16, dtype=torch.int64)
    nc[:, :H, :W] = n_contrib.cpu().long()
    deepest = nc.view(F, ty, 16, tx, 16).amax(dim=(2, 4)).reshape(-1).numpy()        # [F * tiles], tile = y * tx + x
    img, b = fw["img"], fw["binning"]
    ib, bb = (-img.data_ptr()) % 128, (-b.data_ptr()) % 128
    rng = img[ib:ib + F * tx * ty * 8].view(torch.int32).view(-1, 2).cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    off = int(b[bb:bb + 8].view(torch.int64).item())
    live = rng[:, 1] != 0
    starts = (~rng[live, 0]) & 0xFFFFFFFF
    ends = np.minimum(rng[live, 1], starts + deepest[live])
    pos = np.concatenate([np.arange(s, e) for s, e in zip(starts, ends)]) if live.any() else np.zeros(0, np.int64)
    wm = b[bb + off:bb + off + int(ends.max() if live.any() else 0)].cpu().numpy()
    return pos, wm[pos]


def _grads(cam, scene, bg, view, proj, campos, fw, aa, dL):
    out = rz._backward_batched(scene.means3D.shape[0], view.shape[0], scene.shs.shape[1], fw["num_rendered"],
                               scene.means3D, scene.shs, None, scene.opacities, scene.scales, scene.rotations, None,
                               view, proj, campos, bg, cam.height, cam.width, cam.tanfovx, cam.tanfovy, 1.0, 0.2, 100.0,
                               scene.sh_degree, False, fw["radii"], fw["geom"], fw["binning"], fw["img"], dL, None,
                               True, antialiasing=aa)
    torch.cuda.synchronize()
    return [t for t in out if t is not None]


@pytest.mark.parametrize("aa", [False, True])
@pytest.mark.parametrize("name", ["small", "c1"])
def test_scoring_changes_nothing_else(name, aa):
    cam, scene, _, bg, view, proj, campos = pu.make_inputs(name, F=3)
    P, F, W, H = scene.means3D.shape[0], view.shape[0], cam.width, cam.height
    plain = _fwd(cam, scene, bg, view, proj, campos, aa)
    sc = _scores(P)
    scored = _fwd(cam, scene, bg, view, proj, campos, aa, contrib=sc)
    assert int(sc.wsum.sum()) > 0
    for k in ("color", "depth", "radii", "blur"):
        assert torch.equal(plain[k], scored[k]), k
    assert plain["num_rendered"] == scored["num_rendered"]
    d0, d1 = pu.ours_decode(plain, P, F, W, H), pu.ours_decode(scored, P, F, W, H)
    for k in ("final_T", "n_contrib", "point_list", "ranges", "keys"):
        assert torch.equal(d0[k], d1[k]), k
    p0, h0 = _handover_bytes(plain, d0["n_contrib"], W, H)
    p1, h1 = _handover_bytes(scored, d1["n_contrib"], W, H)
    assert np.array_equal(p0, p1) and 0 < p0.size <= plain["num_rendered"] and np.array_equal(h0, h1)
    assert h0.any()
    # gradients of a following backward: within the backward's own run-to-run spread (it reduces with float atomics)
    dL = torch.randn(F, 3, H, W, generator=torch.Generator().manual_seed(4)).cuda() / (H * W)
    ga = _grads(cam, scene, bg, view, proj, campos, plain, aa, dL)
    plain2 = _fwd(cam, scene, bg, view, proj, campos, aa)
    gb = _grads(cam, scene, bg, view, proj, campos, plain2, aa, dL)
    gc = _grads(cam, scene, bg, view, proj, campos, scored, aa, dL)
    for a, b, c in zip(ga, gb, gc):
        spread = (a - b).abs().max().item()
        floor = 1e-6 * a.abs().max().item()
        assert (c - a).abs().max().item() <= 4 * max(spread, floor), (spread, (c - a).abs().max().item())


@pytest.mark.parametrize("aa", [False, True])
@pytest.mark.parametrize("name", ["small", "c1"])
def test_weight_sum_conserves_the_rendered_opacity(name, aa):
    """Per pixel the kernel's weights telescope: sum_k alpha_k T_k = 1 - T_final up to the fp32 roundings of
    1 - alpha, T (1 - alpha) and alpha T (each at most 2^-24 relative, T <= 1: 3 * 2^-24 per blended entry) and the
    fixed-point rounding (2^-27 per blended entry).  n_contrib (last blended list position) bounds the number of blended
    entries of a pixel."""
    cam, scene, _, bg, view, proj, campos = pu.make_inputs(name, F=3)
    P, F, W, H = scene.means3D.shape[0], view.shape[0], cam.width, cam.height
    sc = _scores(P)
    fw = _fwd(cam, scene, bg, view, proj, campos, aa, contrib=sc)
    d = pu.ours_decode(fw, P, F, W, H)
    opacity = (1.0 - d["final_T"].double()).sum().item()
    total = sc.weight_sum.sum().item()
    n = d["n_contrib"].double().sum().item()
    bound = n * (3.01 * 2.0 ** -24 + 2.0 ** -27) + 1e-12 * opacity
    print("%s aa=%d: sum W = %.6f, sum (1 - T) = %.6f, |diff| = %.3g, bound %.3g" % (name, aa, total, opacity,
                                                                                      abs(total - opacity), bound))
    assert abs(total - opacity) <= bound


@pytest.mark.parametrize("name,kind,aa", [("small", "sh", False), ("small", "sh", True), ("small", "colors", False),
                                          ("small", "colors", True), ("c1", "sh", False), ("c1", "sh", True)])
def test_scores_match_float64_oracle(name, kind, aa):
    cam, scene, _, bg, view, proj, campos = pu.make_inputs(name, F=1)
    P, W, H = scene.means3D.shape[0], cam.width, cam.height
    colors = torch.rand(P, 3, generator=torch.Generator().manual_seed(5)).cuda() if kind == "colors" else None
    sc = _scores(P)
    _fwd(cam, scene, bg, view, proj, campos, aa, contrib=sc, colors=colors)
    inputs = dict(scales=scene.scales.double().cpu(), rots=scene.rotations.double().cpu())
    if colors is not None:
        inputs["colors"] = colors.double().cpu()
    else:
        inputs.update(shs=scene.shs.double().cpu(), deg=scene.sh_degree, campos=campos[0].double().cpu())
    ref_sum, ref_max, nblend = ct.contribution_view(scene.means3D.double().cpu(), scene.opacities.double().cpu(),
                                                    view[0].double().cpu(), proj[0].double().cpu(), W, H, cam.tanfovx,
                                                    cam.tanfovy, antialiasing=aa, **inputs)
    got_sum, got_max = sc.weight_sum.cpu(), sc.weight_max.cpu().double()
    err = (got_sum - ref_sum).abs()
    tol = 1e-4 * ref_sum.abs() + nblend.double() * 2.0 ** -27
    frac = (err <= tol).double().mean().item()
    err_max = (got_max - ref_max).abs()
    frac_max = (err_max <= 1e-4 * ref_max + 1e-9).double().mean().item()
    print("%s %s aa=%d: %.5f of sums within the bar (max abs err %.3g), %.5f of maxima (max abs err %.3g)"
          % (name, kind, aa, frac, err.max().item(), frac_max, err_max.max().item()))
    assert frac >= 0.999 and err.max().item() <= 5e-3
    assert frac_max >= 0.999 and err_max.max().item() <= 5e-3
    assert (got_sum[ref_sum > 1e-3] > 0).all()


def test_scores_are_exact_across_calls_batchings_and_the_speculative_rerun():
    cam, scene, _, bg, view, proj, campos = pu.make_inputs("small", F=3)
    P, F, W, H = scene.means3D.shape[0], view.shape[0], cam.width, cam.height
    a, b = _scores(P), _scores(P)
    _fwd(cam, scene, bg, view, proj, campos, contrib=a)
    _fwd(cam, scene, bg, view, proj, campos, contrib=b)
    assert torch.equal(a.wsum, b.wsum) and torch.equal(a.wmax, b.wmax) and int(a.wsum.sum()) > 0
    # batched F = 3 equals the sum (and max) of the three single-sub-frame calls
    singles = []
    for s in range(F):
        sc = _scores(P)
        _fwd(cam, scene, bg, view[s:s + 1], proj[s:s + 1], campos[s:s + 1], contrib=sc)
        singles.append(sc)
    assert torch.equal(a.wsum, sum(sc.wsum for sc in singles))
    assert torch.equal(a.wmax, torch.stack([sc.wmax for sc in singles]).max(0).values)
    # accumulating over two calls equals the sum of each
    acc = _scores(P)
    _fwd(cam, scene, bg, view[:1], proj[:1], campos[:1], contrib=acc)
    _fwd(cam, scene, bg, view[1:], proj[1:], campos[1:], contrib=acc)
    assert torch.equal(acc.wsum, a.wsum) and torch.equal(acc.wmax, a.wmax)
    # a speculative forward whose hint overflows blends empty lists first, then re-runs: no double count
    key = (torch.cuda.current_device(), P, F, H, W)
    rz._CAPACITY_HINT[key] = 1
    spec = _scores(P)
    fw = _fwd(cam, scene, bg, view, proj, campos, contrib=spec, exact=False)
    assert fw["num_rendered"] > 1
    assert torch.equal(spec.wsum, a.wsum) and torch.equal(spec.wmax, a.wmax)
    # ... and with nothing waited for (num_rendered == NULL), an overflowed call adds nothing
    saved = rz._ASYNC
    rz._ASYNC = {"capacity": 1, "geoms": []}
    try:
        none = _scores(P)
        _fwd(cam, scene, bg, view, proj, campos, contrib=none, exact=False)
        torch.cuda.synchronize()
    finally:
        rz._ASYNC = saved
    assert int(none.wsum.abs().sum()) == 0 and int(none.wmax.abs().sum()) == 0


def _ref_cam(cam):
    return types.SimpleNamespace(image_width=cam.width, image_height=cam.height, FoVx=cam.fovx, FoVy=cam.fovy)


def _store(scene, opacity_scale=1.0):
    gp = GaussianParams.from_scene(scene)
    with torch.no_grad():
        gp._opacity.mul_(opacity_scale)
    gp.training_setup()
    return gp


def _store_state(gp, cam, bg, view, proj, campos):
    """The store's batched forward with its state buffers (what renderer.render_blurry runs)."""
    shs, scales, rots, opac = gp.get_activated()
    st = types.SimpleNamespace(means3D=gp.get_xyz.detach(), shs=shs, scales=scales, rotations=rots, opacities=opac,
                               sh_degree=gp.active_sh_degree)
    return _fwd(cam, st, bg, view, proj, campos), st


def test_removing_zero_score_gaussians_changes_no_scored_view():
    cam, scene, _, bg, view, proj, campos = pu.make_inputs("small", F=5)
    gp = _store(scene, opacity_scale=0.03)
    P, F = gp.get_xyz.shape[0], view.shape[0]
    sc = _scores(P)
    with torch.no_grad():
        before = renderer.render_blurry(view, proj, campos, _ref_cam(cam), gp, bg, contrib=sc)
        fw, _ = _store_state(gp, cam, bg, view, proj, campos)
    assert torch.equal(fw["color"], before["render"])
    # precondition: every pixel ends with T > 0.0101, so T (1 - alpha) >= 0.0101 * 0.01 > 1e-4 for any candidate: no
    # pixel stops, and a Gaussian that blends nowhere then has no effect anywhere
    d = pu.ours_decode(fw, P, F, cam.width, cam.height)
    assert d["final_T"].min().item() > 0.0101, d["final_T"].min().item()
    zero = sc.wsum == 0
    assert 0 < int(zero.sum()) < P
    assert torch.equal(zero, sc.wmax == 0)
    mask = gp.prune_by_contribution(sc, min_weight_max=1e-38)
    assert torch.equal(mask, zero) and gp.get_xyz.shape[0] == P - int(zero.sum())
    with torch.no_grad():
        after = renderer.render_blurry(view, proj, campos, _ref_cam(cam), gp, bg)
    assert torch.equal(after["render"], before["render"])
    assert torch.equal(after["blurred"], before["blurred"])


def test_pruning_by_score_beats_random_pruning():
    cam, scene, _, bg, view, proj, campos = pu.make_inputs("small", F=5)
    ref = _store(scene)
    P = ref.get_xyz.shape[0]
    sc = _scores(P)
    with torch.no_grad():
        full = renderer.render_blurry(view, proj, campos, _ref_cam(cam), ref, bg, contrib=sc)["render"]
    by_score = _store(scene)
    by_score.prune_by_contribution(sc, fraction=0.3)
    rnd = _store(scene)
    g = torch.Generator().manual_seed(11)
    mask = torch.zeros(P, dtype=torch.bool)
    mask[torch.randperm(P, generator=g)[:int(0.3 * P)]] = True
    rnd.prune_points(mask.cuda())
    assert by_score.get_xyz.shape[0] == rnd.get_xyz.shape[0]
    with torch.no_grad():
        e_score = (renderer.render_blurry(view, proj, campos, _ref_cam(cam), by_score, bg)["render"] - full).abs().mean()
        e_rnd = (renderer.render_blurry(view, proj, campos, _ref_cam(cam), rnd, bg)["render"] - full).abs().mean()
    ratio = (e_score / e_rnd).item()
    print("mean |image error| after pruning 30%%: by score %.3g, at random %.3g, ratio %.3f"
          % (e_score.item(), e_rnd.item(), ratio))
    assert ratio < 0.5


@pytest.mark.timeout(600)
def test_sharded_scores_equal_unsharded_under_torchrun():
    """render_blurry_sharded + all_reduce_contribution against the unsharded scores (tests/dist_contrib_check.py): two
    ranks on a box with two GPUs, otherwise one rank, which still runs the sharded code path end to end."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n = 2 if torch.cuda.device_count() >= 2 else 1
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29575", os.path.join(root, "tests", "dist_contrib_check.py"),
           "small"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=540, cwd=root)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "contrib sharding OK" in r.stdout, r.stdout[-2000:]
