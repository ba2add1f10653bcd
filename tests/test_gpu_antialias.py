"""GPU: the antialiasing option (Mip-Splatting's screen-space filter, DESIGN.md section 3).

With antialiasing the per-Gaussian forward stores opacity * rho instead of the opacity and nothing else of the
geometry record changes, so binning is identical; images and gradients follow the float64 torch oracle
(oracle/raster_aa_torch.py); a sub-pixel Gaussian keeps its integrated weight when the image is rendered smaller;
batched and single-view renders agree; and a CUDA-graph replay of an antialiased store equals the eager step."""
import math

import numpy as np
import pytest
import torch

from tests import parity_utils as pu
from deblurgs_b200 import rasterizer as rz
from oracle import raster_aa_torch as ra

pytestmark = pytest.mark.gpu


def _forward(cam, scene, bg, view, proj, campos, aa, colors=None, cov3D=None):
    shs = None if colors is not None else scene.shs
    scales = None if cov3D is not None else scene.scales
    rots = None if cov3D is not None else scene.rotations
    color, depth, radii, blur, D, geom, binning, img = rz._forward_batched(
        scene.means3D, shs, colors, scene.opacities, scales, rots, cov3D, view, proj, campos, bg, cam.height,
        cam.width, cam.tanfovx, cam.tanfovy, 1.0, 0.2, 100.0, scene.sh_degree, False, False, True,
        float(view.shape[0]), exact=True, antialiasing=aa)
    return dict(color=color, depth=depth, radii=radii, blur=blur, num_rendered=D, geom=geom, binning=binning, img=img)


def _cov3d_upper(scene):
    S = ra.cov3d_from_scale_rot(scene.scales.double(), scene.rotations.double())
    return torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], 1).float().contiguous()


def _colors(P, dev):
    g = torch.Generator().manual_seed(5)
    return torch.rand(P, 3, generator=g).to(dev)


@pytest.mark.parametrize("name", ["small", "c1"])
def test_same_binning_and_conics_with_and_without_antialiasing(name):
    cam, scene, _, bg, view, proj, campos = pu.make_inputs(name, F=3)
    P, F, W, H = scene.means3D.shape[0], view.shape[0], cam.width, cam.height
    off = _forward(cam, scene, bg, view, proj, campos, False)
    on = _forward(cam, scene, bg, view, proj, campos, True)
    assert off["num_rendered"] == on["num_rendered"] > 0
    assert torch.equal(off["radii"], on["radii"])
    d0, d1 = pu.ours_decode(off, P, F, W, H), pu.ours_decode(on, P, F, W, H)
    for k in ("tiles_touched", "point_offsets", "point_list", "ranges", "keys", "means2D", "depths", "rgb"):
        assert torch.equal(d0[k], d1[k]), k
    assert torch.equal(d0["conic_opacity"][..., :3], d1["conic_opacity"][..., :3])
    vis = off["radii"] > 0
    assert (d1["conic_opacity"][..., 3][vis] < d0["conic_opacity"][..., 3][vis]).all()


@pytest.mark.parametrize("name,kind", [("small", "sh"), ("small", "cov3D"), ("c1", "sh")])
def test_stored_opacity_is_opacity_times_rho(name, kind):
    cam, scene, _, bg, view, proj, campos = pu.make_inputs(name, F=3)
    P, F, W, H = scene.means3D.shape[0], view.shape[0], cam.width, cam.height
    cov3D = _cov3d_upper(scene) if kind == "cov3D" else None
    fw = _forward(cam, scene, bg, view, proj, campos, True, cov3D=cov3D)
    dec = pu.ours_decode(fw, P, F, W, H)
    worst = 0.0
    for s in range(F):
        inputs = dict(cov3D=cov3D.double().cpu()) if cov3D is not None else \
            dict(scales=scene.scales.double().cpu(), rots=scene.rotations.double().cpu())
        pre = ra.project(scene.means3D.double().cpu(), scene.opacities.double().cpu(), view[s].double().cpu(),
                         proj[s].double().cpu(), W, H, cam.tanfovx, cam.tanfovy, colors=torch.zeros(P, 3,
                         dtype=torch.float64), antialiasing=True, **inputs)
        vis = (fw["radii"][s] > 0).cpu()
        got = dec["conic_opacity"][s, :, 3].cpu().double()[vis]
        want = pre["opac"][vis]
        worst = max(worst, ((got - want).abs() / want).max().item())
    assert worst < 1e-4, worst


def _library_render(cam, scene, bg, view, proj, campos, kind, aa):
    """rasterize_blurry through autograd; returns (color [F,3,H,W], leaves dict)."""
    dev = scene.means3D.device
    leaves = {"means3D": scene.means3D.clone(), "opacities": scene.opacities.clone()}
    if kind == "cov3D":
        leaves["cov3D"] = _cov3d_upper(scene)
    else:
        leaves["scales"], leaves["rotations"] = scene.scales.clone(), scene.rotations.clone()
    if kind == "colors":
        leaves["colors"] = _colors(scene.means3D.shape[0], dev)
    else:
        leaves["shs"] = scene.shs.clone()
    for t in leaves.values():
        t.requires_grad_(True)
    rs = rz.GaussianRasterizationSettings(cam.height, cam.width, cam.tanfovx, cam.tanfovy, bg, 1.0, 0.2, 100.0, False,
                                          scene.sh_degree, campos, False, False)
    color, _, radii, _ = rz.rasterize_blurry(
        leaves["means3D"], None, leaves.get("shs"), leaves.get("colors"), leaves["opacities"], leaves.get("scales"),
        leaves.get("rotations"), leaves.get("cov3D"), view, proj, campos, rs, antialiasing=aa)
    return color, leaves


@pytest.mark.parametrize("name,kind", [("small", "sh"), ("small", "colors"), ("small", "cov3D"), ("c1", "sh")])
def test_images_and_gradients_match_float64_oracle(name, kind):
    cam, scene, _, bg, view, proj, campos = pu.make_inputs(name, F=2 if name == "small" else 1)
    F, W, H = view.shape[0], cam.width, cam.height
    color, leaves = _library_render(cam, scene, bg, view, proj, campos, kind, True)
    wgt = torch.randn(F, 3, H, W, generator=torch.Generator().manual_seed(9)).cuda() / (3 * H * W)
    (color * wgt).sum().backward()
    torch.cuda.synchronize()
    ref = {k: v.detach().double().cpu().requires_grad_(True) for k, v in leaves.items()}
    inputs = {"cov3D": ref.get("cov3D"), "scales": ref.get("scales"), "rots": ref.get("rotations"),
              "colors": ref.get("colors"), "shs": ref.get("shs"), "deg": scene.sh_degree}
    inputs = {k: v for k, v in inputs.items() if v is not None}
    loss, imgs = 0.0, []
    for s in range(F):
        img, _ = ra.render_view(ref["means3D"], ref["opacities"], view[s].double().cpu(), proj[s].double().cpu(),
                                bg.double().cpu(), W, H, cam.tanfovx, cam.tanfovy, antialiasing=True,
                                campos=campos[s].double().cpu(), **inputs)
        imgs.append(img.detach())
        loss = loss + (img * wgt[s].double().cpu()).sum()
    loss.backward()
    err = (color.detach().cpu().double() - torch.stack(imgs)).abs()
    assert torch.quantile(err.flatten()[::7], 0.999).item() < 1e-4 and err.max().item() < 2e-2, err.max().item()
    for k, t in ref.items():
        mine = leaves[k].grad.detach().cpu().double()
        rel = (mine - t.grad).abs().max().item() / max(t.grad.abs().max().item(), 1e-30)
        assert rel < 5e-3, (k, rel)


def _single_gaussian(W, H, sigma_px):
    """One Gaussian facing the camera (view = identity), flat in z so that its screen covariance is exactly
    sigma_px^2 I, at the pixel centre (W * 9/16 - 0.5, H * 5/12 - 0.5): for W x H = 128 x 96 that is the centre of a
    16x16 tile, and at W/2 x H/2 it is 3.5 px inside one, so every pixel above the 1/255 cut-off is blended."""
    from deblurgs_b200 import synthetic
    cam = synthetic.make_camera(W, H)
    z = 5.0
    fx = W / (2 * cam.tanfovx)
    ndc_x = (2 * (W * 9 / 16 - 0.5) + 1) / W - 1
    ndc_y = (2 * (H * 5 / 12 - 0.5) + 1) / H - 1
    mean = torch.tensor([[ndc_x * cam.tanfovx * z, ndc_y * cam.tanfovy * z, z]])
    s2 = (sigma_px * z / fx) ** 2
    cov3D = torch.tensor([[s2, 0.0, 0.0, s2 * (fx / (H / (2 * cam.tanfovy))) ** 2, 0.0, 0.0]])
    view = torch.eye(4)
    proj = cam.projection_matrix_t()
    return cam, mean, cov3D, view, proj


def _sum_alpha(W, H, sigma_px, aa):
    cam, mean, cov3D, view, proj = _single_gaussian(W, H, sigma_px)
    dev = torch.device("cuda", 0)
    opac = torch.tensor([[0.9]])
    ones = torch.ones(1, 3)
    bg = torch.zeros(3)
    rs = rz.GaussianRasterizationSettings(H, W, cam.tanfovx, cam.tanfovy, bg.to(dev), 1.0, 0.2, 100.0, False, 0,
                                          torch.zeros(3, device=dev), False, False)
    img, _, radii = rz.rasterize_gaussians(mean.to(dev), None, None, ones.to(dev), opac.to(dev), None, None,
                                           cov3D.to(dev), view.to(dev), proj.to(dev), rs, antialiasing=aa)
    assert int(radii[0]) > 0
    got = img[0].double().sum().item()
    # float64 evaluation at the same pixel centres: same projection (oracle), 1/255 cut-off, 0.99 clamp
    pre = ra.project(mean.double(), opac.double(), view.double(), proj.double(), W, H, cam.tanfovx, cam.tanfovy,
                     cov3D=cov3D.double(), colors=ones.double(), antialiasing=aa)
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    dx, dy = pre["px"][0] - xs, pre["py"][0] - ys
    con = pre["conic"][0]
    power = -0.5 * (con[0] * dx * dx + con[2] * dy * dy) - con[1] * dx * dy
    alpha = torch.clamp_max(pre["opac"][0] * torch.exp(power), 0.99)
    alpha = torch.where((power <= 0) & (alpha >= 1.0 / 255.0), alpha, torch.zeros_like(alpha))
    want = alpha.sum().item()
    assert abs(got - want) <= 1e-3 * want, (W, aa, got, want)
    return got


def test_antialiasing_keeps_the_integrated_weight_of_a_subpixel_gaussian():
    W, H = 128, 96
    full_aa, half_aa = _sum_alpha(W, H, 1.0, True), _sum_alpha(W // 2, H // 2, 0.5, True)
    full, half = _sum_alpha(W, H, 1.0, False), _sum_alpha(W // 2, H // 2, 0.5, False)
    # alpha integrated over the image, in pixels of the full-size image: a pixel at W/2 covers four of them
    assert abs(4.0 * half_aa / full_aa - 1.0) < 0.05, (full_aa, 4 * half_aa)
    assert 4.0 * half / full > 1.5, (full, 4 * half)          # analytically (0.25 + 0.3) * 4 / 1.3 = 1.69
    assert abs(full_aa / (0.9 * 2 * math.pi) - 1.0) < 0.05    # opacity x 2 pi sigma^2 with sigma = 1 px


def test_batched_render_equals_single_view_renders():
    cam, scene, _, bg, view, proj, campos = pu.make_inputs("small", F=3)
    F = view.shape[0]
    color, leaves = _library_render(cam, scene, bg, view, proj, campos, "sh", True)
    wgt = torch.randn(F, 3, cam.height, cam.width, generator=torch.Generator().manual_seed(4)).cuda()
    (color * wgt).sum().backward()
    batched = {k: v.grad.clone() for k, v in leaves.items()}
    for v in leaves.values():
        v.grad = None
    for s in range(F):
        rs = rz.GaussianRasterizationSettings(cam.height, cam.width, cam.tanfovx, cam.tanfovy, bg, 1.0, 0.2, 100.0,
                                              False, scene.sh_degree, campos[s], False, False)
        img, _, _ = rz.GaussianRasterizer(rs, antialiasing=True)(
            leaves["means3D"], torch.zeros_like(leaves["means3D"]), leaves["opacities"], shs=leaves["shs"],
            scales=leaves["scales"], rotations=leaves["rotations"], viewmatrix=view[s], projmatrix=proj[s])
        assert (img.detach() - color[s].detach()).abs().max().item() <= 1e-6
        (img * wgt[s]).sum().backward()
    for k, v in leaves.items():
        rel = (v.grad - batched[k]).abs().max().item() / batched[k].abs().max().item()
        assert rel <= 1e-4, (k, rel)


def test_graph_replay_of_an_antialiased_store_equals_eager_step():
    import bench
    from deblurgs_b200.graph import BlurryViewGraph
    from deblurgs_b200.loss import blur_photometric_loss
    dev = torch.device("cuda", 0)
    w = bench.build_workload("small", 0, dev)
    store, cmm = w["gaussians"], w["cmm"]
    params = store.parameters() + cmm.parameters()
    gt = w["gt_host"].to(dev)
    with torch.no_grad():
        plain = cmm.query(0, "all", background=w["bg"])["blurred"].clone()
    store.antialiasing = True
    with torch.no_grad():
        assert (cmm.query(0, "all", background=w["bg"])["blurred"] - plain).abs().max().item() > 1e-3

    def eager():
        for p in params:
            p.grad = None
        out = cmm.query(0, "all", background=w["bg"])
        loss = blur_photometric_loss(out["blurred"], out["subframes"], gt, 0.0)
        loss.backward()
        torch.cuda.synchronize()
        return loss.item(), [p.grad.clone() for p in params]

    g = BlurryViewGraph(cmm, 0, w["bg"], (3, w["H"], w["W"]), 0.0)
    l_ref, g_ref = eager()
    val = g.step(gt)
    assert abs(val - l_ref) <= 1e-6
    for p, r in zip(params, g_ref):
        assert ((p.grad - r).abs().max() / r.abs().max().clamp_min(1e-30)).item() <= 1e-3
    assert np.isfinite(val)
    # the flag is part of the captured step: a replay after it changed refuses instead of rendering the old setting
    store.antialiasing = False
    with pytest.raises(Exception, match="antialiasing"):
        g.step(gt)
