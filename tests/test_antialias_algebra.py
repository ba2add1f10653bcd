"""CPU: the algebra of the antialiasing option (DESIGN.md section 3) and its C-ABI argument checks.

The per-Gaussian backward splits the gradient g of the stored opacity (opacity * rho) into dL/dopacity = rho g and a
gradient of the undilated 2-D covariance through r = det0 / det; its closed form, as the kernel evaluates it, is
checked here against float64 autograd of the oracle's rho, both where rho is clamped and where it is not."""
import ctypes as C

import numpy as np
import pytest
import torch

from deblurgs_b200 import _lib, synthetic
from oracle import pose_torch as pt, raster_aa_torch as ra, raster_torch_cpu as rt

H = 0.3
R_MIN = 2.5e-5


def _kernel_backward(a0, b, c0, opacity, g):
    """k_preprocess_bwd<*, true>'s arithmetic (dgs_backward.cu), elementwise in the dtype of its inputs:
    (dL/dopacity, dL/da0, dL/db, dL/dc0)."""
    a, c = a0 + H, c0 + H
    inv_det = 1.0 / (a * c - b * b)
    r = (a0 * c0 - b * b) * inv_det
    rho = torch.sqrt(torch.clamp_min(r, R_MIN))
    k = opacity * g * (0.5 * H) / rho * inv_det
    live = r > R_MIN
    da = torch.where(live, k * ((c0 * c + b * b) * inv_det), torch.zeros_like(k))
    dc = torch.where(live, k * ((a0 * a + b * b) * inv_det), torch.zeros_like(k))
    db = torch.where(live, -2.0 * k * (b * (a0 + c) * inv_det), torch.zeros_like(k))
    return rho * g, da, db, dc


def _covariances(n, seed):
    """2-D covariances from far below a pixel to hundreds of pixels, of every anisotropy and orientation, plus
    nearly degenerate ones whose r falls under the clamp."""
    g = torch.Generator().manual_seed(seed)
    s1 = 10.0 ** (torch.rand(n, generator=g, dtype=torch.float64) * 6 - 3.5)    # sigma^2 from 3e-4 to 300 px^2
    s2 = s1 * 10.0 ** (-torch.rand(n, generator=g, dtype=torch.float64) * 3)
    s2[: n // 8] = s1[: n // 8] * 1e-9                                            # degenerate: r below the clamp
    th = torch.rand(n, generator=g, dtype=torch.float64) * np.pi
    cs, sn = torch.cos(th), torch.sin(th)
    a0 = s1 * cs * cs + s2 * sn * sn
    c0 = s1 * sn * sn + s2 * cs * cs
    b = (s1 - s2) * cs * sn
    opacity = torch.rand(n, generator=g, dtype=torch.float64) * 0.98 + 0.01
    grad = torch.randn(n, generator=g, dtype=torch.float64)
    return a0, b, c0, opacity, grad


def test_closed_form_gradient_equals_float64_autograd():
    a0, b, c0, opacity, g = _covariances(4096, 0)
    leaves = [t.clone().requires_grad_(True) for t in (opacity, a0, b, c0)]
    (opacity_l, a0_l, b_l, c0_l) = leaves
    (opacity_l * ra.aa_rho(a0_l, b_l, c0_l) * g).sum().backward()
    auto = [t.grad for t in leaves]
    mine = _kernel_backward(a0, b, c0, opacity, g)
    clamped = (a0 * c0 - b * b) / ((a0 + H) * (c0 + H) - b * b) <= R_MIN
    assert 0 < int(clamped.sum()) < clamped.numel()            # both branches are exercised
    for m, t in zip(mine, auto):
        assert torch.allclose(m, t, rtol=1e-10, atol=1e-12 * t.abs().max().item())
    # the clamp branch: no covariance gradient, the opacity gradient scaled by sqrt(R_MIN)
    for t in auto[1:]:
        assert (t[clamped] == 0).all()
    assert torch.allclose(auto[0][clamped], np.sqrt(R_MIN) * g[clamped], rtol=1e-12)


def test_closed_form_is_the_stated_formula():
    """dr/d(a0, c0, b) = (c0 det - det0 c, a0 det - det0 a, 2 b (det0 - det)) / det^2, regrouped without cancellation."""
    a0, b, c0, _, _ = _covariances(2048, 1)
    a, c = a0 + H, c0 + H
    det0, det = a0 * c0 - b * b, a * c - b * b
    stated = [(c0 * det - det0 * c) / det ** 2, (a0 * det - det0 * a) / det ** 2, 2 * b * (det0 - det) / det ** 2]
    regrouped = [H * (c0 * c + b * b) / det ** 2, H * (a0 * a + b * b) / det ** 2, -2 * H * b * (a0 + c) / det ** 2]
    for s, r in zip(stated, regrouped):
        assert torch.allclose(s, r, rtol=1e-6, atol=1e-9 * r.abs().max().item())


def test_float32_closed_form_is_accurate():
    """In float32 (as the kernel runs it) the regrouped form stays within a few ulps of its float64 value, from
    sub-pixel to very large Gaussians: there is no cancelling difference in it.  (The one cancellation left is det0 =
    a0 c0 - b^2 of a nearly degenerate covariance, which is part of rho itself; those inputs are left out.)"""
    a0, b, c0, opacity, g = (t.float().double() for t in _covariances(4096, 2))
    keep = (a0 * c0 - b * b) > 0.1 * a0 * c0
    m32 = _kernel_backward(*(t.float() for t in (a0, b, c0, opacity, g)))
    m64 = _kernel_backward(a0, b, c0, opacity, g)
    for x, y in zip(m32, m64):
        err = ((x.double() - y).abs() / y.abs().clamp_min(1e-30))[keep & (y != 0)]
        assert err.max().item() < 2e-6, err.max().item()


def _tiny_inputs():
    P, W, Hh, F, order = synthetic.CONFIGS["tiny"]
    cam = synthetic.make_camera(W, Hh)
    sc = synthetic.make_scene(P, cam)
    traj = synthetic.make_trajectory(F, order)
    v, p, c = pt.trajectory(traj.ctrl_trans, traj.ctrl_rot, traj.nu, cam.projection_matrix_t())[0]
    return cam, sc, v.float(), p.float(), c.float(), synthetic.make_background()


def test_oracle_with_rho_forced_to_one_is_the_default_path(monkeypatch):
    cam, sc, v, p, c, bg = _tiny_inputs()
    W, Hh = cam.width, cam.height
    img0, _, pl0, b0 = rt.render_view(sc.means3D, sc.scales, sc.rotations, sc.opacities, sc.shs, 3, v, p, c, bg, W,
                                      Hh, cam.tanfovx, cam.tanfovy)
    monkeypatch.setattr(ra, "aa_rho", lambda a0, b, c0: torch.ones_like(a0))
    img1, pre1 = ra.render_view(sc.means3D, sc.opacities, v, p, bg, W, Hh, cam.tanfovx, cam.tanfovy,
                                antialiasing=True, scales=sc.scales, rots=sc.rotations, shs=sc.shs, deg=3, campos=c)
    assert torch.equal(img0, img1)
    pl1, b1 = rt.bin_tiles(pre1)
    assert torch.equal(pl0, pl1) and torch.equal(b0, b1)


def test_oracle_antialiasing_changes_only_the_opacity():
    cam, sc, v, p, c, bg = _tiny_inputs()
    kw = dict(scales=sc.scales.double(), rots=sc.rotations.double(), shs=sc.shs.double(), deg=3, campos=c.double())
    args = (sc.means3D.double(), sc.opacities.double(), v.double(), p.double(), cam.width, cam.height,
            cam.tanfovx, cam.tanfovy)
    off = ra.project(*args, antialiasing=False, **kw)
    on = ra.project(*args, antialiasing=True, **kw)
    for k in ("px", "py", "depth", "conic", "rgb", "radius"):
        assert torch.equal(off[k], on[k])
    assert torch.equal(on["opac"], off["opac"] * on["rho"])
    assert (on["rho"] > 0).all() and (on["rho"] < 1).all()


def _forward_aa_call(lib, aa, n, cb, one):
    return lib.dgs_blur_forward_aa(cb, None, cb, None, cb, None, 10, 1, 3, 16, one, 32, 32, one, one, None, one, one,
                                   1.0, one, None, one, one, one, 1.0, 1.0, 0.2, 100.0, 0, 0, one, one, one, None,
                                   1.0, 0, C.byref(n), aa, None)


def _backward_aa_call(lib, aa, one):
    return lib.dgs_blur_backward_range_aa(10, 1, 3, 16, 5, one, 32, 32, one, one, None, one, one, 1.0, one, None,
                                          one, one, one, 1.0, 1.0, 0.2, 100.0, 0, one, one, one, one, one, None, None,
                                          1.0, one, None, one, one, one, one, one, None, None, one, one, None, 0, 10,
                                          7, aa, None)


@pytest.mark.parametrize("aa", [2, -1, 255])
def test_antialiasing_outside_0_1_is_rejected_before_device_work(aa):
    lib = _lib.load()
    n = C.c_int64(0)
    cb = _lib.ALLOC_FN(lambda ctx, nbytes: 0)
    one = C.c_void_p(1)    # never dereferenced: validation fails first
    assert _forward_aa_call(lib, aa, n, cb, one) == -1 and b"antialiasing" in lib.dgs_last_error()
    assert _backward_aa_call(lib, aa, one) == -1 and b"antialiasing" in lib.dgs_last_error()


def test_antialiased_entries_keep_the_other_argument_checks():
    lib = _lib.load()
    n = C.c_int64(0)
    cb = _lib.ALLOC_FN(lambda ctx, nbytes: 0)
    one = C.c_void_p(1)
    # both SHs and precomputed colours, as in test_cabi, through the antialiased forward
    rc = lib.dgs_blur_forward_aa(cb, None, cb, None, cb, None, 10, 1, 3, 16, one, 32, 32, one, one, one, one, one,
                                 1.0, one, None, one, one, one, 1.0, 1.0, 0.2, 100.0, 0, 0, one, one, one, None, 1.0,
                                 0, C.byref(n), 1, None)
    assert rc == -1 and b"exactly one" in lib.dgs_last_error()
    # a Gaussian range outside [0, P)
    rc = lib.dgs_blur_backward_range_aa(10, 1, 3, 16, 5, one, 32, 32, one, one, None, one, one, 1.0, one, None,
                                        one, one, one, 1.0, 1.0, 0.2, 100.0, 0, one, one, one, one, one, None, None,
                                        1.0, one, None, one, one, one, one, one, None, None, one, one, None, 0, 11,
                                        7, 1, None)
    assert rc == -1 and b"range" in lib.dgs_last_error()


def test_python_surface_defaults_to_off():
    import inspect
    from deblurgs_b200 import rasterizer as rz
    from deblurgs_b200.motion import GaussianParams
    assert len(rz.GaussianRasterizationSettings._fields) == 13
    for fn in (rz.rasterize_gaussians, rz.rasterize_blurry, rz.render_store_blurry, GaussianParams.__init__,
               rz.GaussianRasterizer.__init__):
        assert inspect.signature(fn).parameters["antialiasing"].default is False
