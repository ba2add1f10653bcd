"""CPU: Mip-Splatting's 3-D smoothing filter (include/dgs_b200.h, dgs_filter3d_depth / dgs_activate_*_filter3d): the
closed-form activation backward the kernel implements against float64 autograd of the torch statement, the per-axis
opacity factor against the determinant form, the finalisation of the sampling depth, the store operations that carry
the filter (rebuild plan, densification_postfix, reset_opacity), and the C-ABI argument checks."""
import ctypes as C
import inspect
import math

import pytest
import torch

from deblurgs_b200 import _lib
from deblurgs_b200 import rasterizer as rz
from deblurgs_b200.filter3d import SamplingDepth
from deblurgs_b200.motion import GaussianParams
from deblurgs_b200.params import activate_gaussians


def _statement(raw_s, raw_o, f, lb, iso):
    """The torch statement (GaussianParams.get_scaling_with_3D_filter / get_opacity_with_3D_filter)."""
    e = torch.exp(raw_s[:, :1].expand(-1, 3)) if iso else torch.exp(raw_s)
    s = e + lb
    sp = torch.sqrt(torch.square(s) + torch.square(f))
    r = s / sp
    return sp, raw_o.clamp(0.0, 1.0) * r[:, 0:1] * r[:, 1:2] * r[:, 2:3]


def _closed_form(raw_s, raw_o, f, lb, iso, gs, go):
    """k_activate_bwd<true>: dL/ds_i = g_s'_i r_i + g_o' clamp(o) prod_{j != i} r_j f^2 / s'_i^3, dL/dclamp(o) =
    g_o' prod r_j, then the exp / isotropic chain and the clamp mask."""
    e = torch.exp(raw_s[:, :1].expand(-1, 3)) if iso else torch.exp(raw_s)
    s = e + lb
    sp = torch.sqrt(s * s + f * f)
    r = s / sp
    oc = raw_o.clamp(0.0, 1.0)
    others = torch.stack([r[:, 1] * r[:, 2], r[:, 0] * r[:, 2], r[:, 0] * r[:, 1]], 1)
    ds = gs * r + go * oc * others * (f * f) / sp ** 3
    if iso:
        dscaling = torch.zeros_like(raw_s)
        dscaling[:, 0] = (ds * e).sum(1)
    else:
        dscaling = ds * e
    mask = ((raw_o >= 0) & (raw_o <= 1)).to(raw_o.dtype)
    dop = go * (r[:, 0:1] * r[:, 1:2] * r[:, 2:3]) * mask
    return dscaling, dop


def _case(kind, P=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    raw_s = torch.randn(P, 3, generator=g, dtype=torch.float64) - 4.0
    raw_o = torch.rand(P, 1, generator=g, dtype=torch.float64) * 1.4 - 0.2     # in and outside [0, 1]
    raw_o[:4, 0] = torch.tensor([0.0, 1.0, -0.1, 1.1], dtype=torch.float64)    # at and outside the clamp bounds
    s_typ = torch.exp(raw_s).mean().item()
    f = torch.rand(P, 1, generator=g, dtype=torch.float64) * s_typ
    if kind == "f_large":
        f = f * 1e3 + 10 * s_typ
    elif kind == "f_small":
        f = f * 1e-4
    elif kind == "tiny":
        raw_s = torch.full_like(raw_s, math.log(1e-7))
        f = torch.full_like(f, 1e-3)
    return raw_s, raw_o, f


@pytest.mark.parametrize("iso", [False, True])
@pytest.mark.parametrize("lb", [0.0, 0.004])
@pytest.mark.parametrize("kind", ["mixed", "f_large", "f_small", "tiny"])
def test_closed_form_backward_matches_float64_autograd(kind, lb, iso):
    raw_s, raw_o, f = _case(kind)
    rs, ro = raw_s.clone().requires_grad_(True), raw_o.clone().requires_grad_(True)
    sp, op = _statement(rs, ro, f, lb, iso)
    g = torch.Generator().manual_seed(3)
    gs = torch.randn(sp.shape, generator=g, dtype=torch.float64)
    go = torch.randn(op.shape, generator=g, dtype=torch.float64)
    torch.autograd.backward((sp, op), (gs, go))
    dscaling, dop = _closed_form(raw_s, raw_o, f, lb, iso, gs, go)
    assert torch.allclose(dscaling, rs.grad, rtol=1e-10, atol=1e-300), (dscaling - rs.grad).abs().max()
    assert torch.allclose(dop, ro.grad, rtol=1e-10, atol=0.0)
    # the clamp bounds pass the gradient, outside them it is zero
    assert dop[0, 0] != 0 and dop[1, 0] != 0 and dop[2, 0] == 0 and dop[3, 0] == 0
    if iso:
        assert (dscaling[:, 1:] == 0).all()


def test_per_axis_opacity_factor_survives_tiny_scales_in_fp32():
    s = torch.full((8, 3), 1e-7, dtype=torch.float32)
    f = torch.full((8, 1), 1e-3, dtype=torch.float32)
    exact = torch.sqrt(torch.tensor(1e-7, dtype=torch.float64) ** 2 /
                       (torch.tensor(1e-7, dtype=torch.float64) ** 2 + 1e-6)) ** 3
    # Mip-Splatting's sqrt(det1 / det2): prod(s_i^2) = 1e-42 is subnormal in fp32
    sq = torch.square(s)
    det = torch.sqrt(sq.prod(1) / (sq + torch.square(f)).prod(1))
    r = s / torch.sqrt(sq + torch.square(f))
    axis = r[:, 0] * r[:, 1] * r[:, 2]
    err_det = ((det.double() - exact).abs() / exact).max().item()
    err_axis = ((axis.double() - exact).abs() / exact).max().item()
    assert err_det > 1e-4, err_det
    assert err_axis < 1e-6, err_axis
    # one decade further the determinant form underflows to zero altogether
    s8 = torch.full((1, 3), 1e-8, dtype=torch.float32)
    assert torch.sqrt(torch.square(s8).prod(1) / (torch.square(s8) + torch.square(f[:1])).prod(1)).item() == 0.0
    r8 = s8 / torch.sqrt(torch.square(s8) + torch.square(f[:1]))
    assert (r8[:, 0] * r8[:, 1] * r8[:, 2]).item() > 0.0


def test_finalize_gives_unseen_gaussians_the_largest_finite_depth():
    d = SamplingDepth(5, "cpu")
    d.min_depth.copy_(torch.tensor([2.0, math.inf, 5.0, 3.0, math.inf]))
    d.max_focal = 400.0
    f = d.filter_3D()
    assert f.shape == (5, 1) and f.dtype == torch.float32
    want = torch.tensor([2.0, 5.0, 5.0, 3.0, 5.0]) / 400.0 * math.sqrt(0.2)
    assert torch.allclose(f[:, 0], want, rtol=1e-6, atol=0)


def test_finalize_of_an_all_unseen_store_raises():
    d = SamplingDepth(3, "cpu")
    d.max_focal = 100.0
    with pytest.raises(ValueError, match="no camera"):
        d.filter_3D()
    with pytest.raises(ValueError):
        SamplingDepth(0, "cpu").filter_3D()


def _store(P=10, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.rand(*s, generator=g)
    gp = GaussianParams(r(P, 3), r(P, 1, 3), r(P, 3, 3), r(P, 3) - 2.0, r(P, 4) + 0.1, r(P, 1), 1)
    gp.training_setup()
    gp.filter_3D = (torch.arange(P, dtype=torch.float32) + 1.0)[:, None] * 1e-3   # row id, recoverable
    return gp


def _rows(gp):
    return (gp.filter_3D[:, 0] * 1e3 - 1.0).round().long().tolist()


def test_rebuild_plan_carries_the_filter_for_prune():
    gp = _store()
    mask = torch.zeros(10, dtype=torch.bool)
    mask[[1, 4, 7]] = True
    gp.prune_points(mask)
    assert _rows(gp) == [0, 2, 3, 5, 6, 8, 9]
    assert gp.filter_3D.shape == (7, 1)


def test_rebuild_plan_carries_the_filter_for_clone_and_split():
    gp = _store()
    grads = torch.zeros(10, 1)
    grads[[2, 6]] = 1.0
    gp.densify_and_clone(grads, 0.5, 1e3)                 # every Gaussian is small against the extent: clone 2, 6
    assert _rows(gp) == list(range(10)) + [2, 6]
    gp = _store()
    gp.densify_and_split(grads, 0.5, 1e-3, N=2, generator=torch.Generator().manual_seed(0))   # all large: split 2, 6
    assert _rows(gp) == [0, 1, 3, 4, 5, 7, 8, 9, 2, 6, 2, 6]
    assert gp._xyz.shape[0] == gp.filter_3D.shape[0] == 12


def test_densification_postfix_zero_extends_the_filter():
    gp = _store()
    n = 3
    gp.densification_postfix(torch.zeros(n, 3), torch.zeros(n, 1, 3), torch.zeros(n, 3, 3), torch.zeros(n, 1),
                             torch.zeros(n, 3), torch.ones(n, 4))
    assert _rows(gp)[:10] == list(range(10))
    assert gp.filter_3D.shape == (13, 1) and (gp.filter_3D[10:] == 0).all()


def test_reset_opacity_caps_the_filtered_opacity():
    gp = _store(P=64, seed=2)
    with torch.no_grad():
        gp._opacity.copy_(torch.linspace(0.0, 1.0, 64)[:, None])
        gp._scaling.copy_(torch.log(torch.linspace(1e-4, 1e-2, 64))[:, None].expand(-1, 3))
        gp.filter_3D = torch.full((64, 1), 3e-3)
    before = gp.get_opacity_with_3D_filter.clone()
    assert (before < 0.1).any() and (before > 0.1).any()
    gp.reset_opacity(0.1)
    after = gp.get_opacity_with_3D_filter
    want = torch.clamp_max(before, 0.1)
    assert torch.allclose(after, want, rtol=1e-6, atol=0), (after - want).abs().max()
    # without the filter the cap applies to the clamped opacity, as before
    gp2 = _store(P=64, seed=2)
    with torch.no_grad():
        gp2._opacity.copy_(torch.linspace(0.0, 1.0, 64)[:, None])
    gp2.filter_3D = None
    gp2.reset_opacity(0.1)
    assert torch.equal(gp2.get_opacity, torch.clamp_max(torch.linspace(0.0, 1.0, 64)[:, None], 0.1))


def test_filtered_getters_equal_the_plain_ones_without_a_filter():
    gp = _store()
    gp.filter_3D = None
    assert torch.equal(gp.get_scaling_with_3D_filter, gp.get_scaling)
    assert torch.equal(gp.get_opacity_with_3D_filter, gp.get_opacity)


def test_depth_entry_rejects_bad_arguments_before_device_work():
    lib = _lib.load()
    one = C.c_void_p(1)     # never dereferenced: validation fails first

    def call(P=10, means=one, n=4, views=one, fx=100.0, fy=100.0, w=64, h=48, out=one):
        return lib.dgs_filter3d_depth(P, means, n, views, fx, fy, w, h, 0.2, out, None)

    for kw in (dict(P=-1), dict(n=-1), dict(fx=0.0), dict(fy=-1.0), dict(fx=float("nan")), dict(w=0), dict(h=-2),
               dict(means=None), dict(views=None), dict(out=None)):
        assert call(**kw) == -1, kw
        assert b"dgs_filter3d_depth" in lib.dgs_last_error()
    # nothing to sweep: no pointer is needed and nothing is launched
    assert call(P=0, means=None, views=None, out=None) == 0
    assert call(n=0, means=None, views=None, out=None) == 0


def test_filtered_activation_entries_reject_a_null_filter():
    lib = _lib.load()
    one = C.c_void_p(1)
    assert lib.dgs_activate_forward_filter3d(10, 1, one, None, one, one, one, 0.0, 0, one, one, one, one, None,
                                             None) == -1
    assert b"filter3d" in lib.dgs_last_error()
    assert lib.dgs_activate_backward_filter3d(10, 1, one, one, one, 0, None, None, None, None, one, None, one, one,
                                              one, 0.0, None, None) == -1
    assert b"filter3d" in lib.dgs_last_error()
    # the other checks stay in front of device work too
    assert lib.dgs_activate_forward_filter3d(-1, 1, one, None, one, one, one, 0.0, 0, one, one, one, one, one,
                                             None) == -1


def test_python_surface_defaults_to_no_filter():
    gp = GaussianParams(torch.zeros(2, 3), torch.zeros(2, 1, 3), torch.zeros(2, 0, 3), torch.zeros(2, 3),
                        torch.ones(2, 4), torch.ones(2, 1), 0)
    assert gp.filter_3D is None
    assert inspect.signature(activate_gaussians).parameters["filter3d"].default is None
    assert inspect.signature(rz.render_store_blurry).parameters["filter3d"].default is None
