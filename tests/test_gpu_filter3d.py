"""GPU: Mip-Splatting's 3-D smoothing filter -- the sampling-depth sweep (k_filter3d_depth) against a float64 oracle
and across call patterns, the filtered activations against the torch statement and float64 autograd, the store render
and the single-view render with the filter, Mip-Splatting's sampling guarantee, the densify rows, and the captured
training step."""
import math

import pytest
import torch

from deblurgs_b200 import rasterizer as rz
from deblurgs_b200 import renderer
from deblurgs_b200.filter3d import SamplingDepth
from deblurgs_b200.motion import GaussianParams, MiniCam
from deblurgs_b200.params import activate_gaussians

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
W, H, Z_NEAR = 64, 48, 0.2
FOVX, FOVY = 2 * math.atan(W / 100.0), 2 * math.atan(H / 100.0)    # focal 50 px on both axes
TOL = 1e-5                                                         # boundary band: either decision is right


def _rot(axis_angle):
    k = torch.zeros(3, 3, dtype=torch.float64)
    x, y, z = axis_angle.tolist()
    k[0, 1], k[0, 2], k[1, 0], k[1, 2], k[2, 0], k[2, 1] = -z, y, z, -x, -y, x
    return torch.matrix_exp(k)


def _cameras(n, seed):
    """n world-to-view transforms in the row-vector layout (p = [x, 1] V): small rotations and translations."""
    g = torch.Generator().manual_seed(seed)
    V = torch.zeros(n, 4, 4, dtype=torch.float64)
    for c in range(n):
        V[c, :3, :3] = _rot((torch.rand(3, generator=g, dtype=torch.float64) - 0.5) * 0.1)
        V[c, 3, :3] = (torch.rand(3, generator=g, dtype=torch.float64) - 0.5) * 0.4
        V[c, 3, 3] = 1.0
    return V


def _oracle(xyz, V, fx, fy):
    """float64 per (Gaussian, camera): z, u, v and the strict / loose visibility (decisions within TOL of a bound
    count as seen in the loose set only)."""
    p = torch.cat([xyz, torch.ones(xyz.shape[0], 1, dtype=torch.float64)], 1) @ V       # [C, P, 4]
    z = p[..., 2]
    zc = z.clamp_min(0.001)
    u, v = p[..., 0] / zc * fx + W / 2.0, p[..., 1] / zc * fy + H / 2.0

    def seen(t):
        return ((z > Z_NEAR + t * Z_NEAR) & (u >= -0.15 * W + t * W) & (u <= 1.15 * W - t * W) &
                (v >= -0.15 * H + t * H) & (v <= 1.15 * H - t * H))
    return z, u, v, seen(TOL), seen(-TOL)


def _min_depth(z, mask):
    return torch.where(mask, z, torch.full_like(z, math.inf)).min(0).values


def _scene(seed=0):
    """Points placed in camera 0's frame (z, u, v), mapped to the world."""
    g = torch.Generator().manual_seed(seed)
    r = lambda n, lo, hi: lo + (hi - lo) * torch.rand(n, generator=g, dtype=torch.float64)
    groups = {
        "regular": (r(300, 1.0, 6.0), r(300, 0, W), r(300, 0, H)),
        "behind": (r(30, -3.0, -0.3), r(30, 0, W), r(30, 0, H)),
        "near": (r(30, 0.01, 0.19), r(30, 0, W), r(30, 0, H)),                       # between 0.001 and z_near
        "u_in": (r(20, 1.5, 4.0), torch.full((20,), 1.15 * W * (1 - 2e-3)), r(20, 0, H)),
        "u_out": (r(20, 1.5, 4.0), torch.full((20,), 1.15 * W * (1 + 2e-3)), r(20, 0, H)),
        "u_in_lo": (r(20, 1.5, 4.0), torch.full((20,), -0.15 * W + 2e-3 * W), r(20, 0, H)),
        "v_out_lo": (r(20, 1.5, 4.0), r(20, 0, W), torch.full((20,), -0.15 * H - 2e-3 * H)),
        "v_in": (r(20, 1.5, 4.0), r(20, 0, W), torch.full((20,), 1.15 * H * (1 - 2e-3))),
        "unseen": (r(20, 1.0, 4.0), torch.full((20,), 12.0 * W), r(20, 0, H)),
    }
    return groups


def _to_world(groups, V0, fx, fy):
    pts = []
    for z, u, v in groups.values():
        cam = torch.stack([(u - W / 2.0) / fx * z, (v - H / 2.0) / fy * z, z], 1)
        pts.append((cam - V0[3, :3]) @ V0[:3, :3].T)      # p = x R + t  =>  x = (p - t) R^T
    return torch.cat(pts)


def test_sweep_equals_the_float64_oracle():
    V = _cameras(6, seed=1)
    V[0, :3, :3] = torch.eye(3, dtype=torch.float64)
    fx = float(torch.tensor(W / (2 * math.tan(FOVX / 2)), dtype=torch.float32))
    fy = float(torch.tensor(H / (2 * math.tan(FOVY / 2)), dtype=torch.float32))
    xyz = _to_world(_scene(), V[0], fx, fy)
    z, u, v, strict, loose = _oracle(xyz, V, fx, fy)
    d_strict, d_loose = _min_depth(z, strict), _min_depth(z, loose)
    # the scene contains every case it targets, as unambiguous decisions
    screen = (u >= -0.15 * W) & (u <= 1.15 * W) & (v >= -0.15 * H) & (v <= 1.15 * H)
    assert (z < 0).any()
    assert ((z > 0.001) & (z < Z_NEAR * (1 - TOL)) & screen).any()
    assert (strict & (1.15 * W - u > TOL * W) & (1.15 * W - u < 0.01 * W)).any()              # just inside
    assert ((z > Z_NEAR * (1 + TOL)) & (u - 1.15 * W > TOL * W) & (u - 1.15 * W < 0.01 * W) &
            (v >= 0) & (v <= H)).any()                                                          # just outside
    assert (strict & (u + 0.15 * W > TOL * W) & (u + 0.15 * W < 0.01 * W)).any()
    assert ((z > Z_NEAR) & (-0.15 * H - v > TOL * H) & (-0.15 * H - v < 0.01 * H)).any()
    assert (strict & (1.15 * H - v > TOL * H) & (1.15 * H - v < 0.01 * H)).any()
    assert torch.isinf(d_loose).sum() >= 20
    sd = SamplingDepth(xyz.shape[0], DEV).add(xyz.float().to(DEV), V.float().to(DEV), W, H, FOVX, FOVY, Z_NEAR)
    got = sd.min_depth.double().cpu()
    inf_ok = torch.isinf(got) <= torch.isinf(d_strict)                  # unseen only where no camera surely sees it
    assert inf_ok.all()
    fin = torch.isfinite(got)
    assert (got[fin] >= d_loose[fin] * (1 - 1e-5)).all()
    assert (got[fin] <= d_strict[fin] * (1 + 1e-5)).all()
    assert torch.isinf(got[torch.isinf(d_loose)]).all()
    assert (d_loose == d_strict).float().mean() > 0.95
    assert sd.max_focal == pytest.approx(50.0)


def test_sweep_is_bit_identical_for_any_order_and_split_of_the_cameras():
    views, F = 20, 16
    V = _cameras(views * F, seed=2).float().to(DEV)        # 320 cameras: more than two shared-memory chunks (128)
    g = torch.Generator().manual_seed(3)
    xyz = (torch.rand(5000, 3, generator=g) * torch.tensor([8.0, 6.0, 6.0]) - torch.tensor([4.0, 3.0, 0.5])).to(DEV)

    def run(batches):
        sd = SamplingDepth(xyz.shape[0], DEV)
        for b in batches:
            sd.add(xyz, b, W, H, FOVX, FOVY, Z_NEAR)
        return sd.min_depth

    ref = run([V])
    assert torch.isfinite(ref).any() and torch.isinf(ref).any()
    for batches in ([V[i * F:(i + 1) * F] for i in range(views)],
                    [V.flip(0)],
                    [V[:100], V[100:250], V[250:]],
                    [V[:129], V[129:257], V[257:]],
                    [V[i:i + 1] for i in range(V.shape[0])][::-1]):
        assert torch.equal(run(batches), ref)


def test_max_focal_over_calls_of_different_intrinsics():
    xyz = torch.tensor([[0.0, 0.0, 2.0], [0.1, 0.0, 3.0]], device=DEV)
    V = torch.eye(4, device=DEV)[None]
    sd = SamplingDepth(2, DEV)
    sd.add(xyz, V, W, H, FOVX, FOVY, Z_NEAR)
    sd.add(xyz, V, 2 * W, 2 * H, FOVX, FOVY, Z_NEAR)         # same FoV at twice the size: twice the focal length
    sd.add(xyz, V, W, H, FOVX, FOVY, Z_NEAR)
    assert sd.max_focal == pytest.approx(100.0)
    f = sd.filter_3D()
    want = torch.tensor([2.0, 3.0], device=DEV) / sd.max_focal * math.sqrt(0.2)
    assert torch.allclose(f[:, 0], want, rtol=1e-6)


def _raw_store(P=3000, iso=False, lb=0.0, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.rand(*s, generator=g)
    raw = dict(xyz=r(P, 3), dc=r(P, 1, 3), rest=r(P, 15, 3) - 0.5, scaling=torch.randn(P, 3, generator=g) - 4.0,
               rotation=r(P, 4) + 0.1, opacity=r(P, 1) * 1.4 - 0.2)
    raw["scaling"][:5] = math.log(1e-7)                       # tiny scales: the per-axis form does not underflow
    gp = GaussianParams(*(raw[k].to(DEV) for k in ("xyz", "dc", "rest", "scaling", "rotation", "opacity")), 3,
                        scale_lower_bound=lb, use_isotropic=iso)
    f = (torch.rand(P, 1, generator=g) * 0.05)
    f[:5] = 1e-3
    f[5:10] = 5.0                                             # f >> s
    f[10:15] = 1e-9                                           # f << s
    gp.filter_3D = f.to(DEV)
    return gp


@pytest.mark.parametrize("iso,lb", [(False, 0.0), (True, 0.0), (False, 0.003)])
def test_filtered_activations_match_the_torch_statement_and_float64_gradients(iso, lb):
    gp = _raw_store(iso=iso, lb=lb)
    leaves = [gp._features_dc, gp._features_rest, gp._scaling, gp._rotation, gp._opacity]
    shs, scales, rots, opac = activate_gaussians(*leaves, lb, iso, gp.filter_3D)
    with torch.no_grad():
        want_s, want_o = gp.get_scaling_with_3D_filter, gp.get_opacity_with_3D_filter
    assert ((scales - want_s).abs() <= 4e-7 * want_s.abs()).all(), ((scales - want_s).abs() / want_s.abs()).max()
    assert ((opac - want_o).abs() <= 4e-7 * want_o.abs()).all(), ((opac - want_o).abs() / want_o.abs().clamp_min(
        1e-30)).max()
    assert (opac[:5] > 0).all()
    g = torch.Generator().manual_seed(1)
    gs = torch.randn(scales.shape, generator=g).to(DEV)
    go = torch.randn(opac.shape, generator=g).to(DEV)
    torch.autograd.backward((scales, opac), (gs, go))
    # float64 autograd of the torch statement
    rs = gp._scaling.detach().double().requires_grad_(True)
    ro = gp._opacity.detach().double().requires_grad_(True)
    e = torch.exp(rs[:, :1].expand(-1, 3)) if iso else torch.exp(rs)
    s = e + lb
    f = gp.filter_3D.double()
    sp = torch.sqrt(s * s + f * f)
    r = s / sp
    op = ro.clamp(0.0, 1.0) * r[:, 0:1] * r[:, 1:2] * r[:, 2:3]
    torch.autograd.backward((sp, op), (gs.double(), go.double()))
    for mine, ref in ((gp._scaling.grad, rs.grad), (gp._opacity.grad, ro.grad)):
        err = (mine.double() - ref).abs()
        assert (err <= 1e-5 * ref.abs() + 1e-6 * ref.abs().max()).all(), (err / ref.abs().clamp_min(1e-30)).max()


def test_unfiltered_activations_are_bit_identical_to_the_plain_entry():
    gp = _raw_store()
    leaves = [gp._features_dc, gp._features_rest, gp._scaling, gp._rotation, gp._opacity]
    plain = activate_gaussians(*leaves, 0.0, False)
    zero = activate_gaussians(*leaves, 0.0, False, torch.zeros_like(gp.filter_3D))   # f = 0: s' = s, r = 1 exactly
    for a, b in zip(plain, zero):
        assert torch.equal(a, b)
    gp.filter_3D = None
    for a, b in zip(plain, gp.get_activated()):
        assert torch.equal(a, b)


def _workload(name="small"):
    import bench
    return bench.build_workload(name, 0, DEV)


def _settings(w, campos):
    cam = w["cam"]
    return rz.GaussianRasterizationSettings(cam.height, cam.width, cam.tanfovx, cam.tanfovy, w["bg"], 1.0, 0.2, 100.0,
                                            False, w["gaussians"].active_sh_degree, campos, False, False)


def test_store_render_with_the_filter_equals_the_activated_render():
    w = _workload()
    store, cmm = w["gaussians"], w["cmm"]
    assert store._xyz.shape[0] >= 4096 * 4                   # four backward ranges: the filter rows are offset per range
    f = cmm.compute_3D_filter() * 20.0                        # enlarged so that it changes the image markedly
    view, proj, campos = (t.detach() for t in cmm.get_trajectory_tensors(0))
    rs = _settings(w, campos)
    raw = [store._xyz, store._features_dc, store._features_rest, store._scaling, store._rotation, store._opacity]
    F, Hh, Ww = view.shape[0], w["H"], w["W"]
    dL = torch.randn(F, 3, Hh, Ww, generator=torch.Generator().manual_seed(2)).to(DEV) / (Hh * Ww)

    def leaves():
        return [t.detach().clone().requires_grad_(True) for t in raw]

    def store_path():
        ls = leaves()
        color, _, _, _ = rz.render_store_blurry(*ls, None, view, proj, campos, rs, n_ranges=4, filter3d=f)
        (color * dL).sum().backward()
        return color.detach(), [t.grad for t in ls]

    def activated_path(filt=f):
        ls = leaves()
        shs, scales, rots, opac = activate_gaussians(*ls[1:], 0.0, False, filt)
        color, _, _, _ = rz.rasterize_blurry(ls[0], None, shs, None, opac, scales, rots, None, view, proj, campos, rs)
        (color * dL).sum().backward()
        return color.detach(), [t.grad for t in ls]

    c_store, g_store = store_path()
    c_a, g_a = activated_path()
    c_b, g_b = activated_path()
    c_plain, _ = activated_path(None)
    assert torch.equal(c_store, c_a)
    assert (c_store - c_plain).abs().max().item() > 1e-2
    for s_, a, b in zip(g_store, g_a, g_b):
        spread = (a - b).abs().max().item()
        floor = 1e-6 * a.abs().max().item()
        assert (s_ - a).abs().max().item() <= 4 * max(spread, floor), (spread, (s_ - a).abs().max().item())


def test_single_view_render_through_the_torch_getters_equals_the_batched_render():
    w = _workload()
    store, cmm = w["gaussians"], w["cmm"]
    store.filter_3D = cmm.compute_3D_filter() * 20.0
    view, proj, campos = (t.detach() for t in cmm.get_trajectory_tensors(0))
    ref = cmm.original_cam[0]
    with torch.no_grad():
        batched = renderer.render_blurry(view, proj, campos, ref, store, w["bg"])["render"]
        for s in range(view.shape[0]):
            mc = MiniCam(ref.image_width, ref.image_height, ref.FoVy, ref.FoVx, ref.znear, ref.zfar, view[s], proj[s],
                         campos[s])
            img = renderer.render(mc, store, w["bg"])["render"]
            err = (img - batched[s]).abs()
            assert torch.quantile(err.flatten()[::3], 0.999).item() < 1e-4 and err.max().item() < 2e-2, err.max()


def test_filter_bounds_every_gaussian_at_the_sampling_limit():
    w = _workload()
    store, cmm = w["gaussians"], w["cmm"]
    with torch.no_grad():                                    # 64 Gaussians 100 units behind the first sub-frame camera
        view0, _, campos0 = cmm.get_trajectory_tensors(0)
        store._xyz[:64] = campos0[0] - 100.0 * view0[0, :3, 2]
    f = cmm.compute_3D_filter()
    assert f is store.filter_3D and f.shape == (store._xyz.shape[0], 1)
    ref = cmm.original_cam[0]
    sd = SamplingDepth(store._xyz.shape[0], DEV)
    view, _, _ = cmm.get_trajectory_tensors(0)
    sd.add(store._xyz, view, ref.image_width, ref.image_height, ref.FoVx, ref.FoVy, store.z_near)
    seen = torch.isfinite(sd.min_depth)
    assert seen.any() and (~seen).any()
    d = torch.where(seen, sd.min_depth, sd.min_depth[seen].max())[:, None]
    with torch.no_grad():
        for sp in (store.get_scaling_with_3D_filter, store.get_activated()[1]):
            bound = sp.min(dim=1, keepdim=True).values * sd.max_focal / d
            assert (bound >= math.sqrt(0.2) * (1 - 1e-6)).all(), bound.min()


def test_gpu_densify_rows_carry_the_filter_as_the_cpu_plan():
    g = torch.Generator().manual_seed(0)
    P = 200
    r = lambda *s: torch.rand(*s, generator=g)
    base = [r(P, 3), r(P, 1, 3), r(P, 3, 3), r(P, 3) - 3.0, r(P, 4) + 0.1, r(P, 1)]
    filt = torch.rand(P, 1, generator=g) * 0.01
    grads = (torch.rand(P, 1, generator=g) > 0.7).float()
    prune = torch.rand(P, generator=g) > 0.8
    out = {}
    for dev in ("cpu", "cuda"):
        gp = GaussianParams(*(t.clone().to(dev) for t in base), 1)
        gp.training_setup()
        gp.filter_3D = filt.clone().to(dev)
        gp.densify_and_clone(grads.to(dev), 0.5, 3.0)
        gp.densify_and_split(torch.cat([grads, torch.zeros(gp._xyz.shape[0] - P, 1)]).to(dev), 0.5, 3.0)
        gp.prune_points(torch.cat([prune, torch.zeros(gp._xyz.shape[0] - P, dtype=torch.bool)]).to(dev))
        assert gp.filter_3D.shape == (gp._xyz.shape[0], 1)
        out[dev] = gp.filter_3D.cpu()
    assert out["cpu"].shape[0] != P
    assert torch.equal(out["cpu"], out["cuda"])


def test_graph_replay_with_the_filter_equals_eager_and_follows_an_in_place_recompute():
    from deblurgs_b200.graph import BlurryViewGraph
    from deblurgs_b200.loss import blur_photometric_loss
    w = _workload()
    store, cmm = w["gaussians"], w["cmm"]
    params = store.parameters() + cmm.parameters()
    gt = w["gt_host"].to(DEV)
    f = cmm.compute_3D_filter()
    with torch.no_grad():
        f.mul_(20.0)                                        # in place: a visible effect on this scene

    def eager():
        for p in params:
            p.grad = None
        out = cmm.query(0, "all", background=w["bg"])
        loss = blur_photometric_loss(out["blurred"], out["subframes"], gt, 0.0)
        loss.backward()
        torch.cuda.synchronize()
        return loss.item(), [p.grad.clone() for p in params]

    def check(g):
        l_ref, g_ref = eager()
        val = g.step(gt)
        assert abs(val - l_ref) <= 1e-6
        for p, r in zip(params, g_ref):
            assert ((p.grad - r).abs().max() / r.abs().max().clamp_min(1e-30)).item() <= 1e-3
        return val

    g = BlurryViewGraph(cmm, 0, w["bg"], (3, w["H"], w["W"]), 0.0)
    v1 = check(g)
    ptr = store.filter_3D.data_ptr()
    old = store.filter_3D.clone()
    with torch.no_grad():
        cmm._trans._control_points.add_(0.05)               # another trajectory: other sampling depths
    cmm.compute_3D_filter()
    assert store.filter_3D.data_ptr() == ptr and not torch.equal(store.filter_3D, old)
    v2 = check(g)
    assert v1 != v2
    saved = store.filter_3D
    store.filter_3D = None
    with pytest.raises(Exception, match="3-D filter"):
        g.replay()
    store.filter_3D = saved.clone()
    with pytest.raises(Exception, match="3-D filter"):
        g.replay()
