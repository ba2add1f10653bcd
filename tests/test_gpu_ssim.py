"""GPU: the fused SSIM (deblurgs_b200.loss.ssim, dgs_ssim.cu) against the float64 restatement of the reference's
`ssim` (oracle/ssim_torch.py) in value and gradient, its determinism across calls and graph replays, the D-SSIM term of
training_loss and of the graph-captured step, and refine.evaluate_views."""
import pytest
import torch

from deblurgs_b200.loss import psnr, ssim, training_loss
from oracle import ssim_torch as ot

pytestmark = pytest.mark.gpu

# (N, C, H, W): tiny, ragged tiles, square, c2, c3; C = 1 and 3; N = 1 and 4
SHAPES = [(1, 1, 5, 7), (4, 3, 5, 7), (1, 3, 37, 53), (4, 1, 37, 53), (1, 3, 256, 256), (4, 1, 256, 256),
          (4, 3, 400, 600), (1, 3, 1080, 1920)]


def _pair(shape, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(shape, generator=g, device="cuda")
    y = (x + 0.15 * torch.randn(shape, generator=g, device="cuda")).clamp(0, 1)
    return x, y


def _torch_fp32(x, y, size_average):
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        return ot.ssim(x, y, size_average=size_average).double()
    finally:
        torch.backends.cudnn.allow_tf32 = prev


def _check_forward(x, y):
    ref_mean = ot.ssim(x.double(), y.double()).item()
    ref_img = ot.ssim(x.double(), y.double(), size_average=False)
    tol_mean = max(2e-6, 2 * abs(_torch_fp32(x, y, True).item() - ref_mean))
    tol_img = (2 * (_torch_fp32(x, y, False) - ref_img).abs()).clamp_min(2e-6)
    got_mean = ssim(x, y).item()
    got_img = ssim(x, y, size_average=False).double()
    assert abs(got_mean - ref_mean) <= tol_mean, (got_mean, ref_mean, tol_mean)
    assert ((got_img - ref_img).abs() <= tol_img).all(), (got_img, ref_img, tol_img)
    assert abs(ssim(x[0], y[0]).item() - ref_img[0].item()) <= tol_img[0].item()      # [C,H,W] input


def _check_gradient(x, y, size_average, seed=3):
    gout = torch.tensor(-1.7, device="cuda") if size_average else \
        torch.randn(x.shape[0], generator=torch.Generator(device="cuda").manual_seed(seed), device="cuda")
    xr = x.clone().requires_grad_(True)
    (ssim(xr, y, size_average=size_average) * gout).sum().backward()
    xd = x.double().requires_grad_(True)
    (ot.ssim(xd, y.double(), size_average=size_average) * gout.double()).sum().backward()
    ref = xd.grad
    err = (xr.grad.double() - ref).abs().max().item()
    assert err <= 1e-3 * ref.abs().max().item(), (err, ref.abs().max().item())


@pytest.mark.parametrize("shape", SHAPES)
def test_forward_matches_the_float64_reference(shape):
    x, y = _pair(shape)
    _check_forward(x, y)
    assert abs(ssim(x, x).item() - 1.0) <= 1e-6


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("size_average", [True, False])
def test_gradient_matches_float64_autograd(shape, size_average):
    x, y = _pair(shape, 1)
    _check_gradient(x, y, size_average)


def test_scene_render_against_its_motion_blurred_copy():
    import bench
    w = bench.build_workload("small", 0, torch.device("cuda", 0))
    with torch.no_grad():
        out = w["cmm"].query(0, "all", background=w["bg"])
    sharp = out["subframes"][0].clamp(0, 1).contiguous()
    blurry = out["blurred"].clamp(0, 1).contiguous()
    pair = (torch.stack([sharp, blurry]), torch.stack([blurry, out["subframes"][-1].clamp(0, 1)]))
    _check_forward(*pair)
    _check_gradient(*pair, size_average=False)


def test_repeated_calls_and_graph_replays_are_bit_identical():
    x, y = _pair((4, 3, 400, 600), 5)
    xr = x.clone().requires_grad_(True)
    a = ssim(xr, y, size_average=False)
    b = ssim(xr, y, size_average=False)
    assert torch.equal(a, b)
    (a.sum()).backward()
    g1 = xr.grad.clone()
    xr.grad = None
    b.sum().backward()
    assert torch.equal(g1, xr.grad)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ssim(x, y)                                       # warm-up before capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = ssim(x, y)
    graph.replay()
    first = loss.clone()
    graph.replay()
    assert torch.equal(first, loss)
    assert torch.equal(first, ssim(x, y))


@pytest.mark.parametrize("lam_t", [0.0, 1e-3])
def test_training_loss_with_dssim_matches_the_reference_mix(lam_t):
    F, H, W, lam = 4, 70, 90, 0.2
    g = torch.Generator(device="cuda").manual_seed(11)
    blurred = torch.rand(3, H, W, generator=g, device="cuda")
    sub = torch.rand(F, 3, H, W, generator=g, device="cuda")
    gt = torch.rand(3, H, W, generator=g, device="cuda")
    b, s = blurred.clone().requires_grad_(True), sub.clone().requires_grad_(True)
    loss = training_loss(b, s, gt, lambda_t_smooth=lam_t, lambda_dssim=lam)
    loss.backward()
    bd, sd = blurred.double().requires_grad_(True), sub.double().requires_grad_(True)
    ref = (1 - lam) * (bd - gt.double()).abs().mean() + lam * (1 - ot.ssim(bd, gt.double())) + \
        lam_t * (sd[1:] - sd[:-1]).abs().mean()
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 2e-6
    for got, want in ((b.grad, bd.grad), (s.grad, sd.grad)):
        if lam_t == 0.0 and want is sd.grad:
            assert got is None
            continue
        assert (got.double() - want).abs().max().item() <= 1e-3 * want.abs().max().item()
    # lambda_dssim = 0 is today's loss, bit for bit
    assert torch.equal(training_loss(blurred, sub, gt, lambda_t_smooth=lam_t),
                       training_loss(blurred, sub, gt, lambda_t_smooth=lam_t, lambda_dssim=0.0))


def test_graph_replay_with_dssim_equals_eager_step():
    import bench
    from deblurgs_b200.graph import BlurryViewGraph
    dev = torch.device("cuda", 0)
    w = bench.build_workload("small", 0, dev)
    params = w["gaussians"].parameters() + w["cmm"].parameters()
    gt = w["gt_host"].to(dev)
    step = BlurryViewGraph(w["cmm"], 0, w["bg"], (3, w["H"], w["W"]), 1e-3, lambda_dssim=0.2)
    for p in params:
        p.grad = None
    out = w["cmm"].query(0, "all", background=w["bg"])
    loss = training_loss(out["blurred"], out["subframes"], gt, lambda_t_smooth=1e-3, lambda_dssim=0.2)
    loss.backward()
    torch.cuda.synchronize()
    l_ref, g_ref = loss.item(), [p.grad.clone() for p in params]
    val = step.step(gt)
    assert abs(val - l_ref) <= 2e-7, (val, l_ref)
    for p, r in zip(params, g_ref):
        # the rasterizer's backward accumulates with float atomics: same tolerance as tests/test_gpu_graph.py
        assert ((p.grad - r).abs().max() / r.abs().max().clamp_min(1e-30)).item() <= 1e-3
    assert step.recaptures == 0


class _Cam:
    pass


def test_evaluate_views_scores_renders_against_original_images():
    from tests import parity_utils as pu
    from deblurgs_b200 import renderer
    from deblurgs_b200.motion import GaussianParams
    from deblurgs_b200.refine import OptimPoseModel, evaluate_views
    cam, scene, traj, bg, view, proj, campos = pu.make_inputs("small")
    gauss = GaussianParams.from_scene(scene)
    cams = []
    for i in (0, 2, 3):
        c = _Cam()
        c.R, c.T = view[i, :3, :3].double().cpu().numpy(), view[i, 3, :3].double().cpu().numpy()
        c.image_width, c.image_height, c.FoVx, c.FoVy, c.znear, c.zfar = cam.width, cam.height, cam.fovx, cam.fovy, 0.01, 100.0
        cams.append(c)
    posed = OptimPoseModel(cams)
    g = torch.Generator(device="cuda").manual_seed(4)
    views, renders = [], []
    with torch.no_grad():
        for i in range(len(cams)):
            v = posed(i)
            r = renderer.render(v, gauss, bg)["render"].clamp(0, 1)
            v.original_image = (r + 0.05 * (i + 1) * torch.randn(r.shape, generator=g, device="cuda")).clamp(0, 1)
            views.append(v)
            renders.append(r)
    res = evaluate_views(views, gauss, bg)
    pred = torch.stack(renders)
    gt = torch.stack([v.original_image for v in views])
    want_psnr = (20 * torch.log10(1.0 / torch.sqrt(((pred - gt) ** 2).reshape(3, -1).mean(1)))).tolist()
    want_ssim = ot.ssim(pred.double(), gt.double(), size_average=False).tolist()
    assert len(res["psnr"]) == len(res["ssim"]) == 3
    for a, b in zip(res["psnr"], want_psnr):
        assert abs(a - b) <= 1e-4 * abs(b)
    for a, b in zip(res["ssim"], want_ssim):
        assert abs(a - b) <= 2e-6
    assert res["psnr"][0] > res["psnr"][1] > res["psnr"][2]          # noisier view, lower score
    assert abs(res["ssim_mean"] - sum(want_ssim) / 3) <= 2e-6
    assert torch.allclose(psnr(pred, gt)[:, 0], torch.tensor(want_psnr, device="cuda"))
