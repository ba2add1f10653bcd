"""CPU: the SSIM oracle (oracle/ssim_torch.py, the reference's `ssim` restated in torch) against an independent scipy
computation, the closed-form three-map gradient the SSIM kernels implement (deblurgs_b200/csrc/dgs_ssim.cu) against
float64 autograd, and the argument checks of the SSIM C entry points and of loss.ssim."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from scipy import ndimage

from deblurgs_b200 import _lib
from deblurgs_b200.loss import ssim as fused_ssim
from deblurgs_b200.loss import training_loss
from oracle import ssim_torch as ot

SHAPES = [(1, 3, 32, 40), (2, 1, 5, 7), (2, 3, 9, 23), (1, 2, 17, 6), (3, 3, 12, 12)]


def _scipy_ssim_map(x, y):
    w = ot.create_window(11, 1)[0, 0].double().numpy()
    N, Cc = x.shape[:2]
    out = np.empty(x.shape)
    for n in range(N):
        for c in range(Cc):
            a, b = x[n, c], y[n, c]
            corr = lambda t: ndimage.correlate(t, w, mode="constant", cval=0.0)   # noqa: E731
            mu1, mu2 = corr(a), corr(b)
            s1, s2, s12 = corr(a * a) - mu1 ** 2, corr(b * b) - mu2 ** 2, corr(a * b) - mu1 * mu2
            C1, C2 = 0.01 ** 2, 0.03 ** 2
            out[n, c] = ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 ** 2 + mu2 ** 2 + C1) * (s1 + s2 + C2))
    return out


def _pair(shape, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(shape, generator=g, dtype=torch.float64)
    y = (x + 0.2 * torch.randn(shape, generator=g, dtype=torch.float64)).clamp(0, 1)
    return x, y


@pytest.mark.parametrize("shape", SHAPES)
def test_oracle_equals_scipy_correlate(shape):
    x, y = _pair(shape, 0)
    m = _scipy_ssim_map(x.numpy(), y.numpy())
    assert abs(ot.ssim(x, y).item() - m.mean()) < 1e-12
    per_image = ot.ssim(x, y, size_average=False).numpy()
    assert per_image.shape == (shape[0],)
    assert np.abs(per_image - m.reshape(shape[0], -1).mean(1)).max() < 1e-12
    assert abs(ot.ssim(x[0], y[0]).item() - m[0].mean()) < 1e-12          # [C,H,W] input


def test_window_is_the_reference_recipe():
    """exp in double stored as fp32, normalised by the double sum of the stored values rounded to fp32: what
    dgs_ssim.cu's host code computes, bit for bit the reference's window."""
    g = np.array([np.exp(-(i - 5) ** 2 / 4.5) for i in range(11)], dtype=np.float32)
    s = np.float32(g.astype(np.float64).sum())
    assert np.array_equal(g / s, ot.gaussian(11, 1.5).numpy())
    w = ot.create_window(11, 3)
    assert w.shape == (3, 1, 11, 11) and torch.equal(w, w.flip(-1)) and torch.equal(w, w.flip(-2))


def _closed_form_grad(x, y, gout, size_average):
    """dL/dx from the three per-pixel maps the forward kernel writes and the windowed sum the backward kernel takes."""
    Cc = x.shape[-3]
    w = ot.create_window(11, Cc).double()
    conv = lambda t: F.conv2d(t, w, padding=5, groups=Cc)   # noqa: E731  (the window is symmetric: its own adjoint)
    mu1, mu2 = conv(x), conv(y)
    s1, s2, s12 = conv(x * x) - mu1 ** 2, conv(y * y) - mu2 ** 2, conv(x * y) - mu1 * mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    A1, A2, B1, B2 = 2 * mu1 * mu2 + C1, 2 * s12 + C2, mu1 ** 2 + mu2 ** 2 + C1, s1 + s2 + C2
    s = A1 * A2 / (B1 * B2)
    d_s1 = -s / B2
    d_s12 = 2 * A1 / (B1 * B2)
    d_mu = 2 * mu2 * A2 / (B1 * B2) - 2 * mu1 * s / B1 - 2 * mu1 * d_s1 - mu2 * d_s12
    if size_average:
        g = gout / x.numel()
    else:
        g = (gout / x[0].numel()).reshape(-1, 1, 1, 1)
    return g * (conv(d_mu) + 2 * x * conv(d_s1) + y * conv(d_s12))


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("size_average", [True, False])
def test_closed_form_gradient_equals_autograd(shape, size_average):
    x, y = _pair(shape, 1)
    g = torch.Generator().manual_seed(7)
    gout = torch.tensor(-2.5, dtype=torch.float64) if size_average else \
        torch.randn(shape[0], generator=g, dtype=torch.float64)
    xr = x.clone().requires_grad_(True)
    (ot.ssim(xr, y, size_average=size_average) * gout).sum().backward()
    got = _closed_form_grad(x, y, gout, size_average)
    assert (got - xr.grad).abs().max().item() < 1e-10 * max(1.0, xr.grad.abs().max().item())


def test_closed_form_gradient_of_a_3d_input():
    x, y = _pair((3, 14, 19), 2)
    xr = x.clone().requires_grad_(True)
    (0.75 * ot.ssim(xr, y)).backward()
    got = _closed_form_grad(x[None], y[None], torch.tensor(0.75, dtype=torch.float64), True)[0]
    assert (got - xr.grad).abs().max().item() < 1e-10


def test_ssim_entry_points_validate_arguments_before_device_work():
    lib = _lib.load()
    one = C.c_void_p(1)   # never dereferenced: validation fails first
    assert lib.dgs_ssim_scratch_bytes(1, 3, 400, 600) == 19 * 25 * 3 * 8      # one double per 32x16 tile and plane
    assert lib.dgs_ssim_scratch_bytes(2, 3, 5, 7) == 2 * 3 * 8
    for dims in [(0, 3, 8, 8), (1, 0, 8, 8), (1, 3, 0, 8), (1, 3, 8, -1), (65536, 1, 8, 8), (300, 300, 8, 8)]:
        assert lib.dgs_ssim_scratch_bytes(*dims) == 0
        assert lib.dgs_ssim_forward(*dims, one, one, one, one, None, None) == -1
        assert b"dgs_ssim_forward" in lib.dgs_last_error()
        assert lib.dgs_ssim_backward(*dims, one, one, one, None, 0, one, None) == -1
    for i in range(4):                     # img1, img2, ssim_out, scratch are required; maps may be NULL
        args = [one] * 4
        args[i] = None
        assert lib.dgs_ssim_forward(1, 3, 8, 8, *args, None, None) == -1
    for i in range(4):                     # img1, img2, maps, dL_dimg1 are required; grad_out NULL means 1
        args = [one, one, one, one]
        args[i] = None
        assert lib.dgs_ssim_backward(1, 3, 8, 8, args[0], args[1], args[2], None, 1, args[3], None) == -1


def test_ssim_rejects_bad_input():
    a = torch.rand(2, 3, 8, 8)
    with pytest.raises(_lib.DgsError, match="same"):
        fused_ssim(a, a[:, :2])
    with pytest.raises(_lib.DgsError, match="same"):
        fused_ssim(a[0, 0], a[0, 0])                       # 2-D
    with pytest.raises(_lib.DgsError, match="empty"):
        fused_ssim(a[:0], a[:0])
    with pytest.raises(_lib.DgsError, match="window_size"):
        fused_ssim(a, a, window_size=7)
    with pytest.raises(_lib.DgsError, match="size_average=False"):
        fused_ssim(a[0], a[0], size_average=False)
    with pytest.raises(_lib.DgsError, match="constant target"):
        fused_ssim(a, a.clone().requires_grad_(True))
    with pytest.raises(_lib.DgsError, match="no CPU path"):
        fused_ssim(a, a)


def test_training_loss_rejects_a_dssim_weight_outside_0_1():
    b = torch.rand(3, 8, 8)
    for lam in (-0.1, 1.0, 1.5):
        with pytest.raises(_lib.DgsError, match="lambda_dssim"):
            training_loss(b, b[None], b, lambda_dssim=lam)
