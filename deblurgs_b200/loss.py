"""Loss block of the blurry-view training step (reference: train.py:147-163, utils/loss_utils.py):
`blur_photometric_loss` = l1_loss(blurred, gt) + lambda_t_smooth * batchwise_smoothness_loss(subframes), forward and
backward in one kernel each; `tv_loss` (depth smoothness) and `hinge_l2` (opacity range penalty), one kernel each way;
`training_loss` = the reference's weighted sum of the four; `ssim` (one tile kernel each way, dgs_ssim.cu) for the
3DGS D-SSIM term and for evaluation, `psnr` (utils/image_utils.py)."""
import ctypes as C

import torch

from . import _lib


class _BlurLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, blurred, subframes, gt, lambda_t_smooth):
        lib = _lib.load()
        if not blurred.is_cuda:
            raise _lib.DgsError("blurred must be a CUDA tensor: libdgs_b200 has no CPU path")
        ctx.set_materialize_grads(False)
        lam = float(lambda_t_smooth)
        b = blurred.detach().float().contiguous()
        g = gt.detach().float().contiguous()
        F = subframes.shape[0]
        chw = b.numel()
        if subframes.numel() != F * chw or g.numel() != chw:
            raise _lib.DgsError("shape mismatch: subframes [F,3,H,W], blurred / gt [3,H,W]")
        # lambda_t_smooth == 0 (plain L1, e.g. pose refinement): the sub-frame stack is neither read nor given a gradient
        s = subframes.detach().float().contiguous() if lam != 0.0 else None
        out = torch.empty(3, dtype=torch.float32, device=b.device)
        scratch = torch.empty(2, dtype=torch.float64, device=b.device)
        with torch.cuda.device(b.device):
            rc = lib.dgs_blur_loss_forward(F, chw, _lib.ptr(s), _lib.ptr(b), _lib.ptr(g), float(lambda_t_smooth),
                                           _lib.ptr(out), _lib.ptr(scratch),
                                           C.c_void_p(torch.cuda.current_stream(b.device).cuda_stream))
        _lib.check(rc, "dgs_blur_loss_forward")
        ctx.save_for_backward(b, g) if s is None else ctx.save_for_backward(b, g, s)
        ctx.lam = lam
        ctx.F = F
        ctx.shapes = (blurred.shape, subframes.shape)
        ctx.parts = out
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        lib = _lib.load()
        if grad_out is None:
            return None, None, None, None
        saved = ctx.saved_tensors
        b, g = saved[0], saved[1]
        s = saved[2] if len(saved) > 2 else None
        F, chw = ctx.F, b.numel()
        go = grad_out.detach().float().contiguous().reshape(1)
        db = torch.empty_like(b)
        ds = torch.empty_like(s) if s is not None else None
        with torch.cuda.device(b.device):
            rc = lib.dgs_blur_loss_backward(F, chw, _lib.ptr(s), _lib.ptr(b), _lib.ptr(g), ctx.lam, _lib.ptr(go),
                                            _lib.ptr(db), _lib.ptr(ds),
                                            C.c_void_p(torch.cuda.current_stream(b.device).cuda_stream))
        _lib.check(rc, "dgs_blur_loss_backward")
        return db.view(ctx.shapes[0]), (ds.view(ctx.shapes[1]) if ds is not None else None), None, None


def blur_photometric_loss(blurred, subframes, gt, lambda_t_smooth=0.0):
    """l1_loss(blurred, gt) + lambda_t_smooth * batchwise_smoothness_loss(subframes) as a 0-dim tensor."""
    return _BlurLoss.apply(blurred, subframes, gt, lambda_t_smooth)


def _st(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


class _TV(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        lib = _lib.load()
        if not x.is_cuda:
            raise _lib.DgsError("tv_loss: CUDA tensor required (libdgs_b200 has no CPU path)")
        if x.dim() != 4:
            raise _lib.DgsError("tv_loss: x must be [B,C,H,W]")
        xc = x.detach().float().contiguous()
        B, Cc, H, W = xc.shape
        out = torch.empty(1, dtype=torch.float32, device=xc.device)
        scratch = torch.empty(2, dtype=torch.float64, device=xc.device)
        with torch.cuda.device(xc.device):
            _lib.check(lib.dgs_tv_loss_forward(B * Cc, H, W, _lib.ptr(xc), _lib.ptr(out), _lib.ptr(scratch), _st(xc)),
                       "dgs_tv_loss_forward")
        ctx.save_for_backward(xc)
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        lib = _lib.load()
        (xc,) = ctx.saved_tensors
        B, Cc, H, W = xc.shape
        go = grad_out.detach().float().contiguous().reshape(1)
        dx = torch.empty_like(xc)
        with torch.cuda.device(xc.device):
            _lib.check(lib.dgs_tv_loss_backward(B * Cc, H, W, _lib.ptr(xc), _lib.ptr(go), _lib.ptr(dx), _st(xc)),
                       "dgs_tv_loss_backward")
        return dx


class _Hinge(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        lib = _lib.load()
        if not x.is_cuda:
            raise _lib.DgsError("hinge_l2: CUDA tensor required (libdgs_b200 has no CPU path)")
        xc = x.detach().float().contiguous()
        out = torch.empty(1, dtype=torch.float32, device=xc.device)
        scratch = torch.empty(2, dtype=torch.float64, device=xc.device)
        with torch.cuda.device(xc.device):
            _lib.check(lib.dgs_hinge_l2_forward(xc.numel(), _lib.ptr(xc), _lib.ptr(out), _lib.ptr(scratch), _st(xc)),
                       "dgs_hinge_l2_forward")
        ctx.save_for_backward(xc)
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        lib = _lib.load()
        (xc,) = ctx.saved_tensors
        go = grad_out.detach().float().contiguous().reshape(1)
        dx = torch.empty_like(xc)
        with torch.cuda.device(xc.device):
            _lib.check(lib.dgs_hinge_l2_backward(xc.numel(), _lib.ptr(xc), _lib.ptr(go), _lib.ptr(dx), _st(xc)),
                       "dgs_hinge_l2_backward")
        return dx


class _SSIM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img1, img2, size_average):
        lib = _lib.load()
        x = img1.detach().float().contiguous()
        y = img2.detach().float().contiguous()
        N, Cc, H, W = (1,) + tuple(x.shape) if x.dim() == 3 else tuple(x.shape)
        out = torch.empty(1 + N, dtype=torch.float32, device=x.device)
        nbytes = int(lib.dgs_ssim_scratch_bytes(N, Cc, H, W))
        scratch = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=x.device)
        # dS/dmu1, dS/dsigma1^2, dS/dsigma12 per pixel: only when img1 wants a gradient
        maps = torch.empty((3,) + tuple(x.shape), dtype=torch.float32, device=x.device) if ctx.needs_input_grad[0] else None
        with torch.cuda.device(x.device):
            _lib.check(lib.dgs_ssim_forward(N, Cc, H, W, _lib.ptr(x), _lib.ptr(y), _lib.ptr(out), _lib.ptr(scratch),
                                            _lib.ptr(maps), _st(x)), "dgs_ssim_forward")
        if maps is not None:
            ctx.save_for_backward(x, y, maps)
        ctx.dims, ctx.size_average, ctx.shape = (N, Cc, H, W), size_average, img1.shape
        return out[0] if size_average else out[1:]

    @staticmethod
    def backward(ctx, grad_out):
        lib = _lib.load()
        x, y, maps = ctx.saved_tensors
        N, Cc, H, W = ctx.dims
        go = grad_out.detach().float().contiguous().reshape(-1)
        dx = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(lib.dgs_ssim_backward(N, Cc, H, W, _lib.ptr(x), _lib.ptr(y), _lib.ptr(maps), _lib.ptr(go),
                                             0 if ctx.size_average else 1, _lib.ptr(dx), _st(x)), "dgs_ssim_backward")
        return dx.view(ctx.shape), None, None


def ssim(img1, img2, window_size=11, size_average=True):
    """utils/loss_utils.py `ssim` (3DGS): SSIM of [C,H,W] or [N,C,H,W] images with an 11x11 Gaussian window
    (sigma 1.5, zero padding).  size_average=True: the mean over every pixel and channel (0-dim tensor); False: one
    mean per image ([N], 4-D input only).  Differentiable in img1; img2 is a constant target."""
    if img1.shape != img2.shape or img1.dim() not in (3, 4):
        raise _lib.DgsError("ssim: img1 and img2 must have the same [C,H,W] or [N,C,H,W] shape, got %s and %s"
                            % (tuple(img1.shape), tuple(img2.shape)))
    if img1.numel() == 0:
        raise _lib.DgsError("ssim: empty input %s" % (tuple(img1.shape),))
    if window_size != 11:
        raise _lib.DgsError("ssim: only window_size=11 is implemented")
    if not size_average and img1.dim() != 4:
        raise _lib.DgsError("ssim: size_average=False needs [N,C,H,W] input (one mean per image)")
    if img2.requires_grad:
        raise _lib.DgsError("ssim: img2 is treated as a constant target and gets no gradient; pass img2.detach()")
    if not (img1.is_cuda and img2.is_cuda):
        raise _lib.DgsError("ssim: CUDA tensors required (libdgs_b200 has no CPU path)")
    if img1.device != img2.device:
        raise _lib.DgsError("ssim: img1 and img2 are on different devices")
    return _SSIM.apply(img1, img2, bool(size_average))


def psnr(img1, img2):
    """utils/image_utils.py `psnr`: 20 log10(1 / sqrt(mse)) per leading index, shape [N, 1]."""
    mse = ((img1 - img2) ** 2).reshape(img1.shape[0], -1).mean(1, keepdim=True)
    return 20 * torch.log10(1.0 / torch.sqrt(mse))


def tv_loss(x):
    """utils/loss_utils.py:66-78 on a [B,C,H,W] tensor: l2 of the vertical + l2 of the horizontal neighbour differences."""
    return _TV.apply(x)


def hinge_l2(x):
    """utils/loss_utils.py:95-104: mean of x^2 where x <= 0 and (x - 1)^2 where x >= 1."""
    return _Hinge.apply(x)


def photometric_loss(blurred, subframes, gt, lambda_t_smooth=0.0, lambda_dssim=0.0):
    """Ll1 + lambda_t_smooth * L_t_smooth; with lambda_dssim > 0 the L1 term becomes the 3DGS D-SSIM mix
    (1 - lambda_dssim) * Ll1 + lambda_dssim * (1 - ssim(blurred, gt)).  lambda_dssim == 0 runs no SSIM kernel."""
    lam = float(lambda_dssim)
    if lam == 0.0:
        return blur_photometric_loss(blurred, subframes, gt, lambda_t_smooth)
    if not 0.0 < lam < 1.0:
        raise _lib.DgsError("lambda_dssim must lie in [0, 1), got %r" % (lambda_dssim,))
    # (1 - lam) * (Ll1 + lambda_t / (1 - lam) * L_t_smooth): the fused L1 kernel keeps the smoothness weight unchanged
    l1 = blur_photometric_loss(blurred, subframes, gt, float(lambda_t_smooth) / (1.0 - lam))
    return (1.0 - lam) * l1 + lam * (1.0 - ssim(blurred, gt.detach()))


def mcmc_regularization(gaussians, opacity_reg=0.01, scale_reg=0.01):
    """3DGS-MCMC's regularisers, opacity_reg * mean|get_opacity| + scale_reg * mean|get_scaling| (unfiltered getters):
    they push unused Gaussians towards transparency, where relocation picks them up.  Two torch reductions,
    differentiable in the raw opacity and scaling."""
    return opacity_reg * gaussians.get_opacity.abs().mean() + scale_reg * gaussians.get_scaling.abs().mean()


def training_loss(blurred, subframes, gt, depths=None, opacity=None, lambda_t_smooth=0.0, lambda_depth_tv=0.0,
                  lambda_hinge=0.0, lambda_dssim=0.0):
    """The reference's loss (train.py:147-163): Ll1 + lambda_t_smooth * L_t_smooth + lambda_depth_tv * L_depth_tv +
    lambda_hinge * L_hinge, with the reference's gating (a term whose weight is 0 is not evaluated).
    lambda_dssim > 0 replaces Ll1 by (1 - lambda_dssim) * Ll1 + lambda_dssim * (1 - SSIM(blurred, gt)).
    depths [F,1,H,W] (query()['depths']), opacity = gaussians._opacity."""
    loss = photometric_loss(blurred, subframes, gt, lambda_t_smooth, lambda_dssim)
    if lambda_depth_tv > 0.0:
        loss = loss + lambda_depth_tv * tv_loss(depths)
    if lambda_hinge > 0.0:
        loss = loss + lambda_hinge * hinge_l2(opacity)
    return loss
