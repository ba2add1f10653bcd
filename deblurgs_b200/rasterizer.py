"""Drop-in for the reference's `diff_gaussian_rasterization` Python package, backed by
libdgs_b200.so through its C-ABI.

Mirrors submodules/diff-gaussian-rasterization/diff_gaussian_rasterization/__init__.py of
taekkii/deblurgs: `GaussianRasterizationSettings` (same 13 fields, same order, :172-187),
`GaussianRasterizer` (same forward kwargs / 3-tuple return / error messages, :189-241),
`_RasterizeGaussians` (same saved state and gradient tuple order, :48-170) -- plus the batched
`rasterize_blurry` that renders all F sub-frames of a blurry view in one call.
"""
import ctypes as C
import os
from typing import NamedTuple

import torch
import torch.nn as nn

from . import _lib


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    z_near: float
    z_far: float
    use_sigmoid: bool
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


class _Buffer:
    """Growable device byte buffer handed to the library's resize callback (the reference's
    `resizeFunctional`, rasterize_points.cu:27-33)."""

    def __init__(self, device):
        self.device = device
        self.t = torch.empty(0, dtype=torch.uint8, device=device)
        self.cb = _lib.ALLOC_FN(self._alloc)

    def _alloc(self, _ctx, nbytes):
        try:
            self.t = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            return self.t.data_ptr()
        except Exception:  # never let an exception cross the C boundary
            return 0


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _f32c(t):
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _require_cuda(t, name):
    if not t.is_cuda:
        raise _lib.DgsError("%s must be a CUDA tensor: libdgs_b200 has no CPU path" % name)


# Expected number of (Gaussian, tile) duplicates per workload shape, learnt from the previous call: lets the
# forward size its binning buffer without waiting for the device (dgs_blur_forward_hint).  The first call of a
# shape (and every call with DGS_EXACT_BINNING=1) runs in exact mode with one host synchronisation.
_CAPACITY_HINT = {}
_KEEP_SCRATCH = False
_last_scratch = None
# Fully asynchronous mode (CUDA-graph capture, graph.BlurryViewGraph): a fixed binning capacity, nothing is waited
# for, num_rendered stays on the device; the geometry buffers of the calls made in this mode are collected so that
# the owner can read their status records.
_ASYNC = None   # None, or {"capacity": int, "geoms": [(tensor, P, F), ...]}

CONTRIB_SCALE = 1 << 26     # DGS_CONTRIB_SCALE: fixed-point scale of the contribution weight sums


class ContributionScores:
    """Per-Gaussian contribution scores, accumulated by every forward it is passed to (`contrib=`): over every pixel
    of every rendered sub-frame where the blend used Gaussian g, with its blending weight w = alpha * T,
      weight_sum[g] = sum of w   (LightGaussian's global significance; held as fixed point in `wsum`)
      weight_max[g] = max of w   (RadSplat's pruning score; held as float bits in `wmax`).
    Exact integer sums and maxima: the same bits on every run, batching and sharding of the same sub-frames.
    The scores are those of the stored (with antialiasing: opacity * rho) opacity that is actually blended."""

    def __init__(self, P, device):
        self.wsum = torch.zeros(int(P), dtype=torch.int64, device=device)
        self.wmax = torch.zeros(int(P), dtype=torch.int32, device=device)

    @property
    def num_points(self):
        return self.wsum.shape[0]

    @property
    def weight_sum(self):
        """float64 [P]: sum of the blending weights (each rounded to a multiple of 2^-26)."""
        return self.wsum.double() / CONTRIB_SCALE

    @property
    def weight_max(self):
        """float32 [P]: the largest blending weight."""
        return self.wmax.view(torch.float32)

    def reset(self):
        self.wsum.zero_()
        self.wmax.zero_()

    def _check(self, P, device):
        if self.num_points != P:
            raise _lib.DgsError("ContributionScores holds %d Gaussians but the forward renders %d (the store changed "
                                "size: make new scores after densify / prune)" % (self.num_points, P))
        if self.wsum.device != device:
            raise _lib.DgsError("ContributionScores live on %s, the forward runs on %s" % (self.wsum.device, device))


def _forward_batched(means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                     viewmatrix, projmatrix, campos, bg, H, W, tanfovx, tanfovy, scale_modifier,
                     z_near, z_far, sh_degree, prefiltered, use_sigmoid, want_blur, blur_denominator, exact=False,
                     antialiasing=False, contrib=None):
    """Runs dgs_blur_forward_aa, or dgs_blur_forward_contrib with a `ContributionScores` to accumulate into.
    viewmatrix/projmatrix [F,4,4], campos [F,3]."""
    lib = _lib.load()
    _require_cuda(means3D, "means3D")
    if means3D.dim() != 2 or means3D.shape[1] != 3:
        raise _lib.DgsError("means3D must have dimensions (num_points, 3)")
    dev = means3D.device
    P = means3D.shape[0]
    F = viewmatrix.shape[0]
    if contrib is not None:
        contrib._check(P, dev)
    M = sh.shape[1] if (sh is not None and sh.numel() != 0) else 0
    color = torch.empty((F, 3, H, W), dtype=torch.float32, device=dev)
    depth = torch.empty((F, 1, H, W), dtype=torch.float32, device=dev)
    radii = torch.empty((F, P), dtype=torch.int32, device=dev)
    blur = torch.empty((3, H, W), dtype=torch.float32, device=dev) if want_blur else None
    geom, binning, img = _Buffer(dev), _Buffer(dev), _Buffer(dev)
    num_rendered = C.c_int64(0)
    if P == 0:
        # reference: kernels skipped, zero images returned (rasterize_points.cu:85)
        color.zero_()
        depth.zero_()
        if blur is not None:
            blur.zero_()
        return color, depth, radii, blur, 0, geom.t, binning.t, img.t
    shape_key = (dev.index, P, F, H, W)
    hint = 0 if (exact or os.environ.get("DGS_EXACT_BINNING") == "1") else _CAPACITY_HINT.get(shape_key, 0)
    if _ASYNC is not None:
        hint = int(_ASYNC["capacity"])
    args = (geom.cb, None, binning.cb, None, img.cb, None,
            P, F, int(sh_degree), int(M),
            _lib.ptr(bg), int(W), int(H),
            _lib.ptr(means3D), _lib.ptr(sh), _lib.ptr(colors_precomp),
            _lib.ptr(opacities), _lib.ptr(scales), float(scale_modifier),
            _lib.ptr(rotations), _lib.ptr(cov3Ds_precomp),
            _lib.ptr(viewmatrix), _lib.ptr(projmatrix), _lib.ptr(campos),
            float(tanfovx), float(tanfovy), float(z_near), float(z_far),
            int(bool(prefiltered)), int(bool(use_sigmoid)),
            _lib.ptr(color), _lib.ptr(depth), _lib.ptr(radii),
            _lib.ptr(blur), float(blur_denominator),
            int(hint), None if _ASYNC is not None else C.byref(num_rendered), int(bool(antialiasing)))
    entry = "dgs_blur_forward_aa" if contrib is None else "dgs_blur_forward_contrib"
    with torch.cuda.device(dev):
        if contrib is None:
            rc = lib.dgs_blur_forward_aa(*args, _stream_ptr(dev))
        else:
            rc = lib.dgs_blur_forward_contrib(*args, _lib.ptr(contrib.wsum), _lib.ptr(contrib.wmax), _stream_ptr(dev))
    # drop the ctypes callbacks: they close over the _Buffer objects (a reference cycle), and a cycle
    # would keep hundreds of MB of state buffers alive until Python's cyclic GC runs, forcing the caching
    # allocator to cudaMalloc fresh blocks every step in the meantime
    geom.cb = binning.cb = img.cb = None
    _lib.check(rc, entry)
    if _ASYNC is not None:
        _ASYNC["geoms"].append((geom.t, P, F))
        return color, depth, radii, blur, -1, geom.t, binning.t, img.t    # -1: number of duplicates unknown on the host
    D = int(num_rendered.value)
    _CAPACITY_HINT[shape_key] = D + D // 4 + 65536
    return color, depth, radii, blur, D, geom.t, binning.t, img.t


BWD_BLEND, BWD_GAUSSIANS, BWD_FINISH, BWD_ALL = 1, 2, 4, 7


def _backward_batched(P, F, M, num_rendered, means3D, sh, colors_precomp, opacities, scales, rotations,
                      cov3Ds_precomp, viewmatrix, projmatrix, campos, bg, H, W, tanfovx, tanfovy,
                      scale_modifier, z_near, z_far, sh_degree, use_sigmoid, radii, geom, binning, img,
                      grad_color, grad_depth, want_means2D, grad_blur=None, blur_denominator=1.0, want_stats=False,
                      ranges=None, outputs=None, on_range=None, antialiasing=False):
    """Runs dgs_blur_backward_range_aa (`antialiasing` must be the forward's).  ranges: list of (g0, g1) covering [0, P) -- the per-Gaussian stage is launched
    once per range and `on_range(g0, g1, out)` is called after each (e.g. to start a collective on those rows while
    the next range computes); outputs: preallocated (dmeans3D, dsh, dopacity, dscales, drot) to write into."""
    lib = _lib.load()
    dev = means3D.device
    f32 = dict(dtype=torch.float32, device=dev)
    has_sh = sh is not None and sh.numel() != 0
    has_colors = colors_precomp is not None and colors_precomp.numel() != 0
    has_scales = scales is not None and scales.numel() != 0
    has_cov = cov3Ds_precomp is not None and cov3Ds_precomp.numel() != 0
    # every output below is fully written by the kernels (no zero-fill needed, unlike the reference's
    # 12 torch::zeros per sub-frame, rasterize_points.cu:163-175)
    alloc = torch.zeros if (P == 0 or F == 0) else torch.empty
    dmeans2D = alloc((F, P, 3), **f32) if want_means2D else None
    if outputs is not None:
        dmeans3D, dsh, dopacity, dscales, drot = outputs
    else:
        dmeans3D = alloc((P, 3), **f32)
        dsh = alloc((P, M, 3), **f32) if has_sh else torch.zeros((P, 0, 3), **f32)
        dopacity = alloc((P, 1), **f32)
        dscales = alloc((P, 3), **f32) if has_scales else None
        drot = alloc((P, 4), **f32) if has_scales else None
    dcolors = alloc((P, 3), **f32) if has_colors else None
    dcov = alloc((P, 6), **f32) if has_cov else None
    dview = alloc((F, 4, 4), **f32)
    dproj = alloc((F, 4, 4), **f32)
    stats = alloc((P, 3), **f32) if want_stats else None
    if P == 0 or F == 0:
        return dmeans2D, dmeans3D, dsh, dopacity, dscales, drot, dcolors, dcov, dview, dproj, stats
    scratch = torch.empty(int(lib.dgs_blur_backward_scratch_bytes(P, F)), dtype=torch.uint8, device=dev)

    def call(g0, g1, stages):
        with torch.cuda.device(dev):
            rc = lib.dgs_blur_backward_range_aa(
                P, F, int(sh_degree), int(M), int(num_rendered),
                _lib.ptr(bg), int(W), int(H),
                _lib.ptr(means3D), _lib.ptr(sh), _lib.ptr(colors_precomp),
                _lib.ptr(opacities), _lib.ptr(scales), float(scale_modifier),
                _lib.ptr(rotations), _lib.ptr(cov3Ds_precomp),
                _lib.ptr(viewmatrix), _lib.ptr(projmatrix), _lib.ptr(campos),
                float(tanfovx), float(tanfovy), float(z_near), float(z_far), int(bool(use_sigmoid)),
                _lib.ptr(radii), _lib.ptr(geom), _lib.ptr(binning), _lib.ptr(img),
                _lib.ptr(grad_color), _lib.ptr(grad_depth), _lib.ptr(grad_blur), float(blur_denominator),
                _lib.ptr(scratch),
                _lib.ptr(dmeans2D), _lib.ptr(dmeans3D), _lib.ptr(dsh), _lib.ptr(dopacity),
                _lib.ptr(dscales), _lib.ptr(drot), _lib.ptr(dcolors), _lib.ptr(dcov),
                _lib.ptr(dview), _lib.ptr(dproj), _lib.ptr(stats), int(g0), int(g1), int(stages),
                int(bool(antialiasing)), _stream_ptr(dev))
        _lib.check(rc, "dgs_blur_backward_range_aa")

    if ranges is None:
        call(0, P, BWD_ALL)
    else:
        call(0, 0, BWD_BLEND)
        for (g0, g1) in ranges:
            call(g0, g1, BWD_GAUSSIANS)
            if on_range is not None:
                on_range(g0, g1, (dmeans3D, dsh, dopacity, dscales, drot))
        call(0, 0, BWD_FINISH)
    if _KEEP_SCRATCH:   # test hook: the per-(sub-frame, Gaussian) screen-space gradients the blend backward produced
        global _last_scratch
        _last_scratch = scratch
    return dmeans2D, dmeans3D, dsh, dopacity, dscales, drot, dcolors, dcov, dview, dproj, stats


def _empty_like_input(t):
    return torch.zeros_like(t) if (t is not None and t.numel() != 0) else None


class _RasterizeGaussians(torch.autograd.Function):
    """Single view. Same argument order, saved state and gradient tuple as the reference's
    `_RasterizeGaussians` (diff_gaussian_rasterization/__init__.py:48-170), plus trailing `antialiasing` and `contrib`."""

    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                cov3Ds_precomp, viewmatrix, projmatrix, raster_settings, antialiasing=False, contrib=None):
        rs = raster_settings
        ctx.set_materialize_grads(False)   # an unused output (depth) arrives as None, not as a zero-filled image
        means3D_c, sh_c, colors_c = _f32c(means3D), _f32c(sh), _f32c(colors_precomp)
        opac_c, scales_c, rot_c, cov_c = _f32c(opacities), _f32c(scales), _f32c(rotations), _f32c(cov3Ds_precomp)
        view_c = _f32c(viewmatrix).reshape(1, 4, 4)
        proj_c = _f32c(projmatrix).reshape(1, 4, 4)
        campos_c = _f32c(rs.campos).reshape(1, 3)
        bg_c = _f32c(rs.bg)
        color, depth, radii, _, num_rendered, geom, binning, img = _forward_batched(
            means3D_c, sh_c, colors_c, opac_c, scales_c, rot_c, cov_c, view_c, proj_c, campos_c, bg_c,
            rs.image_height, rs.image_width, rs.tanfovx, rs.tanfovy, rs.scale_modifier, rs.z_near,
            rs.z_far, rs.sh_degree, rs.prefiltered, rs.use_sigmoid, False, 1.0, antialiasing=antialiasing,
            contrib=contrib)
        ctx.raster_settings = rs
        ctx.num_rendered = num_rendered
        ctx.antialiasing = bool(antialiasing)
        ctx.save_for_backward(colors_c, means3D_c, scales_c, rot_c, cov_c, radii, sh_c, opac_c, geom, binning,
                              img, view_c, proj_c, campos_c, bg_c)
        ctx.mark_non_differentiable(radii)
        return color[0], depth[0], radii[0]

    @staticmethod
    def backward(ctx, grad_out_color, grad_out_depth, _):
        rs = ctx.raster_settings
        (colors_c, means3D, scales, rot, cov, radii, sh, opac, geom, binning, img, view, proj, campos,
         bg) = ctx.saved_tensors
        P = means3D.shape[0]
        M = sh.shape[1] if sh.numel() != 0 else 0
        gc = _f32c(grad_out_color) if grad_out_color is not None else None
        gd = _f32c(grad_out_depth) if grad_out_depth is not None else None
        (dmeans2D, dmeans3D, dsh, dopacity, dscales, drot, dcolors, dcov, dview, dproj, _) = _backward_batched(
            P, 1, M, ctx.num_rendered, means3D, sh, colors_c, opac, scales, rot, cov, view, proj, campos, bg,
            rs.image_height, rs.image_width, rs.tanfovx, rs.tanfovy, rs.scale_modifier, rs.z_near, rs.z_far,
            rs.sh_degree, rs.use_sigmoid, radii, geom, binning, img, gc, gd, True, antialiasing=ctx.antialiasing)
        # reference order: means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
        # cov3Ds_precomp, viewmatrix, projmatrix, raster_settings
        return (dmeans3D, dmeans2D[0], dsh if sh.numel() != 0 else None, dcolors, dopacity, dscales, drot, dcov,
                dview[0], dproj[0], None, None, None)


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        viewmatrix, projmatrix, raster_settings, antialiasing=False, contrib=None):
    """`antialiasing`: Mip-Splatting's screen-space filter (include/dgs_b200.h, dgs_blur_forward_aa).
    `contrib`: a `ContributionScores` the forward adds this view's contribution scores to."""
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                     cov3Ds_precomp, viewmatrix, projmatrix, raster_settings, bool(antialiasing),
                                     contrib)


class _RasterizeBlurry(torch.autograd.Function):
    """All F sub-frames of one blurry view. Inputs as `_RasterizeGaussians` except that
    viewmatrix/projmatrix are [F,4,4], campos [F,3] is explicit (no gradient, as in the
    reference where it rides in the settings tuple) and means2D is an [F,P,3] gradient sink.
    Returns (color [F,3,H,W], depth [F,1,H,W], radii [F,P], blurred [3,H,W])."""

    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                viewmatrix, projmatrix, campos, raster_settings, blur_denominator, stats_holder=None,
                antialiasing=False, contrib=None):
        rs = raster_settings
        # outputs the loss does not use (typically the [F,3,H,W] / [F,1,H,W] stacks when only `blurred` is) arrive
        # as None in backward instead of zero-filled tensors the kernel would then have to read
        ctx.set_materialize_grads(False)
        ctx.stats_holder = stats_holder
        means3D_c, sh_c, colors_c = _f32c(means3D), _f32c(sh), _f32c(colors_precomp)
        opac_c, scales_c, rot_c, cov_c = _f32c(opacities), _f32c(scales), _f32c(rotations), _f32c(cov3Ds_precomp)
        view_c, proj_c, campos_c, bg_c = _f32c(viewmatrix), _f32c(projmatrix), _f32c(campos), _f32c(rs.bg)
        F = view_c.shape[0]
        denom = float(blur_denominator) if blur_denominator else float(F)
        color, depth, radii, blur, num_rendered, geom, binning, img = _forward_batched(
            means3D_c, sh_c, colors_c, opac_c, scales_c, rot_c, cov_c, view_c, proj_c, campos_c, bg_c,
            rs.image_height, rs.image_width, rs.tanfovx, rs.tanfovy, rs.scale_modifier, rs.z_near,
            rs.z_far, rs.sh_degree, rs.prefiltered, rs.use_sigmoid, True, denom, antialiasing=antialiasing,
            contrib=contrib)
        ctx.raster_settings = rs
        ctx.num_rendered = num_rendered
        ctx.denom = denom
        ctx.antialiasing = bool(antialiasing)
        ctx.want_means2D = means2D is not None and means2D.requires_grad
        ctx.save_for_backward(colors_c, means3D_c, scales_c, rot_c, cov_c, radii, sh_c, opac_c, geom, binning,
                              img, view_c, proj_c, campos_c, bg_c)
        ctx.mark_non_differentiable(radii)
        return color, depth, radii, blur

    @staticmethod
    def backward(ctx, grad_color, grad_depth, _radii, grad_blur):
        rs = ctx.raster_settings
        (colors_c, means3D, scales, rot, cov, radii, sh, opac, geom, binning, img, view, proj, campos,
         bg) = ctx.saved_tensors
        P = means3D.shape[0]
        F = view.shape[0]
        M = sh.shape[1] if sh.numel() != 0 else 0
        gc = _f32c(grad_color) if grad_color is not None else None
        # blurred = sum_s color_s / denom: its gradient is folded in by the kernel (dL_dblur argument)
        gb = _f32c(grad_blur) if grad_blur is not None else None
        gd = _f32c(grad_depth) if grad_depth is not None else None
        holder = ctx.stats_holder
        (dmeans2D, dmeans3D, dsh, dopacity, dscales, drot, dcolors, dcov, dview, dproj, stats) = _backward_batched(
            P, F, M, ctx.num_rendered, means3D, sh, colors_c, opac, scales, rot, cov, view, proj, campos, bg,
            rs.image_height, rs.image_width, rs.tanfovx, rs.tanfovy, rs.scale_modifier, rs.z_near, rs.z_far,
            rs.sh_degree, rs.use_sigmoid, radii, geom, binning, img, gc, gd, ctx.want_means2D, gb, ctx.denom,
            holder is not None, antialiasing=ctx.antialiasing)
        if holder is not None:
            # denominator of the view's blur = number of sub-frames of the WHOLE view (a rank that renders a shard of
            # the sub-frames still normalises its visible-count by all of them, train.py:193: 1 / len(render_pkgs))
            holder.fill(stats, ctx.denom)
        return (dmeans3D, dmeans2D, dsh if sh.numel() != 0 else None, dcolors, dopacity, dscales, drot, dcov,
                dview, dproj, None, None, None, None, None, None)


class _RenderStoreBlurry(torch.autograd.Function):
    """Parameter store -> blurry view in one autograd node: the activations of the six raw parameter tensors
    (dgs_activate_forward), the batched render, and a backward that finishes the Gaussians range by range -- the
    per-Gaussian rasterizer backward and the activation chain rule of rows [g0, g1) -- so that a gradient sink
    (dist.FlatGradBuffer) can start the NCCL all-reduce of those rows while the next range is computed.
    With a sink the Gaussian gradients are WRITTEN into the sink's views (= the parameters' .grad) and this node
    returns None for them; without one it returns them like any autograd node."""

    @staticmethod
    def forward(ctx, xyz, f_dc, f_rest, scaling, rotation, opacity, means2D, viewmatrix, projmatrix, campos,
                raster_settings, blur_denominator, stats_holder, scale_lb, isotropic, grad_sink, n_ranges,
                antialiasing=False, contrib=None, filter3d=None):
        lib = _lib.load()
        rs = raster_settings
        _require_cuda(xyz, "xyz")
        ctx.set_materialize_grads(False)
        raw = [_f32c(t.detach()) for t in (xyz, f_dc, f_rest, scaling, rotation, opacity)]
        xyz_c, dc_c, rest_c, sc_c, rot_c, op_c = raw
        P = xyz_c.shape[0]
        M = 1 + (rest_c.shape[1] if rest_c.dim() == 3 else 0)
        dev = xyz_c.device
        f32 = dict(dtype=torch.float32, device=dev)
        shs, scales = torch.empty((P, M, 3), **f32), torch.empty((P, 3), **f32)
        rots, opac = torch.empty((P, 4), **f32), torch.empty((P, 1), **f32)
        filt = None if filter3d is None else _f32c(filter3d.detach())
        if filt is not None and filt.numel() != P:
            raise _lib.DgsError("filter_3D holds %d values, the store %d Gaussians" % (filt.numel(), P))
        if P > 0:
            with torch.cuda.device(dev):
                args = (P, M, _lib.ptr(dc_c), _lib.ptr(rest_c), _lib.ptr(sc_c), _lib.ptr(rot_c), _lib.ptr(op_c),
                        float(scale_lb), int(bool(isotropic)), _lib.ptr(shs), _lib.ptr(scales), _lib.ptr(rots),
                        _lib.ptr(opac))
                if filt is None:
                    rc = lib.dgs_activate_forward(*args, _stream_ptr(dev))
                else:
                    rc = lib.dgs_activate_forward_filter3d(*args, filt.data_ptr(), _stream_ptr(dev))
            _lib.check(rc, "dgs_activate_forward")
        view_c, proj_c, campos_c, bg_c = _f32c(viewmatrix), _f32c(projmatrix), _f32c(campos), _f32c(rs.bg)
        F = view_c.shape[0]
        denom = float(blur_denominator) if blur_denominator else float(F)
        color, depth, radii, blur, num_rendered, geom, binning, img = _forward_batched(
            xyz_c, shs, None, opac, scales, rots, None, view_c, proj_c, campos_c, bg_c, rs.image_height,
            rs.image_width, rs.tanfovx, rs.tanfovy, rs.scale_modifier, rs.z_near, rs.z_far, rs.sh_degree,
            rs.prefiltered, rs.use_sigmoid, True, denom, antialiasing=antialiasing, contrib=contrib)
        ctx.raster_settings, ctx.num_rendered, ctx.denom = rs, num_rendered, denom
        ctx.antialiasing = bool(antialiasing)
        ctx.want_means2D = means2D is not None and means2D.requires_grad
        ctx.stats_holder, ctx.sink, ctx.n_ranges = stats_holder, grad_sink, max(1, int(n_ranges))
        ctx.meta = (M, bool(isotropic), f_dc.shape, f_rest.shape, float(scale_lb))
        ctx.filter3d = filt
        ctx.save_for_backward(xyz_c, sc_c, rot_c, op_c, shs, scales, rots, opac, radii, geom, binning, img, view_c,
                              proj_c, campos_c, bg_c)
        ctx.mark_non_differentiable(radii)
        return color, depth, radii, blur

    @staticmethod
    def backward(ctx, grad_color, grad_depth, _radii, grad_blur):
        lib = _lib.load()
        rs = ctx.raster_settings
        (xyz, sc, rot, op, shs, scales, rots, opac, radii, geom, binning, img, view, proj, campos, bg) = ctx.saved_tensors
        M, isotropic, dc_shape, rest_shape, scale_lb = ctx.meta
        filt = ctx.filter3d
        P, F, dev = xyz.shape[0], view.shape[0], xyz.device
        f32 = dict(dtype=torch.float32, device=dev)
        gc = _f32c(grad_color) if grad_color is not None else None
        gb = _f32c(grad_blur) if grad_blur is not None else None
        gd = _f32c(grad_depth) if grad_depth is not None else None
        sink, holder = ctx.sink, ctx.stats_holder
        if sink is not None:
            v = sink.views
            dxyz, ddc, drest, dsc, drot_raw, dop_raw = (v[k] for k in ("xyz", "f_dc", "f_rest", "scaling", "rotation", "opacity"))
            sink.begin()
        else:
            dxyz, ddc, drest = torch.empty((P, 3), **f32), torch.empty(dc_shape, **f32), torch.empty(rest_shape, **f32)
            dsc, drot_raw, dop_raw = torch.empty((P, 3), **f32), torch.empty((P, 4), **f32), torch.empty((P, 1), **f32)
        # activated-space gradients (inputs of the activation chain rule); dL/dxyz needs no chain rule
        dsh, dopac = torch.empty((P, M, 3), **f32), torch.empty((P, 1), **f32)
        dscales, drots = torch.empty((P, 3), **f32), torch.empty((P, 4), **f32)
        n = ctx.n_ranges if P >= 4096 * ctx.n_ranges else 1
        step = -(-P // n)
        step = -(-step // 128) * 128                 # ranges start on a block boundary (keeps 16-B aligned rows)
        ranges = [(g0, min(P, g0 + step)) for g0 in range(0, P, step)] if P > 0 else []
        st = _stream_ptr(dev)

        def after_range(g0, g1, _out):
            rows = g1 - g0
            o = lambda t, w: t.data_ptr() + g0 * w * 4
            args = (rows, M, o(sc, 3), o(rot, 4), o(op, 1), int(isotropic), o(dsh, 3 * M), o(dscales, 3), o(drots, 4),
                    o(dopac, 1), o(ddc, 3), o(drest, 3 * (M - 1)) if M > 1 else None, o(dsc, 3), o(drot_raw, 4),
                    o(dop_raw, 1))
            with torch.cuda.device(dev):
                if filt is None:
                    rc = lib.dgs_activate_backward(*args, st)
                else:
                    rc = lib.dgs_activate_backward_filter3d(*args, scale_lb, o(filt, 1), st)
            _lib.check(rc, "dgs_activate_backward")
            if sink is not None:
                sink.rows_done(g0, g1)

        (dmeans2D, _, _, _, _, _, _, _, dview, dproj, stats) = _backward_batched(
            P, F, M, ctx.num_rendered, xyz, shs, None, opac, scales, rots, None, view, proj, campos, bg,
            rs.image_height, rs.image_width, rs.tanfovx, rs.tanfovy, rs.scale_modifier, rs.z_near, rs.z_far,
            rs.sh_degree, rs.use_sigmoid, radii, geom, binning, img, gc, gd, ctx.want_means2D, gb, ctx.denom,
            holder is not None, ranges=ranges, outputs=(dxyz, dsh, dopac, dscales, drots), on_range=after_range,
            antialiasing=ctx.antialiasing)
        if holder is not None:
            holder.fill(stats, ctx.denom)
        if sink is not None:
            sink.finish()
            return (None, None, None, None, None, None, dmeans2D, dview, dproj) + (None,) * 11
        return (dxyz, ddc, drest, dsc, drot_raw, dop_raw, dmeans2D, dview, dproj) + (None,) * 11


def render_store_blurry(xyz, features_dc, features_rest, scaling, rotation, opacity, means2D, viewmatrix, projmatrix,
                        campos, raster_settings, blur_denominator=None, stats_holder=None, scale_lower_bound=0.0,
                        isotropic=False, grad_sink=None, n_ranges=4, antialiasing=False, contrib=None, filter3d=None):
    """`filter3d` [P,1]: Mip-Splatting's 3-D smoothing filter applied in the fused activations (params.activate_gaussians)."""
    return _RenderStoreBlurry.apply(xyz, features_dc, features_rest, scaling, rotation, opacity, means2D, viewmatrix,
                                    projmatrix, campos, raster_settings, blur_denominator, stats_holder,
                                    scale_lower_bound, isotropic, grad_sink, n_ranges, bool(antialiasing), contrib,
                                    filter3d)


class DensificationStats:
    """Filled by the backward pass of `rasterize_blurry`: per Gaussian, over the sub-frames of the view,
    sum of |dL/dmeans2D[:, :2]| where visible, number of visible sub-frames, and max screen radius --
    exactly what the reference's training loop accumulates sub-frame by sub-frame (train.py:188-193,
    scene/gaussian_model.py:456-458), without materialising or re-reading the [F,P,3] gradient."""

    def __init__(self):
        self.grad_norm_sum = None    # [P,1]
        self.visible_count = None    # [P,1]
        self.max_radius = None       # [P] int32
        self.num_subframes = 0

    def fill(self, stats, F):
        self.grad_norm_sum = stats[:, 0:1]
        self.visible_count = stats[:, 1:2]
        self.max_radius = stats[:, 2].to(torch.int32)
        self.num_subframes = F      # sub-frames of the whole view (the blur denominator), also on a sub-frame shard

    @property
    def ready(self):
        return self.grad_norm_sum is not None


def rasterize_blurry(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                     viewmatrix, projmatrix, campos, raster_settings, blur_denominator=None, stats_holder=None,
                     antialiasing=False, contrib=None):
    empty = torch.Tensor([])
    return _RasterizeBlurry.apply(
        means3D, means2D, sh if sh is not None else empty,
        colors_precomp if colors_precomp is not None else empty, opacities,
        scales if scales is not None else empty, rotations if rotations is not None else empty,
        cov3Ds_precomp if cov3Ds_precomp is not None else empty,
        viewmatrix, projmatrix, campos, raster_settings, blur_denominator, stats_holder, bool(antialiasing), contrib)


class GaussianRasterizer(nn.Module):
    """`antialiasing` and `contrib` (a `ContributionScores` every forward adds to) are constructor arguments, not
    settings fields: GaussianRasterizationSettings keeps the reference's 13 fields."""

    def __init__(self, raster_settings, antialiasing=False, contrib=None):
        super().__init__()
        self.raster_settings = raster_settings
        self.antialiasing = bool(antialiasing)
        self.contrib = contrib

    def markVisible(self, positions, viewmatrix=None, projmatrix=None):
        """Frustum test. The reference reads `raster_settings.viewmatrix`, a field that no longer
        exists (SURVEY.md 2.2: dead code); here the matrices are explicit arguments."""
        lib = _lib.load()
        with torch.no_grad():
            positions = _f32c(positions)
            _require_cuda(positions, "positions")
            if viewmatrix is None:
                viewmatrix = getattr(self.raster_settings, "viewmatrix")  # AttributeError like the reference
                projmatrix = getattr(self.raster_settings, "projmatrix")
            P = positions.shape[0]
            present = torch.zeros(P, dtype=torch.uint8, device=positions.device)
            with torch.cuda.device(positions.device):
                rc = lib.dgs_mark_visible(P, _lib.ptr(positions), _lib.ptr(_f32c(viewmatrix)),
                                          _lib.ptr(_f32c(projmatrix)) if projmatrix is not None else None,
                                          _lib.ptr(present), _stream_ptr(positions.device))
            _lib.check(rc, "dgs_mark_visible")
        return present.bool()

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None, viewmatrix=None, projmatrix=None):
        raster_settings = self.raster_settings

        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')

        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')

        if shs is None:
            shs = torch.Tensor([])
        if colors_precomp is None:
            colors_precomp = torch.Tensor([])
        if scales is None:
            scales = torch.Tensor([])
        if rotations is None:
            rotations = torch.Tensor([])
        if cov3D_precomp is None:
            cov3D_precomp = torch.Tensor([])

        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations,
                                   cov3D_precomp, viewmatrix, projmatrix, raster_settings, self.antialiasing,
                                   self.contrib)
