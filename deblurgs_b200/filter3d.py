"""Mip-Splatting's 3-D smoothing filter (Yu et al., CVPR 2024): the per-Gaussian sampling depth over the training
cameras and the filter size it sets.

Restates `GaussianModel.compute_3D_filter` of mip-splatting (scene/gaussian_model.py): every Gaussian is bounded from
below at the Nyquist limit of the closest camera that sees it, filter = d_min / max focal * sqrt(0.2).  Here the
cameras are the sub-frame poses along the learned trajectories (`CameraMotionModule.compute_3D_filter`), swept on the
device by `dgs_filter3d_depth` (include/dgs_b200.h); the store applies the filter in its fused activations.
"""
import ctypes as C
import math

import torch

from . import _lib


class SamplingDepth:
    """Per-Gaussian smallest depth over the cameras that see it (`min_depth`, float32 [P], +inf = seen by none) and the
    largest focal length of the cameras swept (`max_focal`).  `add` sweeps a batch of cameras; calls compose, and the
    result is bit-identical for any order or batching of the same cameras."""

    def __init__(self, P, device):
        self.min_depth = torch.full((int(P),), math.inf, dtype=torch.float32, device=device)
        self.max_focal = 0.0

    @torch.no_grad()
    def add(self, xyz, world_view_transforms, width, height, fovx, fovy, z_near):
        """xyz [P,3]; world_view_transforms [C,4,4] (row-vector layout, as MiniCam.world_view_transform); all C cameras
        of one image size and field of view.  A camera sees a Gaussian when its depth exceeds `z_near` and its
        centre projects within 15 % of the image border."""
        P = self.min_depth.shape[0]
        if xyz.shape[0] != P:
            raise ValueError("SamplingDepth holds %d Gaussians, xyz %d" % (P, xyz.shape[0]))
        if not xyz.is_cuda:
            raise _lib.DgsError("SamplingDepth.add needs CUDA tensors: libdgs_b200 has no CPU path")
        lib = _lib.load()
        fx = width / (2.0 * math.tan(fovx / 2.0))
        fy = height / (2.0 * math.tan(fovy / 2.0))
        pts = xyz.detach().float().contiguous()
        views = world_view_transforms.detach().to(pts.device, torch.float32).reshape(-1, 16).contiguous()
        dev = pts.device
        with torch.cuda.device(dev):
            rc = lib.dgs_filter3d_depth(P, _lib.ptr(pts), views.shape[0], _lib.ptr(views), fx, fy, int(width),
                                        int(height), float(z_near), _lib.ptr(self.min_depth),
                                        C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        _lib.check(rc, "dgs_filter3d_depth")
        if views.shape[0] > 0:
            self.max_focal = max(self.max_focal, fx)
        return self

    @torch.no_grad()
    def filter_3D(self):
        """[P,1] filter sizes: min_depth / max_focal * sqrt(0.2), with the Gaussians no camera saw at the largest finite
        depth.  Raises ValueError when no camera saw any Gaussian (the only host round trip)."""
        d = self.min_depth
        seen = torch.isfinite(d)
        if d.numel() == 0 or not bool(seen.any()):
            raise ValueError("no camera sees any Gaussian: the 3-D filter is undefined")
        d_max = torch.where(seen, d, -math.inf).max()
        d = torch.where(seen, d, d_max)
        return (d / self.max_focal * (0.2 ** 0.5))[:, None]
