"""deblurgs_b200: B200-native (sm_100a) blurry-view Gaussian-splatting rasterizer.

A from-scratch implementation of the hot path of taekkii/deblurgs behind the reference's own
API: `GaussianRasterizationSettings` / `GaussianRasterizer` (diff_gaussian_rasterization),
`render` (gaussian_renderer), `distCUDA2` (simple_knn), plus the batched blurry-view entry points.
All compute runs in libdgs_b200.so (hand-written CUDA, C-ABI in include/dgs_b200.h); there is no
CPU or PyTorch fallback.
"""
from . import _lib
from .rasterizer import (GaussianRasterizationSettings, GaussianRasterizer, rasterize_gaussians,
                         rasterize_blurry)
from .renderer import render, render_blurry
from .pose import bezier_se3_poses
from .knn import distCUDA2
from .loss import blur_photometric_loss, hinge_l2, psnr, ssim, training_loss, tv_loss
from .params import FusedAdam, activate_gaussians

__all__ = ["GaussianRasterizationSettings", "GaussianRasterizer", "rasterize_gaussians", "rasterize_blurry",
           "render", "render_blurry", "bezier_se3_poses", "distCUDA2", "blur_photometric_loss", "tv_loss", "hinge_l2",
           "training_loss", "ssim", "psnr", "FusedAdam", "activate_gaussians"]
