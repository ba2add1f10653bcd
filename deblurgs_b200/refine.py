"""Test-time camera pose refinement (SURVEY.md 8f rank 4): the second consumer of the rasterizer's
view / projection-matrix gradients.

Mirrors test.py of taekkii/deblurgs:
  OptimPoseModel        test.py:39-91    per-view unit quaternion (XYZW, `roma`'s convention) + w2c translation
  optimize_test_pose    test.py:131-186  iNeRF-style loop: L1(render, gt), Adam(rot 5e-5, trans 5e-4, eps 1e-15),
                                         StepLR(step = iters / 20, gamma 0.9), views visited in shuffled epochs
  evaluate_views        test.py:401-439  per-view PSNR / SSIM of the renders against original_image (no LPIPS)
`roma` is not a dependency here: the quaternion algebra lives in `pose.py`. Rendering goes through the
drop-in `renderer.render` (single view) and the update through `params.FusedAdam`.
"""
import copy
import math
import random

import torch
import torch.nn as nn

from . import renderer
from .loss import psnr, ssim
from .params import FusedAdam
from .pose import rotmat_to_unitquat, unitquat_to_rotmat


def get_projection_matrix(znear, zfar, fovX, fovY):
    """Perspective matrix of the reference (utils/graphics_utils.py:51-71): z in [0,1], w = z_view."""
    tan_y, tan_x = math.tan(fovY / 2), math.tan(fovX / 2)
    top, right = tan_y * znear, tan_x * znear
    P = torch.zeros(4, 4)
    P[0, 0] = 2.0 * znear / (2 * right)
    P[1, 1] = 2.0 * znear / (2 * top)
    P[3, 2] = 1.0
    P[2, 2] = zfar / (zfar - znear)
    P[2, 3] = -(zfar * znear) / (zfar - znear)
    return P


class OptimPoseModel(nn.Module):
    """cams: objects with R [3,3] (c2w rotation, as CameraInfo.R), T [3] (w2c translation), image size, FoV,
    znear / zfar and optionally original_image.  forward(idx) returns a copy of cams[idx] carrying
    differentiable world_view_transform / full_proj_transform and its camera_center."""

    def __init__(self, cams, device="cuda"):
        super().__init__()
        self.cams = cams
        rots = torch.stack([torch.as_tensor(c.R, dtype=torch.float64) for c in cams]).to(device)
        trans = torch.stack([torch.as_tensor(c.T, dtype=torch.float64) for c in cams]).to(device)
        self._rot = nn.Parameter(rotmat_to_unitquat(rots).float().contiguous())     # [n,4]
        self._trans = nn.Parameter(trans.float().contiguous())                      # [n,3]

    def forward(self, idx):
        cam = copy.copy(self.cams[idx])
        quat = self._rot[idx] + 1e-8
        rotmat = unitquat_to_rotmat((quat / quat.norm())[None])[0]
        dev = rotmat.device
        # w2c = [R^T | T]; stored transposed, so the upper-left block is R itself and T sits in row 3
        view = torch.cat([torch.cat([rotmat, torch.zeros(3, 1, device=dev)], dim=1),
                          torch.cat([self._trans[idx], torch.ones(1, device=dev)])[None]], dim=0)
        proj_t = get_projection_matrix(cam.znear, cam.zfar, cam.FoVx, cam.FoVy).transpose(0, 1).to(dev)
        cam.world_view_transform = view
        cam.projection_matrix = proj_t
        cam.full_proj_transform = view @ proj_t
        cam.camera_center = torch.inverse(view.detach())[3, :3]
        return cam


def optimize_test_pose(cams, gaussians, bg_color, num_iter_per_view=2000, tone_mapping=None, seed=None,
                       progress=None):
    """Fit the poses of `cams` to a trained scene. Returns (list of refined cameras, per-iteration mean L1)."""
    rng = random.Random(seed)
    n = len(cams)
    model = OptimPoseModel(cams, device=bg_color.device)
    groups = [{"params": [model._rot], "lr": 5e-5, "name": "rot"},
              {"params": [model._trans], "lr": 5e-4, "name": "trans"}]
    optimizer = FusedAdam(groups, lr=5e-4, eps=1e-15)
    step_size = max(num_iter_per_view // 20, 1)
    history = []
    for iteration in range(num_iter_per_view):
        order = list(range(n))
        rng.shuffle(order)
        total = 0.0
        while order:
            idx = order.pop()
            cam = model(idx)
            image = renderer.render(cam, gaussians, bg_color)["render"]
            if tone_mapping is not None:
                image = tone_mapping(image)
            loss = (image.clamp(0.0, 1.0) - cam.original_image).abs().mean()
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            total += float(loss.detach())
        history.append(total / n)
        if (iteration + 1) % step_size == 0:      # StepLR(step_size, gamma=0.9)
            for g in optimizer.param_groups:
                g["lr"] *= 0.9
        if progress is not None:
            progress(iteration, history[-1])
    with torch.no_grad():
        refined = [model(i) for i in range(n)]
    return refined, history


def evaluate_views(cams, gaussians, bg_color, tone_mapping=None):
    """Image quality of a scene at `cams` (e.g. the cameras optimize_test_pose returns): each view rendered without
    gradients, tone-mapped if given, clamped to [0,1] and scored against cam.original_image with one batched SSIM call
    and PSNR.  Returns {"psnr": [per view], "ssim": [per view], "psnr_mean": float, "ssim_mean": float}."""
    with torch.no_grad():
        renders = []
        for cam in cams:
            image = renderer.render(cam, gaussians, bg_color)["render"]
            if tone_mapping is not None:
                image = tone_mapping(image)
            renders.append(image.clamp(0.0, 1.0))
        pred = torch.stack(renders)
        gt = torch.stack([cam.original_image[0:3] for cam in cams]).to(pred)
        ssims = ssim(pred, gt, size_average=False).tolist()
        psnrs = psnr(pred, gt)[:, 0].tolist()
    return {"psnr": psnrs, "ssim": ssims, "psnr_mean": sum(psnrs) / len(psnrs), "ssim_mean": sum(ssims) / len(ssims)}
