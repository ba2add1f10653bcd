#!/usr/bin/env python
"""A DeblurGS-style training loop on the deblurgs_b200 API, end to end on synthetic data (needs a B200).

What the reference's train.py does per iteration (train.py:120-215), with this repository's pieces:

  reference                                         here
  ------------------------------------------------  ---------------------------------------------------------
  CameraMotionModule(cam_infos, args)               CameraMotionModule.from_poses(cams, R, t, ...)   (se3_log_map init)
  gaussians.training_setup(opt)                     GaussianParams.training_setup(...)                (FusedAdam, 1 launch/step)
  camera_motion_module.add_training_setup(...)      same name
  query(cam_idx) -> F x render(), stack, mean       query(cam_idx): ONE batched forward for the F sub-frames
  l1_loss + lambda * batchwise_smoothness_loss      training_loss (fused L1 / smoothness kernel each way)
  (1-l) * L1 + l * (1 - ssim)   (--lambda-dssim)    training_loss(..., lambda_dssim=l)  (fused SSIM kernel each way)
  loss.backward()                                   one batched backward (+ pose kernel backward)
  for pkg in render_pkgs: add_densification_stats   add_densification_stats_blurry(pkg)  (computed in the backward)
  clip_grad_value_; optimizer.step(); zero_grad     optimizer.step(clip_grad_value=...); zero_grad
  gaussians.densify_and_prune(threshold, extent)    same name (deblurgs_b200/densify.py; optimizer state follows)

The "ground truth" blurry images are rendered from a hidden scene / trajectories; training starts from perturbed
colours, opacities and trajectories and must bring the photometric loss down.  At the end the deblurred scene is
scored the way DeblurGS is judged: the trained and the hidden scene rendered sharp at each view's true mid-exposure
pose, PSNR / SSIM before and after training (refine.evaluate_views), at full size and at half resolution (a camera of
W/2 x H/2 with the same field of view, scored against the full-size sharp truth averaged over 2x2 pixel boxes).
--antialiasing renders both the hidden and the trained scene with the screen-space antialiasing filter.
--prune-fraction f: at iteration --prune-at (default: half of --iters) every training view is swept for the
contribution scores (CameraMotionModule.accumulate_contribution) and the fraction f of Gaussians with the lowest
blending-weight sum is removed (prune_by_contribution); training then continues on the smaller store.
--filter3d: Mip-Splatting's 3-D smoothing filter on the trained store, computed from the sub-frame poses of every
training view after initialisation, every --filter3d-every iterations and after each densify round.  The views are
also scored at double size (a camera of 2W x 2H with the same field of view, against the hidden scene rendered sharp
at that size without the filter): the zoom-in case the filter is for.
--mcmc: 3DGS-MCMC densification instead of densify_and_prune: every --densify-every iterations the dead Gaussians
(opacity <= 0.005) are relocated onto live ones and the store grows by 5 % up to --cap-max (default 2x --gaussians);
SGLD position noise after every optimizer step and the opacity / scale regularisers (0.01 each) in the loss.

  python examples/train_blurry_views.py [--iters 200] [--views 4] [--gaussians 20000] [--lambda-dssim 0.2]
                                        [--antialiasing] [--prune-fraction 0.5 [--prune-at 100]]
                                        [--filter3d [--filter3d-every 100]] [--mcmc [--cap-max N]]
"""
import argparse
import os
import sys
import time
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deblurgs_b200 import mcmc, renderer, synthetic, training_loss  # noqa: E402
from deblurgs_b200.loss import mcmc_regularization  # noqa: E402
from deblurgs_b200.motion import CameraMotionModule, GaussianParams  # noqa: E402
from deblurgs_b200.pose import bezier_se3_poses  # noqa: E402
from deblurgs_b200.refine import evaluate_views  # noqa: E402


class RefCamera:
    """The fields CameraMotionModule / render read from the reference's Camera objects."""

    def __init__(self, cam, device):
        self.image_width, self.image_height = cam.width, cam.height
        self.FoVx, self.FoVy, self.znear, self.zfar = cam.fovx, cam.fovy, cam.znear, cam.zfar
        self.projection_matrix = cam.projection_matrix_t().to(device)
        self.original_image = None


class SharpView:
    """A camera at one fixed pose (what renderer.render reads), scored against `original_image`."""

    def __init__(self, cam, view, proj, campos, image):
        self.image_width, self.image_height = cam.width, cam.height
        self.FoVx, self.FoVy = cam.fovx, cam.fovy
        self.world_view_transform, self.full_proj_transform, self.camera_center = view, proj, campos
        self.original_image = image


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--views", type=int, default=4)
    ap.add_argument("--gaussians", type=int, default=20000)
    ap.add_argument("--subframes", type=int, default=8)
    ap.add_argument("--width", type=int, default=200)
    ap.add_argument("--height", type=int, default=136)
    ap.add_argument("--densify-every", type=int, default=100, help="0: never")
    ap.add_argument("--lambda-dssim", type=float, default=0.0, help="weight of the D-SSIM term (3DGS uses 0.2)")
    ap.add_argument("--antialiasing", action="store_true", help="screen-space antialiasing filter (Mip-Splatting)")
    ap.add_argument("--prune-fraction", type=float, default=0.0,
                    help="prune this fraction of Gaussians by contribution score (0: never)")
    ap.add_argument("--prune-at", type=int, default=None, help="iteration of the contribution pruning (default iters/2)")
    ap.add_argument("--filter3d", action="store_true", help="3-D smoothing filter on the trained store (Mip-Splatting)")
    ap.add_argument("--filter3d-every", type=int, default=100, help="recompute the 3-D filter every N iterations")
    ap.add_argument("--mcmc", action="store_true", help="3DGS-MCMC relocation / growth / SGLD noise instead of "
                    "densify_and_prune")
    ap.add_argument("--cap-max", type=int, default=None, help="--mcmc: Gaussian budget (default 2x --gaussians)")
    args = ap.parse_args()
    cap_max = 2 * args.gaussians if args.cap_max is None else args.cap_max
    mcmc_gen = torch.Generator().manual_seed(7)
    prune_at = args.iters // 2 if args.prune_at is None else args.prune_at
    if args.width % 2 or args.height % 2:
        raise SystemExit("--width and --height must be even (the half-resolution views average 2x2 pixel boxes)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    order, F = 3, args.subframes

    cam = synthetic.make_camera(args.width, args.height)
    scene = synthetic.make_scene(args.gaussians, cam, seed=0).to(dev)
    bg = torch.zeros(3, device=dev)

    # ---- hidden truth: one trajectory per view around the base pose; blurry observations rendered from it
    truth = GaussianParams.from_scene(scene, antialiasing=args.antialiasing)
    cams = [RefCamera(cam, dev) for _ in range(args.views)]
    true_traj = [synthetic.make_trajectory(F, order, seed=10 + i).to(dev) for i in range(args.views)]
    base = torch.tensor([synthetic.BASE_SE3], dtype=torch.float32, device=dev).repeat(args.views, 1)
    oracle_cmm = CameraMotionModule(cams, base, curve_order=order, num_subframes=F)
    with torch.no_grad():
        for i, t in enumerate(true_traj):
            oracle_cmm._trans._control_points[i].copy_(t.ctrl_trans)
            oracle_cmm._rot._control_points[i].copy_(t.ctrl_rot)
    oracle_cmm.link_gaussian(truth)
    with torch.no_grad():
        for i in range(args.views):
            cams[i].original_image = oracle_cmm.query(i, "all", background=bg)["blurred"].clone()

    # ---- the model being trained: same geometry, perturbed appearance; trajectories initialised from the mid pose
    g = torch.Generator().manual_seed(123)
    gauss = GaussianParams.from_scene(scene, antialiasing=args.antialiasing)
    with torch.no_grad():
        gauss._features_dc.add_(0.5 * torch.randn(gauss._features_dc.shape, generator=g).to(dev))
        gauss._features_rest.mul_(0.0)
        gauss._opacity.mul_(0.7)
    opt = gauss.training_setup(position_lr_init=1.6e-5, feature_lr=0.01, opacity_lr=0.02, scaling_lr=0.002,
                               rotation_lr=0.001)
    # mid-trajectory camera pose of every view -> (c2w rotation, camera position), as COLMAP would give them
    half_cam = types.SimpleNamespace(width=cam.width // 2, height=cam.height // 2, fovx=cam.fovx, fovy=cam.fovy)
    double_cam = types.SimpleNamespace(width=cam.width * 2, height=cam.height * 2, fovx=cam.fovx, fovy=cam.fovy)
    mid_R, mid_t, sharp, sharp_half, sharp_double = [], [], [], [], []
    for t in true_traj:
        view, proj, campos = bezier_se3_poses(t.ctrl_trans, t.ctrl_rot, torch.tensor([0.5], device=dev),
                                              cams[0].projection_matrix)
        mid_R.append(view[0, :3, :3])
        mid_t.append(campos[0])
        with torch.no_grad():     # the hidden scene, sharp at the true mid-exposure pose: what deblurring should recover
            v = SharpView(cam, view[0], proj[0], campos[0], None)
            v.original_image = renderer.render(v, truth, bg)["render"].clamp(0.0, 1.0)
        sharp.append(v)
        # the same pose and field of view at half the resolution, scored against the truth box-filtered to that size
        box = torch.nn.functional.avg_pool2d(v.original_image[None], 2)[0]
        sharp_half.append(SharpView(half_cam, view[0], proj[0], campos[0], box))
        with torch.no_grad():     # zoom-in: the same pose and field of view at twice the resolution
            v2 = SharpView(double_cam, view[0], proj[0], campos[0], None)
            v2.original_image = renderer.render(v2, truth, bg)["render"].clamp(0.0, 1.0)
        sharp_double.append(v2)
    cmm = CameraMotionModule.from_poses(cams, torch.stack(mid_R), torch.stack(mid_t), curve_order=order,
                                        num_subframes=F)
    cmm.link_gaussian(gauss)
    if args.filter3d:
        cmm.compute_3D_filter()
    before, before_half, before_double = (evaluate_views(v, gauss, bg) for v in (sharp, sharp_half, sharp_double))
    cmm.add_training_setup(gauss, {"curve_rot": 2e-4, "curve_trans": 2e-3, "curve_alignment": 0.0})

    lam0, lam1 = 1e-3, 1e-5     # lambda_t_smooth_init / final (arguments/__init__.py:97-98)
    log, t0 = [], time.perf_counter()
    t_prune, it_prune = None, 0
    for it in range(args.iters):
        if args.prune_fraction > 0 and it == prune_at:
            torch.cuda.synchronize()
            t_prune, it_prune = time.perf_counter(), it
            n_before = gauss.get_xyz.shape[0]
            scores = cmm.accumulate_contribution(bg)
            gauss.prune_by_contribution(scores, fraction=args.prune_fraction)
            torch.cuda.synchronize()
            print("iter %4d  contribution prune: %d -> %d Gaussians (sweep + prune %.1f ms); %.2f ms / iteration before"
                  % (it, n_before, gauss.get_xyz.shape[0], 1e3 * (time.perf_counter() - t_prune),
                     1e3 * (t_prune - t0) / max(it, 1)), flush=True)
            t_prune = time.perf_counter()
        idx = it % args.views
        lam = lam0 * (lam1 / lam0) ** (it / max(args.iters - 1, 1))
        out = cmm.query(idx, "all", background=bg)
        loss = training_loss(out["blurred"], out["subframes"], out["gt"], lambda_t_smooth=lam,
                             lambda_dssim=args.lambda_dssim)
        if args.mcmc:
            loss = loss + mcmc_regularization(gauss)
        loss.backward()
        with torch.no_grad():
            gauss.add_densification_stats_blurry(out["batched"])    # train.py:188-193, from the backward's epilogue
        opt.step(clip_grad_value=1.0)
        opt.zero_grad(set_to_none=True)
        if args.mcmc:
            mcmc.add_sgld_noise(gauss, opt.param_groups[0]["lr"], it)
        if args.mcmc and args.densify_every and it > 0 and it % args.densify_every == 0 and it < args.iters - 1:
            n_before = gauss.get_xyz.shape[0]
            n_moved = gauss.relocate_gs(generator=mcmc_gen)
            n_added = gauss.add_new_gs(cap_max, generator=mcmc_gen)
            print("iter %4d  MCMC: %d relocated, %d added: %d -> %d Gaussians (cap %d)"
                  % (it, n_moved, n_added, n_before, gauss.get_xyz.shape[0], cap_max), flush=True)
            if args.filter3d and n_added:
                cmm.compute_3D_filter()
        elif args.densify_every and it > 0 and it % args.densify_every == 0 and it < args.iters - 1:
            n_before = gauss.get_xyz.shape[0]
            gauss.densify_and_prune(max_grad=2e-4, extent=5.0)       # train.py:195-196
            print("iter %4d  densify/prune: %d -> %d Gaussians" % (it, n_before, gauss.get_xyz.shape[0]), flush=True)
            if args.filter3d:
                cmm.compute_3D_filter()
        elif args.filter3d and args.filter3d_every and it > 0 and it % args.filter3d_every == 0:
            cmm.compute_3D_filter()
        if it % max(args.iters // 10, 1) == 0 or it == args.iters - 1:
            log.append((it, float(loss.detach())))
            print("iter %4d  loss %.5f" % log[-1], flush=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if t_prune is not None:
        print("%.2f ms / iteration after the contribution prune; %d Gaussians at the end"
              % (1e3 * (time.perf_counter() - t_prune) / max(args.iters - it_prune, 1), gauss.get_xyz.shape[0]))
    print("%d iterations in %.2f s (%.2f ms / blurry view incl. optimizer); loss %.5f -> %.5f; "
          "densification: %d Gaussians seen, max screen radius %d px"
          % (args.iters, dt, 1e3 * dt / args.iters, log[0][1], log[-1][1], int((gauss.denom > 0).sum()),
             int(gauss.max_radii2D.max())))
    after, after_half, after_double = (evaluate_views(v, gauss, bg) for v in (sharp, sharp_half, sharp_double))
    for label, b, a in (("full size %dx%d" % (cam.width, cam.height), before, after),
                        ("half size %dx%d" % (half_cam.width, half_cam.height), before_half, after_half),
                        ("double size %dx%d" % (double_cam.width, double_cam.height), before_double, after_double)):
        print("sharp mid-exposure views vs the hidden scene, %s, antialiasing %s, 3-D filter %s: PSNR %.2f -> %.2f dB, "
              "SSIM %.4f -> %.4f" % (label, "on" if args.antialiasing else "off", "on" if args.filter3d else "off",
                                     b["psnr_mean"], a["psnr_mean"], b["ssim_mean"], a["ssim_mean"]))
    assert log[-1][1] < 0.8 * log[0][1], "training did not reduce the loss"


if __name__ == "__main__":
    main()
