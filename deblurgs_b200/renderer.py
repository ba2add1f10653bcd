"""Drop-in for the reference's `gaussian_renderer` package plus the batched blurry-view entry.

`render` mirrors gaussian_renderer/__init__.py:18-90 of taekkii/deblurgs (same signature, same
returned dict). `render_blurry` replaces the loop of CameraMotionModule.query
(scene/motion.py:138-150): all F sub-frames in one batched rasterizer call, blurred image included.
"""
import math

import torch

from .rasterizer import (DensificationStats, GaussianRasterizationSettings, GaussianRasterizer,
                         rasterize_blurry, render_store_blurry)


def render(viewpoint_camera, pc, bg_color, scaling_modifier=1.0, override_color=None, *_compat, contrib=None):
    """Render the scene from one camera. Background tensor (bg_color) must be on the GPU.

    Also tolerates the upstream-3DGS call form render(cam, pc, pipe, bg_color, ...): a third
    positional argument that is not a Tensor is taken to be `pipe` and ignored.
    Antialiasing follows `pc.antialiasing` (off when the store has no such attribute).  With `pc.filter_3D` set, the
    scales and opacities are Mip-Splatting's filtered ones (`get_scaling_with_3D_filter` / `get_opacity_with_3D_filter`).
    `contrib`: a `rasterizer.ContributionScores` this render adds its contribution scores to.
    """
    if not torch.is_tensor(bg_color):
        bg_color = scaling_modifier
        scaling_modifier = override_color if isinstance(override_color, (int, float)) else 1.0
        override_color = _compat[0] if _compat else None

    screenspace_points = torch.zeros_like(pc.get_xyz, dtype=pc.get_xyz.dtype, requires_grad=True,
                                          device=pc.get_xyz.device) + 0
    try:
        screenspace_points.retain_grad()
    except Exception:
        pass

    tanfovx = math.tan(viewpoint_camera.FoVx * 0.5)
    tanfovy = math.tan(viewpoint_camera.FoVy * 0.5)
    raster_settings = GaussianRasterizationSettings(
        image_height=int(viewpoint_camera.image_height),
        image_width=int(viewpoint_camera.image_width),
        tanfovx=tanfovx,
        tanfovy=tanfovy,
        bg=bg_color,
        scale_modifier=scaling_modifier,
        z_near=pc.z_near,
        z_far=pc.z_far,
        use_sigmoid=pc.use_sigmoid,
        sh_degree=pc.active_sh_degree,
        campos=viewpoint_camera.camera_center,
        prefiltered=False,
        debug=False,
    )
    rasterizer = GaussianRasterizer(raster_settings=raster_settings, antialiasing=getattr(pc, "antialiasing", False),
                                    contrib=contrib)

    shs = None
    colors_precomp = None
    if override_color is None:
        shs = pc.get_features
    else:
        colors_precomp = override_color

    if getattr(pc, "filter_3D", None) is not None:
        opacities, scales = pc.get_opacity_with_3D_filter, pc.get_scaling_with_3D_filter
    else:
        opacities, scales = pc.get_opacity, pc.get_scaling
    rendered_image, rendered_depth, radii = rasterizer(
        means3D=pc.get_xyz,
        means2D=screenspace_points,
        shs=shs,
        colors_precomp=colors_precomp,
        opacities=opacities,
        scales=scales,
        rotations=pc.get_rotation,
        cov3D_precomp=None,
        viewmatrix=viewpoint_camera.world_view_transform,
        projmatrix=viewpoint_camera.full_proj_transform)

    return {"render": rendered_image,
            "depth": rendered_depth,
            "viewspace_points": screenspace_points,
            "visibility_filter": radii > 0,
            "radii": radii}


def render_blurry(world_view_transforms, full_proj_transforms, camera_centers, ref_cam, pc, bg_color,
                  scaling_modifier=1.0, override_color=None, blur_denominator=None, grad_sink=None, *, contrib=None):
    """Render all F sub-frames of a blurry view in one batched call.

    world_view_transforms / full_proj_transforms [F,4,4], camera_centers [F,3]: the MiniCam tensors of
    the sub-frames (e.g. from `pose.bezier_se3_poses`); `ref_cam` supplies image size and FoV.
    The Gaussian activations (pc.get_*) are evaluated once for the whole view, not once per sub-frame.
    Returns the reference's per-render dict with a leading sub-frame axis, plus "blurred".
    Antialiasing, the 3-D filter (`pc.filter_3D`) and `contrib` as in `render`.
    """
    xyz = pc.get_xyz
    F = world_view_transforms.shape[0]
    # Gradient sink for the per-sub-frame screen-space means (the reference allocates zeros_like(xyz)
    # per sub-frame, gaussian_renderer/__init__.py:26): a zero-stride view, so no F*P*3 zero-fill; its
    # .grad is the [F,P,3] tensor the backward kernel writes.
    screenspace_points = torch.zeros(1, dtype=xyz.dtype, device=xyz.device).expand((F,) + tuple(xyz.shape))
    screenspace_points.requires_grad_(True)
    raster_settings = GaussianRasterizationSettings(
        image_height=int(ref_cam.image_height),
        image_width=int(ref_cam.image_width),
        tanfovx=math.tan(ref_cam.FoVx * 0.5),
        tanfovy=math.tan(ref_cam.FoVy * 0.5),
        bg=bg_color,
        scale_modifier=scaling_modifier,
        z_near=pc.z_near,
        z_far=pc.z_far,
        use_sigmoid=pc.use_sigmoid,
        sh_degree=pc.active_sh_degree,
        campos=camera_centers,
        prefiltered=False,
        debug=False,
    )
    stats = DensificationStats()   # filled by the backward pass
    sink = grad_sink if grad_sink is not None else getattr(pc, "grad_sink", None)
    filter3d = getattr(pc, "filter_3D", None)
    if sink is not None and override_color is None and hasattr(pc, "_features_rest"):
        # parameter store + gradient sink (dist.FlatGradBuffer): activations, render and a range-by-range backward in one
        # autograd node, so that the all-reduce of finished rows overlaps the rest of the backward
        color, depth, radii, blurred = render_store_blurry(
            pc._xyz, pc._features_dc, pc._features_rest, pc._scaling, pc._rotation, pc._opacity, screenspace_points,
            world_view_transforms, full_proj_transforms, camera_centers, raster_settings, blur_denominator, stats,
            getattr(pc, "scale_lower_bound", 0.0), getattr(pc, "use_isotropic", False), sink,
            int(getattr(sink, "n_ranges", 4)), getattr(pc, "antialiasing", False), contrib, filter3d)
        return {"render": color, "depth": depth, "blurred": blurred, "viewspace_points": screenspace_points,
                "visibility_filter": radii > 0, "radii": radii, "densification": stats}
    if hasattr(pc, "get_activated"):
        # parameter store with the fused activation kernel (params.activate_gaussians): one launch
        shs, scales, rotations, opacities = pc.get_activated()
    else:
        # any object with the reference's GaussianModel getters
        shs, scales, rotations, opacities = pc.get_features, pc.get_scaling, pc.get_rotation, pc.get_opacity
        if filter3d is not None:
            scales, opacities = pc.get_scaling_with_3D_filter, pc.get_opacity_with_3D_filter
    if override_color is not None:
        shs = None
    color, depth, radii, blurred = rasterize_blurry(
        xyz, screenspace_points, shs, override_color, opacities, scales, rotations, None,
        world_view_transforms, full_proj_transforms, camera_centers, raster_settings, blur_denominator, stats,
        getattr(pc, "antialiasing", False), contrib)
    return {"render": color,
            "depth": depth,
            "blurred": blurred,
            "viewspace_points": screenspace_points,
            "visibility_filter": radii > 0,
            "radii": radii,
            "densification": stats}
