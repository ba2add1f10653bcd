"""Host-side mirror of the reference's camera-motion interface for the hot path.

Mirrors, for curve_type == "se3" (the reference default, arguments/__init__.py:49-74):
  BezierModel                 scene/bezier.py:20-85       (control points [n, C+1, d])
  CameraMotionModule.query / get_trajectory / _sample_nu_from_alignment
                              scene/motion.py:78-178, 209-219
  MiniCam                     scene/cameras.py:63-74
  GaussianModel getters       scene/gaussian_model.py:114-137, scene/gaussian_activation.py:29-52
The sub-frame loop of `query` is replaced by ONE batched render (`renderer.render_blurry`) and the
pose chain by the on-device generator (`pose.bezier_se3_poses`); names, arguments and the returned
dictionary keep the reference's meaning. Also provided (SURVEY.md 8f rank 4): initialisation of the
control points from camera poses (`from_poses`, the reference's `_set_initial_parameters` with
`se3_log_map`), `add_training_setup`, and curve_type == "quarternion_cartesian" (roma-free quaternion
algebra in `pose.py`; pose chain in torch, rendering on the same batched kernels). Dataset loading and
save/load are outside the hot path and not provided.
"""
import math

import torch
import torch.nn as nn

from . import renderer
from .densify import DensificationMixin
from .params import FusedAdam, activate_gaussians
from .pose import (bezier_se3_poses, c2w_to_minicam_tensors, rotmat_to_unitquat, se3_log_map,
                   unitquat_to_rotmat)


def inverse_sigmoid(x):
    return torch.log(x / (1 - x))


class MiniCam:
    """Same fields as the reference's MiniCam; camera_center is supplied (it equals the
    camera-to-world translation) instead of being obtained from a matrix inverse."""

    def __init__(self, width, height, fovy, fovx, znear, zfar, world_view_transform, full_proj_transform,
                 camera_center=None):
        self.image_width = width
        self.image_height = height
        self.FoVy = fovy
        self.FoVx = fovx
        self.znear = znear
        self.zfar = zfar
        self.world_view_transform = world_view_transform
        self.full_proj_transform = full_proj_transform
        if camera_center is None:
            camera_center = torch.inverse(world_view_transform)[3][:3]
        self.camera_center = camera_center


class BezierModel(nn.Module):
    """[n, C+1, d] control points; sample = sum_k binom(C,k) t^(C-k) (1-t)^k ctrl[k]."""

    def __init__(self, initial_points, curve_order, initial_noise=0.001, generator=None):
        super().__init__()
        self.curve_order = curve_order
        pts = initial_points.float()[:, None, :].repeat(1, curve_order + 1, 1)
        noise = torch.randn(pts.shape, generator=generator).to(pts.device) * initial_noise
        self._control_points = nn.Parameter((pts + noise).contiguous().requires_grad_(True))

    @property
    def device(self):
        return self._control_points.device

    def __len__(self):
        return self._control_points.shape[0]

    def forward(self, t, idx):
        """[f] -> [f, d]: sum_k binom(C,k) t^(C-k) (1-t)^k ctrl[idx, k] in torch (scene/bezier.py:54-83; fp64
        like the reference, whose binomials are fp64). The se3 curve type does this inside the pose kernel."""
        C_ = self.curve_order
        binom = torch.tensor([float(math.comb(C_, k)) for k in range(C_ + 1)], dtype=torch.float64, device=t.device)
        k = torch.arange(C_ + 1, device=t.device)
        coeff = (t[:, None] ** (C_ - k)) * ((1 - t)[:, None] ** k) * binom
        return (coeff[:, :, None] * self._control_points[idx][None]).sum(dim=1)


class GaussianParams(DensificationMixin):
    """Minimal stand-in for the reference's GaussianModel on the hot path: raw parameters plus the
    activations `render` reads (opacity = clamp(.,0,1), scale = exp(.) + lb, rotation = normalize,
    features = cat(dc, rest)), the optimizer (`training_setup`) and the densify / prune mechanics
    (`densify.DensificationMixin`)."""

    def __init__(self, xyz, features_dc, features_rest, scaling, rotation, opacity, active_sh_degree,
                 z_near=0.2, z_far=100.0, use_sigmoid=False, scale_lower_bound=0.0, use_isotropic=False,
                 antialiasing=False):
        self._xyz = nn.Parameter(xyz.contiguous())
        self._features_dc = nn.Parameter(features_dc.contiguous())
        self._features_rest = nn.Parameter(features_rest.contiguous())
        self._scaling = nn.Parameter(scaling.contiguous())
        self._rotation = nn.Parameter(rotation.contiguous())
        self._opacity = nn.Parameter(opacity.contiguous())
        self.active_sh_degree = active_sh_degree
        self.z_near = z_near
        self.z_far = z_far
        self.use_sigmoid = use_sigmoid
        self.scale_lower_bound = scale_lower_bound
        self.use_isotropic = use_isotropic
        self.antialiasing = antialiasing   # screen-space antialiasing filter, read by renderer.render / render_blurry
        # Mip-Splatting's 3-D smoothing filter [P,1] (CameraMotionModule.compute_3D_filter); None: off
        self.filter_3D = None
        self.optimizer = None
        self.grad_sink = None      # optional dist.FlatGradBuffer.for_gaussians(self): gradients all-reduced under the backward

    @classmethod
    def from_scene(cls, scene, **kw):
        """Build from activated synthetic values (synthetic.Scene): stores log-scales etc."""
        return cls(scene.means3D.clone(), scene.shs[:, :1, :].clone(), scene.shs[:, 1:, :].clone(),
                   torch.log(scene.scales), scene.rotations.clone(), scene.opacities.clone(), scene.sh_degree, **kw)

    def parameters(self):
        return [self._xyz, self._features_dc, self._features_rest, self._scaling, self._rotation, self._opacity]

    # ---- densification bookkeeping (reference: scene/gaussian_model.py:456-458, train.py:188-193)
    def _ensure_stats(self):
        if not hasattr(self, "xyz_gradient_accum"):
            P, dev = self._xyz.shape[0], self._xyz.device
            self.xyz_gradient_accum = torch.zeros((P, 1), device=dev)
            self.denom = torch.zeros((P, 1), device=dev)
            self.max_radii2D = torch.zeros(P, device=dev)

    def add_densification_stats(self, viewspace_point_tensor, update_filter, denom_count):
        """Reference semantics, one sub-frame at a time. `viewspace_point_tensor` may be the [F,P,3] sink of
        a batched render together with its sub-frame index: pass `(tensor, s)`."""
        self._ensure_stats()
        if isinstance(viewspace_point_tensor, tuple):
            t, s = viewspace_point_tensor
            grad = t.grad[s]
        else:
            grad = viewspace_point_tensor.grad
        self.xyz_gradient_accum[update_filter] += torch.norm(grad[update_filter, :2], dim=-1, keepdim=True)
        self.denom[update_filter] += denom_count

    @torch.no_grad()
    def add_densification_stats_blurry(self, pkg):
        """The whole loop `for render_pkg in render_pkgs: max_radii2D[...] = max(...);
        add_densification_stats(..., 1/len(render_pkgs))` of the reference (train.py:188-193) for one batched
        render, from the statistics the backward kernel produced in the same pass."""
        self._ensure_stats()
        st = pkg["densification"]
        if not st.ready:
            raise RuntimeError("densification statistics are produced by the backward pass: call loss.backward() first")
        self.xyz_gradient_accum += st.grad_norm_sum
        self.denom += st.visible_count / float(st.num_subframes)
        self.max_radii2D = torch.max(self.max_radii2D, st.max_radius.to(self.max_radii2D.dtype))

    def training_setup(self, position_lr_init=0.00016, feature_lr=0.0025, opacity_lr=0.05, scaling_lr=0.005,
                       rotation_lr=0.001, spatial_lr_scale=1.0, percent_dense=0.01, optimizer_cls=None):
        """The reference's optimizer (scene/gaussian_model.py:175-190: Adam, eps=1e-15, one parameter per
        named group), stepped by one fused launch (`params.FusedAdam`)."""
        groups = [
            {"params": [self._xyz], "lr": position_lr_init * spatial_lr_scale, "name": "xyz"},
            {"params": [self._features_dc], "lr": feature_lr, "name": "f_dc"},
            {"params": [self._features_rest], "lr": feature_lr / 20.0, "name": "f_rest"},
            {"params": [self._opacity], "lr": opacity_lr, "name": "opacity"},
            {"params": [self._scaling], "lr": scaling_lr, "name": "scaling"},
            {"params": [self._rotation], "lr": rotation_lr, "name": "rotation"},
        ]
        self.percent_dense = percent_dense
        self.optimizer = (optimizer_cls or FusedAdam)(groups, lr=0.0, eps=1e-15)
        return self.optimizer

    def get_activated(self):
        """(get_features, get_scaling, get_rotation, get_opacity) from ONE fused launch; what the batched
        renderer reads once per blurry view.  With `filter_3D` set, the scaling and opacity are the filtered ones
        (get_scaling_with_3D_filter / get_opacity_with_3D_filter)."""
        return activate_gaussians(self._features_dc, self._features_rest, self._scaling, self._rotation,
                                  self._opacity, self.scale_lower_bound, self.use_isotropic, self.filter_3D)

    @property
    def get_xyz(self):
        return self._xyz

    @property
    def get_scaling(self):
        if self.use_isotropic:
            return torch.exp(self._scaling[:, :1].expand(-1, 3)) + self.scale_lower_bound
        return torch.exp(self._scaling) + self.scale_lower_bound

    @property
    def get_rotation(self):
        return torch.nn.functional.normalize(self._rotation)

    @property
    def get_opacity(self):
        return self._opacity.clamp(0.0, 1.0)

    @property
    def get_features(self):
        return torch.cat((self._features_dc, self._features_rest), dim=1)

    # ---- Mip-Splatting's 3-D filter in torch (scene/gaussian_model.py get_*_with_3D_filter): what `renderer.render`
    # reads, and the statement the fused kernel is tested against.  The opacity factor sqrt(det1 / det2) is written
    # as the product of per-axis ratios s_i / s'_i, which does not underflow in fp32 for tiny scales.
    @property
    def get_scaling_with_3D_filter(self):
        s = self.get_scaling
        if self.filter_3D is None:
            return s
        return torch.sqrt(torch.square(s) + torch.square(self.filter_3D))

    @property
    def get_opacity_with_3D_filter(self):
        o = self.get_opacity
        if self.filter_3D is None:
            return o
        r = self._filter_3D_ratios()
        return o * r[:, 0:1] * r[:, 1:2] * r[:, 2:3]

    def _filter_3D_ratios(self):
        s = self.get_scaling
        return s / torch.sqrt(torch.square(s) + torch.square(self.filter_3D))


class CameraMotionModule:
    """Per-image Bezier trajectory in se(3) and the blurry-view query.

    cameras: list of reference cameras (need image_width/height, FoVx/FoVy, znear/zfar,
    projection_matrix [4,4] (already transposed, as in scene/cameras.py:58) and optionally
    original_image). initial_se3: [n,6] = [log_translation | log_rotation] of each image's c2w.
    """

    def __init__(self, cameras, initial_se3, curve_order=9, num_subframes=21, curve_random_sample=False,
                 generator=None, curve_type="se3"):
        """initial_se3: [n,6] for curve_type "se3"; for "quarternion_cartesian" a tuple
        (unit quaternions [n,4] XYZW, camera positions [n,3]) (use `from_poses` to build either)."""
        self.curve_order = curve_order
        self.n_subframes = num_subframes
        self.curve_type = curve_type
        self.curve_random_sample = curve_random_sample
        self.gaussians = None
        self.original_cam = cameras
        if curve_type == "se3":
            self._trans = BezierModel(initial_se3[:, :3], curve_order, generator=generator)
            self._rot = BezierModel(initial_se3[:, 3:], curve_order, generator=generator)
        elif curve_type == "quarternion_cartesian":
            quats, positions = initial_se3
            self._rot = BezierModel(quats, curve_order, generator=generator)
            self._trans = BezierModel(positions, curve_order, initial_noise=0.01, generator=generator)
            initial_se3 = positions
        else:
            raise NotImplementedError(curve_type)
        n, f = initial_se3.shape[0], num_subframes
        nu0 = torch.linspace(1 / (f - 1), 1.0 - (1 / (f - 1)), f - 2) if f > 2 else torch.zeros(0)
        self._nu = nn.Parameter(inverse_sigmoid(nu0)[None, :].repeat(n, 1).to(initial_se3.device).contiguous()
                                .requires_grad_(True))

    @classmethod
    def from_poses(cls, cameras, rotations, translations, curve_type="se3", **kw):
        """The reference's constructor path (scene/motion.py:36-49, 180-207): `rotations` [n,3,3] are the
        c2w rotations (CameraInfo.R), `translations` [n,3] the camera positions (-T @ R^T). se3: control
        points start at se3_log_map of the transposed c2w matrix; quaternion: at (unit quaternion, position)."""
        n = rotations.shape[0]
        if curve_type == "se3":
            c2w = torch.zeros(n, 4, 4, dtype=rotations.dtype, device=rotations.device)
            c2w[:, :3, :3] = rotations.transpose(-2, -1)
            c2w[:, 3, :3] = translations
            c2w[:, 3, 3] = 1.0
            init = se3_log_map(c2w)
        elif curve_type == "quarternion_cartesian":
            init = (rotmat_to_unitquat(rotations), translations)
        else:
            raise NotImplementedError(curve_type)
        return cls(cameras, init, curve_type=curve_type, **kw)

    def add_training_setup(self, gaussians, lr_dict):
        """Append the curve parameters to the Gaussians' optimizer as groups 'curve_rot', 'curve_trans',
        'curve_alignment', replacing earlier curve groups and their state (scene/motion.py:63-77)."""
        opt = gaussians.optimizer
        for group in opt.param_groups:
            if "curve_" in group["name"] and group["params"][0] in opt.state:
                del opt.state[group["params"][0]]
        opt.param_groups = [e for e in opt.param_groups if "curve_" not in e["name"]]
        opt.add_param_group({"params": [self._rot._control_points], "lr": lr_dict["curve_rot"], "name": "curve_rot"})
        opt.add_param_group({"params": [self._trans._control_points], "lr": lr_dict["curve_trans"],
                             "name": "curve_trans"})
        opt.add_param_group({"params": [self._nu], "lr": lr_dict["curve_alignment"], "name": "curve_alignment"})

    def __len__(self):
        return len(self._trans)

    @property
    def device(self):
        return self._trans.device

    def link_gaussian(self, gaussians):
        self.gaussians = gaussians

    def parameters(self):
        return [self._trans._control_points, self._rot._control_points, self._nu]

    def _sample_nu_from_alignment(self, idx):
        device = self._nu.device
        nu_mid = torch.sigmoid(self._nu[idx])
        if self.curve_random_sample:
            nu_mid = nu_mid + torch.rand_like(nu_mid) / self.n_subframes - (1 / (2 * self.n_subframes))
        return torch.cat([torch.zeros(1, device=device), nu_mid, torch.ones(1, device=device)]) \
            .clamp(0.0, 1.0).sort().values

    def get_trajectory_tensors(self, idx, nu=None):
        """(world_view_transform [F,4,4], full_proj_transform [F,4,4], camera_center [F,3])."""
        if nu is None:
            nu = self._sample_nu_from_alignment(idx)
        ref_cam = self.original_cam[0]
        if self.curve_type == "quarternion_cartesian":
            # scene/motion.py:242-246: Bezier in quaternion components, renormalised, positions in R^3
            q = self._rot(nu, idx)
            q = q / q.norm(dim=1, keepdim=True)
            return c2w_to_minicam_tensors(unitquat_to_rotmat(q), self._trans(nu, idx), ref_cam.projection_matrix)
        return bezier_se3_poses(self._trans._control_points[idx], self._rot._control_points[idx], nu,
                                ref_cam.projection_matrix)

    def get_trajectory(self, idx, t=None):
        """List of MiniCam objects, as the reference returns."""
        view, proj, campos = self.get_trajectory_tensors(idx, t)
        ref = self.original_cam[0]
        return [MiniCam(ref.image_width, ref.image_height, ref.FoVy, ref.FoVx, ref.znear, ref.zfar,
                        view[i], proj[i], campos[i]) for i in range(view.shape[0])]

    def get_gt_image(self, idx):
        return getattr(self.original_cam[idx], "original_image", None)

    def query(self, cam_idx, subframe_indice="all", post_process=None, background="random", contrib=None):
        """Render a blurry view. Same arguments and returned keys as the reference
        (scene/motion.py:78-160): 'blurred', 'gt', 'subframes', 'depths', 'render_pkgs'.
        `contrib`: a `rasterizer.ContributionScores` the view's sub-frames add their contribution scores to."""
        assert self.gaussians is not None
        gaussians = self.gaussians
        if isinstance(background, str) and background == "random":
            bg = torch.rand(3, device=gaussians.get_xyz.device)
        else:
            bg = background

        if isinstance(subframe_indice, str) and subframe_indice == "all":
            nu = None
        else:
            nu = self._sample_nu_from_alignment(cam_idx)
            if isinstance(subframe_indice, int):
                subfr_idx = torch.linspace(0, nu.shape[0] - 1, subframe_indice, device=nu.device).long()
            else:
                subfr_idx = subframe_indice
            nu = nu[subfr_idx]
        view, proj, campos = self.get_trajectory_tensors(cam_idx, nu)
        pkg = renderer.render_blurry(view, proj, campos, self.original_cam[0], gaussians, bg, contrib=contrib)

        blurred = pkg["blurred"]
        if post_process is not None:
            blurred = post_process(blurred)
        F = view.shape[0]
        render_pkgs = [{"render": pkg["render"][s], "depth": pkg["depth"][s],
                        "viewspace_points": pkg["viewspace_points"], "viewspace_index": s,
                        "visibility_filter": pkg["visibility_filter"][s], "radii": pkg["radii"][s]}
                       for s in range(F)]
        return {"blurred": blurred, "gt": self.get_gt_image(cam_idx), "subframes": pkg["render"],
                "depths": pkg["depth"], "render_pkgs": render_pkgs, "batched": pkg}

    @torch.no_grad()
    def compute_3D_filter(self, cam_indices=None):
        """Mip-Splatting's compute_3D_filter over the sub-frame poses of the training views `cam_indices` (default:
        all): sets and returns `gaussians.filter_3D` [P,1].  When the store already holds a filter of this size it is
        overwritten in place, so that a captured `graph.BlurryViewGraph` replays with the new values."""
        from .filter3d import SamplingDepth
        assert self.gaussians is not None
        g, ref = self.gaussians, self.original_cam[0]
        xyz = g.get_xyz
        depth = SamplingDepth(xyz.shape[0], xyz.device)
        for idx in (range(len(self)) if cam_indices is None else cam_indices):
            view, _, _ = self.get_trajectory_tensors(idx)
            depth.add(xyz, view, ref.image_width, ref.image_height, ref.FoVx, ref.FoVy, g.z_near)
        f = depth.filter_3D()
        if g.filter_3D is not None and g.filter_3D.shape == f.shape and g.filter_3D.device == f.device:
            g.filter_3D.copy_(f)
        else:
            g.filter_3D = f
        return g.filter_3D

    @torch.no_grad()
    def accumulate_contribution(self, background, cam_indices=None, scores=None):
        """Contribution scores of the linked Gaussians over the training views: renders every sub-frame of the views
        `cam_indices` (default: all) and returns `scores` (a new `rasterizer.ContributionScores` when None) with
        their weights added.  Antialiasing follows the store, like every render, so the scores measure the opacity
        that is actually blended.  Feed them to `gaussians.prune_by_contribution`."""
        from .rasterizer import ContributionScores
        assert self.gaussians is not None
        if scores is None:
            scores = ContributionScores(self.gaussians.get_xyz.shape[0], self.gaussians.get_xyz.device)
        for idx in (range(len(self)) if cam_indices is None else cam_indices):
            view, proj, campos = self.get_trajectory_tensors(idx)
            renderer.render_blurry(view, proj, campos, self.original_cam[0], self.gaussians, background,
                                   contrib=scores)
        return scores
