"""Densify / prune mechanics of the Gaussian parameter store (SURVEY.md 8f rank 3, second half).

Mirrors GaussianModel.{replace_tensor_to_optimizer, _prune_optimizer, prune_points, cat_tensors_to_optimizer,
densification_postfix, densify_and_split, densify_and_clone, densify_and_prune, reset_opacity} of taekkii/deblurgs
(scene/gaussian_model.py:247-254, 300-454) on `GaussianParams` + `FusedAdam` (or any optimizer with torch's
`param_groups` / `state` layout): same selection rules, same new-Gaussian construction, same optimizer-state
surgery (moments masked / zero-extended, the per-tensor step count kept), 'curve_*' groups left alone.

Every one of these operations is "new row r of every per-Gaussian tensor = old row src[r], Adam moments of appended
rows zeroed".  On the GPU the whole store -- 6 parameter tensors, their 12 moment tensors, the 3 statistics vectors --
is rebuilt by ONE launch of the library's row-gather kernel (`dgs_rows_gather`, csrc/dgs_params.cu) from an index
plan; the reference runs ~40 torch index / cat launches for the same thing, and a split is a single rebuild here
instead of the reference's append followed by a prune.  The selection rules are a handful of P-sized torch ops.
With CPU tensors (unit tests of the semantics) the same plan is executed with torch indexing.  The per-step part --
accumulating the statistics these rounds consume -- is fused into the backward kernel (`DensificationStats`).
The WHEN (thresholds, schedules) remains the caller's policy, as in the reference's train.py:188-199.

The 3DGS-MCMC alternative (`relocate_gs`, `add_new_gs`; mcmc.py) reads no gradient statistics: dead Gaussians are
moved onto live ones drawn by opacity, in place (`dgs_mcmc_relocate`), and the store grows by a bounded fraction per
round up to a cap.
"""
import ctypes as C
import math

import torch
import torch.nn as nn

from . import _lib


def build_rotation(r):
    """Quaternions (r, x, y, z), not necessarily normalised, -> rotation matrices (utils/general_utils.py:117-138)."""
    q = r / torch.sqrt((r * r).sum(dim=1))[:, None]
    w, x, y, z = q.unbind(1)
    return torch.stack([
        torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], -1),
        torch.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], -1),
        torch.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], -1)], -2)


_GROUP_ATTR = {"xyz": "_xyz", "f_dc": "_features_dc", "f_rest": "_features_rest", "opacity": "_opacity",
               "scaling": "_scaling", "rotation": "_rotation"}


class DensificationMixin:
    """Needs: the six raw parameter attributes, `optimizer` (param_groups named as in training_setup),
    `get_scaling` / `get_opacity` / `get_xyz`, `scale_lower_bound`, and the statistics buffers; optionally `filter_3D`
    (Mip-Splatting's 3-D filter), which every rebuild carries along.  The selection rules read the unfiltered getters,
    as Mip-Splatting's do."""

    percent_dense = 0.01          # arguments/__init__.py:94
    alpha_lower_bound = 0.0       # arguments/__init__.py:68

    # ---- optimizer-state surgery -----------------------------------------------------------------
    def _swap_param(self, group, new_tensor, new_state_fn):
        old = group["params"][0]
        stored = self.optimizer.state.get(old, None)
        new = nn.Parameter(new_tensor.requires_grad_(True))
        if stored is not None:
            stored["exp_avg"] = new_state_fn(stored["exp_avg"])
            stored["exp_avg_sq"] = new_state_fn(stored["exp_avg_sq"])
            del self.optimizer.state[old]
            self.optimizer.state[new] = stored
        group["params"][0] = new
        return new

    def _assign(self, tensors):
        for name, attr in _GROUP_ATTR.items():
            if name in tensors:
                setattr(self, attr, tensors[name])

    def replace_tensor_to_optimizer(self, tensor, name):
        out = {}
        for group in self.optimizer.param_groups:
            if group["name"] == name:
                out[name] = self._swap_param(group, tensor, lambda m: torch.zeros_like(tensor))
        return out

    def _prune_optimizer(self, mask):
        out = {}
        for group in self.optimizer.param_groups:
            if "curve_" in group["name"]:
                continue
            out[group["name"]] = self._swap_param(group, group["params"][0].detach()[mask], lambda m: m[mask])
        return out

    def cat_tensors_to_optimizer(self, tensors_dict):
        out = {}
        for group in self.optimizer.param_groups:
            assert len(group["params"]) == 1
            if group["name"] not in tensors_dict:
                continue
            ext = tensors_dict[group["name"]]
            out[group["name"]] = self._swap_param(
                group, torch.cat((group["params"][0].detach(), ext), dim=0),
                lambda m, ext=ext: torch.cat((m, torch.zeros_like(ext)), dim=0))
        return out

    # ---- the whole store from an index plan ---------------------------------------------------------
    @torch.no_grad()
    def _rebuild(self, src, n_kept, keep_stats, xyz_new=None, scaling_new=None):
        """New store: row r of every per-Gaussian tensor = old row src[r].  Rows [0, n_kept) are surviving
        Gaussians (their Adam moments come along), rows [n_kept, len(src)) are appended ones (zero moments;
        `xyz_new` / `scaling_new` replace the gathered values there).  keep_stats: gather the densification
        statistics too (prune) instead of resetting them (append).  One kernel launch on the GPU."""
        self._ensure_stats()
        dev = self._xyz.device
        n_out = int(src.numel())
        groups = {g["name"]: g for g in self.optimizer.param_groups if g["name"] in _GROUP_ATTR}
        items = []      # (kind, name, old tensor, zero_new)
        for name, attr in _GROUP_ATTR.items():
            p = getattr(self, attr)
            items.append(("param", name, p.detach(), 0))
            st = self.optimizer.state.get(groups[name]["params"][0], None) if name in groups else None
            if st is not None and "exp_avg" in st:
                items.append(("exp_avg", name, st["exp_avg"], 1))
                items.append(("exp_avg_sq", name, st["exp_avg_sq"], 1))
        if keep_stats:
            items += [("stat", "xyz_gradient_accum", self.xyz_gradient_accum, 0), ("stat", "denom", self.denom, 0),
                      ("stat", "max_radii2D", self.max_radii2D.float(), 0)]
        filter_3D = getattr(self, "filter_3D", None)
        if filter_3D is not None:
            # Mip-Splatting's 3-D filter: appended (clone / split) rows inherit their parent's value
            items.append(("filter", "filter_3D", filter_3D, 0))
        outs = [torch.empty((n_out,) + tuple(t.shape[1:]), dtype=torch.float32, device=dev) for (_, _, t, _) in items]
        if dev.type == "cuda":
            lib = _lib.load()
            ins = [t.float().contiguous() for (_, _, t, _) in items]
            n = len(items)
            carry = None
            if n_kept < n_out:
                carry = torch.zeros(n_out, dtype=torch.uint8, device=dev)
                carry[:n_kept] = 1
            src_c = src.to(torch.int64).contiguous()
            with torch.cuda.device(dev):
                rc = lib.dgs_rows_gather(
                    n, (C.c_void_p * n)(*[t.data_ptr() for t in ins]), (C.c_void_p * n)(*[t.data_ptr() for t in outs]),
                    (C.c_int * n)(*[int(math.prod(t.shape[1:])) for t in ins]),
                    (C.c_int * n)(*[z for (_, _, _, z) in items]), n_out, _lib.ptr(src_c), _lib.ptr(carry),
                    C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
            _lib.check(rc, "dgs_rows_gather")
        else:   # CPU tensors: the same plan with torch indexing (semantics tests)
            for o, (_, _, t, zero_new) in zip(outs, items):
                o.copy_(t.float()[src])
                if zero_new:
                    o[n_kept:] = 0
        new = {}
        for o, (kind, name, _, _) in zip(outs, items):
            new[(kind, name)] = o
        if xyz_new is not None:
            new[("param", "xyz")][n_kept:] = xyz_new
        if scaling_new is not None:
            new[("param", "scaling")][n_kept:] = scaling_new
        tensors = {}
        for name, attr in _GROUP_ATTR.items():
            param = nn.Parameter(new[("param", name)].requires_grad_(True))
            if name in groups:
                g = groups[name]
                old = g["params"][0]
                st = self.optimizer.state.pop(old, None)
                if st is not None:
                    if ("exp_avg", name) in new:
                        st["exp_avg"], st["exp_avg_sq"] = new[("exp_avg", name)], new[("exp_avg_sq", name)]
                    self.optimizer.state[param] = st
                g["params"][0] = param
            tensors[name] = param
        self._assign(tensors)
        if filter_3D is not None:
            self.filter_3D = new[("filter", "filter_3D")]
        if keep_stats:
            self.xyz_gradient_accum = new[("stat", "xyz_gradient_accum")]
            self.denom = new[("stat", "denom")]
            self.max_radii2D = new[("stat", "max_radii2D")]
        else:
            self.xyz_gradient_accum = torch.zeros((n_out, 1), device=dev)
            self.denom = torch.zeros((n_out, 1), device=dev)
            self.max_radii2D = torch.zeros(n_out, device=dev)

    # ---- store-level operations ------------------------------------------------------------------
    @torch.no_grad()
    def prune_points(self, mask):
        """Remove the Gaussians where `mask` is True; parameters, Adam moments and statistics are compacted."""
        src = torch.nonzero(~mask).squeeze(1)
        self._rebuild(src, int(src.numel()), keep_stats=True)

    @torch.no_grad()
    def prune_by_contribution(self, scores, fraction=0.0, min_weight_max=0.0):
        """Contribution-based pruning (LightGaussian's global significance, RadSplat's max weight): remove the
        `fraction` of Gaussians with the lowest weight sum -- ties broken by index, lower first -- plus every
        Gaussian whose largest blending weight is below `min_weight_max`.  `scores`: a `rasterizer.ContributionScores`
        of this store (e.g. `CameraMotionModule.accumulate_contribution`).  One `prune_points` rebuild; returns the
        boolean mask of the removed Gaussians."""
        P = self._xyz.shape[0]
        if scores.num_points != P:
            raise ValueError("contribution scores hold %d Gaussians, the store %d" % (scores.num_points, P))
        if not 0.0 <= fraction <= 1.0:
            raise ValueError("fraction must be in [0, 1]")
        dev = self._xyz.device
        wsum = scores.wsum.to(dev)
        mask = scores.weight_max.to(dev) < min_weight_max
        n = int(math.floor(fraction * P))
        if n > 0:
            # stable sort of the exact integer sums: equal scores keep index order
            order = torch.sort(wsum, stable=True).indices
            mask[order[:n]] = True
        self.prune_points(mask)
        return mask

    @torch.no_grad()
    def densification_postfix(self, new_xyz, new_features_dc, new_features_rest, new_opacities, new_scaling,
                              new_rotation):
        """Append new Gaussians (zero Adam moments) and reset the densification statistics.  With the 3-D filter on,
        the new Gaussians get a zero filter (unfiltered) until the next `CameraMotionModule.compute_3D_filter`."""
        self._assign(self.cat_tensors_to_optimizer({"xyz": new_xyz, "f_dc": new_features_dc,
                                                    "f_rest": new_features_rest, "opacity": new_opacities,
                                                    "scaling": new_scaling, "rotation": new_rotation}))
        P, dev = self._xyz.shape[0], self._xyz.device
        filter_3D = getattr(self, "filter_3D", None)
        if filter_3D is not None:
            self.filter_3D = torch.cat((filter_3D, filter_3D.new_zeros((P - filter_3D.shape[0], 1))), dim=0)
        self.xyz_gradient_accum = torch.zeros((P, 1), device=dev)
        self.denom = torch.zeros((P, 1), device=dev)
        self.max_radii2D = torch.zeros(P, device=dev)

    def _scaling_inverse(self, s):
        # LowerBoundLog (scene/gaussian_activation.py:54-64)
        return torch.log((s - self.scale_lower_bound).clamp_min(0.001))

    @torch.no_grad()
    def densify_and_split(self, grads, grad_threshold, scene_extent, N=2, generator=None):
        """Large Gaussians with a large view-space gradient are replaced by N samples of themselves, scaled down
        by 0.8 N (scene/gaussian_model.py:396-420)."""
        P, dev = self._xyz.shape[0], self._xyz.device
        padded = torch.zeros(P, device=dev)
        padded[:grads.shape[0]] = grads.squeeze()
        scaling = self.get_scaling
        sel = (padded >= grad_threshold) & (scaling.max(dim=1).values > self.percent_dense * scene_extent)
        stds = scaling[sel].repeat(N, 1)
        samples = torch.normal(mean=torch.zeros_like(stds), std=stds, generator=generator)
        rots = build_rotation(self._rotation[sel]).repeat(N, 1, 1)
        new_xyz = torch.bmm(rots, samples.unsqueeze(-1)).squeeze(-1) + self._xyz[sel].repeat(N, 1)
        new_scaling = self._scaling_inverse(scaling[sel].repeat(N, 1) / (0.8 * N))
        # reference: append the N copies (densification_postfix), then prune the originals (prune_points): the
        # surviving rows keep their order and moments, the copies follow with zero moments -- one rebuild
        kept, sel_idx = torch.nonzero(~sel).squeeze(1), torch.nonzero(sel).squeeze(1)
        self._rebuild(torch.cat((kept, sel_idx.repeat(N))), int(kept.numel()), keep_stats=False,
                      xyz_new=new_xyz, scaling_new=new_scaling)

    @torch.no_grad()
    def densify_and_clone(self, grads, grad_threshold, scene_extent):
        """Small Gaussians with a large view-space gradient are duplicated in place (scene/gaussian_model.py:422-436)."""
        sel = (torch.norm(grads, dim=-1) >= grad_threshold) & \
              (self.get_scaling.max(dim=1).values <= self.percent_dense * scene_extent)
        P = self._xyz.shape[0]
        self._rebuild(torch.cat((torch.arange(P, device=self._xyz.device), torch.nonzero(sel).squeeze(1))), P,
                      keep_stats=False)

    @torch.no_grad()
    def densify_and_prune(self, max_grad, extent, generator=None):
        """One densification round from the accumulated statistics (scene/gaussian_model.py:438-449)."""
        self._ensure_stats()
        grads = self.xyz_gradient_accum / self.denom
        grads[grads.isnan()] = 0.0
        self.densify_and_clone(grads, max_grad, extent)
        self.densify_and_split(grads, max_grad, extent, generator=generator)
        min_opacity = self.alpha_lower_bound + (1 - self.alpha_lower_bound) * 0.005
        self.prune_points((self.get_opacity < min_opacity).squeeze(-1))

    # ---- 3DGS-MCMC (Kheradmand et al., NeurIPS 2024): relocation and growth --------------------------------------
    @torch.no_grad()
    def _relocate(self, dst, src):
        """In place: row dst[r] of every per-Gaussian tensor becomes a copy of row src[r]; the opacity and scale of
        every source are split between it and its copies (mcmc.relocation_values); the Adam moments and the
        densification statistics of the source and destination rows are zeroed.  Every tensor keeps its identity and
        storage.  Precondition: dst rows distinct and disjoint from the src rows.  One `dgs_mcmc_relocate` on the GPU."""
        from . import mcmc
        self._ensure_stats()
        P, dev = self._xyz.shape[0], self._xyz.device
        ratio = mcmc.relocation_ratio(src, P)
        groups = {g["name"]: g for g in self.optimizer.param_groups if g["name"] in _GROUP_ATTR}
        kind_of = {"opacity": 1, "scaling": 2}      # DGS_RELOCATE_OPACITY / _SCALING; parameters otherwise copied (0)
        items = []                                   # (tensor, kind)
        for name, attr in _GROUP_ATTR.items():
            items.append((getattr(self, attr).detach(), kind_of.get(name, 0)))
            st = self.optimizer.state.get(groups[name]["params"][0], None) if name in groups else None
            if st is not None and "exp_avg" in st:
                items += [(st["exp_avg"], 3), (st["exp_avg_sq"], 3)]
        items += [(self.xyz_gradient_accum, 3), (self.denom, 3), (self.max_radii2D, 3)]
        if getattr(self, "filter_3D", None) is not None:
            items.append((self.filter_3D, 0))
        if dev.type == "cuda":
            for t, _ in items:
                if t.dtype != torch.float32 or not t.is_contiguous() or t.device != dev or t.shape[0] != P:
                    raise _lib.DgsError("relocation rewrites the store in place: every per-Gaussian tensor must be a "
                                        "contiguous float32 [P, ...] tensor on %s" % dev)
            lib = _lib.load()
            n, nt = int(dst.numel()), len(items)
            dst_c, src_c = dst.to(torch.int64).contiguous(), src.to(torch.int64).contiguous()
            scratch = torch.empty(int(lib.dgs_mcmc_relocate_scratch_bytes(n)), dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                rc = lib.dgs_mcmc_relocate(
                    nt, (C.c_void_p * nt)(*[t.data_ptr() for t, _ in items]),
                    (C.c_int * nt)(*[int(math.prod(t.shape[1:])) for t, _ in items]),
                    (C.c_int * nt)(*[k for _, k in items]), n, _lib.ptr(dst_c), _lib.ptr(src_c), _lib.ptr(ratio),
                    float(self.scale_lower_bound), int(bool(self.use_isotropic)), _lib.ptr(scratch),
                    C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
            _lib.check(rc, "dgs_mcmc_relocate")
        else:   # CPU tensors: the same plan with torch indexing, the values from the fp64 statement
            op, sc, _, _ = mcmc.relocation_values(self._opacity.detach()[src], self._scaling.detach()[src], ratio,
                                                  self.scale_lower_bound, self.use_isotropic)
            for t, kind in items:
                if kind == 0:
                    t[dst] = t[src]
                else:
                    v = op if kind == 1 else sc if kind == 2 else 0.0
                    t[dst] = v
                    t[src] = v

    @torch.no_grad()
    def relocate_gs(self, dead_mask=None, min_opacity=0.005, generator=None):
        """3DGS-MCMC relocation: every dead Gaussian (default: get_opacity <= min_opacity, the unfiltered getter) is
        replaced, in place, by a copy of a live one drawn with probability proportional to its opacity
        (mcmc.sample_by_opacity); the opacity and scale of each drawn source are split between it and its copies so
        that the rendered image stays the same to first order.  Parameters, optimizer state, `filter_3D` and the
        statistics keep their identity (a captured graph.BlurryViewGraph stays valid); the moments and statistics of
        the touched rows are zeroed; step counts are kept.  Returns the number of rows relocated (0, doing nothing,
        when no row is dead or none is live)."""
        from . import mcmc
        opac = self.get_opacity.detach().reshape(-1)
        dead = (opac <= min_opacity) if dead_mask is None else dead_mask.reshape(-1).to(device=opac.device,
                                                                                      dtype=torch.bool)
        n_dead = int(dead.sum())
        weights = torch.where(dead, torch.zeros_like(opac), opac)
        if n_dead == 0 or float(torch.floor(weights.double().clamp(0.0, 1.0) * 2.0 ** 24).max()) <= 0.0:
            return 0
        dst = torch.nonzero(dead).squeeze(1)
        src = mcmc.sample_by_opacity(weights, n_dead, generator)
        self._relocate(dst, src)
        return n_dead

    @torch.no_grad()
    def add_new_gs(self, cap_max, growth=0.05, generator=None):
        """3DGS-MCMC growth: append min(cap_max, floor((1 + growth) P)) - P Gaussians, copies of rows drawn by opacity,
        with the same opacity / scale split as `relocate_gs` (one `_rebuild` that appends the copies, then one
        relocation whose destinations are the appended rows).  P changes: a captured graph must be rebuilt, as after
        densify_and_prune.  Returns the number of rows added."""
        from . import mcmc
        P = self._xyz.shape[0]
        n_new = mcmc.growth_target(P, cap_max, growth)
        if n_new == 0:
            return 0
        src = mcmc.sample_by_opacity(self.get_opacity.detach(), n_new, generator)
        self._rebuild(torch.cat((torch.arange(P, device=src.device), src)), P, keep_stats=True)
        self._relocate(torch.arange(P, P + n_new, device=src.device), src)
        return n_new

    @torch.no_grad()
    def reset_opacity(self, new_opacity=None):
        """Cap every opacity at `new_opacity` (default 0.1) and zero its Adam moments (scene/gaussian_model.py:247-254).
        With the 3-D filter on, the cap applies to the filtered opacity, as in Mip-Splatting's reset_opacity: the new
        clamped opacity is min(o, cap / prod_i r_i), so that the filtered one is min(o prod_i r_i, cap)."""
        if new_opacity is None:
            lb = self.alpha_lower_bound
            new_opacity = lb + (1 - lb) * 0.1
        opac = self.get_opacity
        if getattr(self, "filter_3D", None) is not None:
            r = self._filter_3D_ratios()
            capped = torch.min(opac, new_opacity / (r[:, 0:1] * r[:, 1:2] * r[:, 2:3])).clamp(0.0, 1.0)
        else:
            capped = torch.min(opac, torch.ones_like(opac) * new_opacity).clamp(0.0, 1.0)
        self._assign(self.replace_tensor_to_optimizer(capped, "opacity"))
