"""Gaussian parameter store: fused activations and the fused Adam step (SURVEY.md 8f rank 3).

Mirrors, for the hot path only:
  GaussianModel.get_scaling / get_rotation / get_opacity / get_features
                                scene/gaussian_model.py:114-137, scene/gaussian_activation.py:29-52
  GaussianModel.training_setup  scene/gaussian_model.py:175-190   (torch.optim.Adam, eps=1e-15, one
                                parameter per group, per-group learning rates)
  train.py:204-208              clip_grad_value_ -> optimizer.step() -> zero_grad(set_to_none=True)
Both are single launches of libdgs_b200.so (`dgs_activate_forward/backward`, `dgs_adam_step`); there is
no torch fallback.
"""
import ctypes as C

import torch

from . import _lib


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


class _ActivateGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, features_dc, features_rest, scaling, rotation, opacity, scale_lower_bound, isotropic,
                filter3d=None):
        lib = _lib.load()
        if not scaling.is_cuda:
            raise _lib.DgsError("Gaussian parameters must be CUDA tensors: libdgs_b200 has no CPU path")
        dc, rest = features_dc.detach().float().contiguous(), features_rest.detach().float().contiguous()
        sc, rot, op = (t.detach().float().contiguous() for t in (scaling, rotation, opacity))
        P = sc.shape[0]
        M = 1 + (rest.shape[1] if rest.dim() == 3 else 0)
        dev = sc.device
        shs = torch.empty((P, M, 3), dtype=torch.float32, device=dev)
        scales = torch.empty((P, 3), dtype=torch.float32, device=dev)
        rots = torch.empty((P, 4), dtype=torch.float32, device=dev)
        opac = torch.empty((P, 1), dtype=torch.float32, device=dev)
        filt = None if filter3d is None else filter3d.detach().float().contiguous()
        if filt is not None and filt.numel() != P:
            raise _lib.DgsError("filter_3D holds %d values, the store %d Gaussians" % (filt.numel(), P))
        with torch.cuda.device(dev):
            if filt is None:
                rc = lib.dgs_activate_forward(P, M, _lib.ptr(dc), _lib.ptr(rest), _lib.ptr(sc), _lib.ptr(rot),
                                              _lib.ptr(op), float(scale_lower_bound), int(bool(isotropic)),
                                              _lib.ptr(shs), _lib.ptr(scales), _lib.ptr(rots), _lib.ptr(opac),
                                              _stream(dev))
            else:
                rc = lib.dgs_activate_forward_filter3d(P, M, _lib.ptr(dc), _lib.ptr(rest), _lib.ptr(sc), _lib.ptr(rot),
                                                       _lib.ptr(op), float(scale_lower_bound), int(bool(isotropic)),
                                                       _lib.ptr(shs), _lib.ptr(scales), _lib.ptr(rots), _lib.ptr(opac),
                                                       filt.data_ptr(), _stream(dev))
        _lib.check(rc, "dgs_activate_forward")
        ctx.save_for_backward(sc, rot, op)
        ctx.filter3d = filt
        ctx.meta = (P, M, bool(isotropic), features_dc.shape, features_rest.shape, float(scale_lower_bound))
        return shs, scales, rots, opac

    @staticmethod
    def backward(ctx, dshs, dscales, drots, dopac):
        lib = _lib.load()
        sc, rot, op = ctx.saved_tensors
        P, M, isotropic, dc_shape, rest_shape, lb = ctx.meta
        dev = sc.device
        f = lambda t: None if t is None else t.float().contiguous()
        dshs, dscales, drots, dopac = f(dshs), f(dscales), f(drots), f(dopac)
        ddc = torch.empty(dc_shape, dtype=torch.float32, device=dev)
        drest = torch.empty(rest_shape, dtype=torch.float32, device=dev)
        dsc, drot, dop = torch.empty_like(sc), torch.empty_like(rot), torch.empty_like(op)
        args = (P, M, _lib.ptr(sc), _lib.ptr(rot), _lib.ptr(op), int(isotropic), _lib.ptr(dshs), _lib.ptr(dscales),
                _lib.ptr(drots), _lib.ptr(dopac), _lib.ptr(ddc), _lib.ptr(drest), _lib.ptr(dsc), _lib.ptr(drot),
                _lib.ptr(dop))
        with torch.cuda.device(dev):
            if ctx.filter3d is None:
                rc = lib.dgs_activate_backward(*args, _stream(dev))
            else:
                rc = lib.dgs_activate_backward_filter3d(*args, lb, ctx.filter3d.data_ptr(), _stream(dev))
        _lib.check(rc, "dgs_activate_backward")
        return ddc, drest, dsc, drot, dop, None, None, None


def activate_gaussians(features_dc, features_rest, scaling, rotation, opacity, scale_lower_bound=0.0,
                       isotropic=False, filter3d=None):
    """(get_features [P,M,3], get_scaling [P,3], get_rotation [P,4], get_opacity [P,1]) of the reference's
    GaussianModel in one launch, differentiable with respect to the five raw parameter tensors.
    `filter3d` [P,1]: Mip-Splatting's 3-D smoothing filter (a constant without gradient); scales and opacities are
    then those of get_scaling_with_3D_filter / get_opacity_with_3D_filter (include/dgs_b200.h)."""
    return _ActivateGaussians.apply(features_dc, features_rest, scaling, rotation, opacity, scale_lower_bound,
                                    isotropic, filter3d)


class FusedAdam:
    """`torch.optim.Adam(groups, lr=..., eps=...)` for float32 CUDA parameters, every parameter tensor of
    every group updated by ONE kernel launch per step.  Keeps torch's surface where the reference touches
    it: `param_groups` (list of dicts with 'params', 'lr', 'name', ...), `state[p]` with 'step', 'exp_avg',
    'exp_avg_sq', `step()`, `zero_grad(set_to_none=True)`, `state_dict()` / `load_state_dict()`.
    amsgrad, weight decay and maximize are not provided (the reference does not use them)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        params = list(params)
        if params and not isinstance(params[0], dict):
            params = [{"params": params}]
        self.defaults = {"lr": lr, "betas": tuple(betas), "eps": eps}
        self.param_groups = []
        for g in params:
            g = dict(g)
            g["params"] = list(g["params"])
            for k, v in self.defaults.items():
                g.setdefault(k, v)
            self.param_groups.append(g)
        self.state = {}

    def add_param_group(self, group):
        g = dict(group)
        g["params"] = list(g["params"])
        for k, v in self.defaults.items():
            g.setdefault(k, v)
        self.param_groups.append(g)

    def zero_grad(self, set_to_none=True):
        for g in self.param_groups:
            for p in g["params"]:
                if p.grad is not None:
                    if set_to_none:
                        p.grad = None
                    else:
                        p.grad.zero_()

    @torch.no_grad()
    def step(self, clip_grad_value=None):
        """One Adam update of every parameter that has a gradient. `clip_grad_value` folds
        torch.nn.utils.clip_grad_value_ (train.py:204-205) into the same pass."""
        lib = _lib.load()
        batches = {}   # (device, betas, eps) -> list of (p, grad, state, lr)
        for g in self.param_groups:
            for p in g["params"]:
                if p.grad is None:
                    continue
                if not p.is_cuda or p.dtype != torch.float32:
                    raise _lib.DgsError("FusedAdam updates float32 CUDA parameters only: libdgs_b200 has no CPU path")
                if not p.is_contiguous():
                    raise _lib.DgsError("FusedAdam needs contiguous parameters")
                st = self.state.get(p)
                if st is None or len(st) == 0:
                    st = self.state[p] = {"step": 0, "exp_avg": torch.zeros_like(p),
                                          "exp_avg_sq": torch.zeros_like(p)}
                st["step"] = int(st["step"]) + 1
                grad = p.grad if (p.grad.is_contiguous() and p.grad.dtype == torch.float32) \
                    else p.grad.float().contiguous()
                key = (p.device, tuple(g["betas"]), float(g["eps"]))
                batches.setdefault(key, []).append((p, grad, st, float(g["lr"])))
        n_max = 8   # DGS_ADAM_MAX_TENSORS
        for (dev, betas, eps), items in batches.items():
            for i0 in range(0, len(items), n_max):
                chunk = items[i0:i0 + n_max]
                n = len(chunk)
                arr_p = (C.c_void_p * n)(*[it[0].data_ptr() for it in chunk])
                arr_g = (C.c_void_p * n)(*[it[1].data_ptr() for it in chunk])
                arr_m = (C.c_void_p * n)(*[it[2]["exp_avg"].data_ptr() for it in chunk])
                arr_v = (C.c_void_p * n)(*[it[2]["exp_avg_sq"].data_ptr() for it in chunk])
                arr_n = (C.c_int64 * n)(*[it[0].numel() for it in chunk])
                arr_lr = (C.c_double * n)(*[it[3] for it in chunk])
                arr_t = (C.c_int64 * n)(*[it[2]["step"] for it in chunk])
                with torch.cuda.device(dev):
                    rc = lib.dgs_adam_step(n, arr_p, arr_g, arr_m, arr_v, arr_n, arr_lr, arr_t, float(betas[0]),
                                           float(betas[1]), eps, float(clip_grad_value or 0.0), _stream(dev))
                _lib.check(rc, "dgs_adam_step")

    def state_dict(self):
        """Same layout as torch.optim.Optimizer.state_dict() (indices in param_groups, state by index)."""
        index, groups = {}, []
        for g in self.param_groups:
            ids = []
            for p in g["params"]:
                index.setdefault(id(p), len(index))
                ids.append(index[id(p)])
            groups.append({**{k: v for k, v in g.items() if k != "params"}, "params": ids})
        state = {}
        for p, st in self.state.items():
            if id(p) in index:
                state[index[id(p)]] = {"step": torch.tensor(float(st["step"])), "exp_avg": st["exp_avg"],
                                       "exp_avg_sq": st["exp_avg_sq"]}
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, sd):
        flat = [p for g in self.param_groups for p in g["params"]]
        for g, sg in zip(self.param_groups, sd["param_groups"]):
            for k, v in sg.items():
                if k != "params":
                    g[k] = v
        self.state = {}
        for i, st in sd["state"].items():
            p = flat[int(i)]
            self.state[p] = {"step": int(float(st["step"])), "exp_avg": st["exp_avg"].to(p.device).float().clone(),
                             "exp_avg_sq": st["exp_avg_sq"].to(p.device).float().clone()}
