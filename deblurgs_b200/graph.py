"""One blurry-view training step as a CUDA graph.

The step -- sub-frame poses from the Bezier control points, the Gaussian activations, the batched render of all F
sub-frames, the fused photometric loss and the complete backward down to the Gaussian parameters and the control
points -- is ~60 kernel launches and a few hundred microseconds of Python.  Nothing in it needs the host once the
binning buffer is sized from a capacity instead of the device-side duplicate count (`dgs_blur_forward_hint` with
num_rendered = NULL), so the whole step is captured once and replayed with a single launch; the 24-byte status record
of the forward (duplicate count, overflow flag) rides back to pinned host memory as a memcpy node of the same graph
and is looked at after the caller's own synchronisation (reading the loss).  If the scene outgrew the capacity the
step is re-captured with a larger one and replayed: results are always complete.

Reference semantics: one iteration of train.py:121-163 for one image, without the optimizer step
(`CameraMotionModule.query` + `l1_loss` (+ lambda_t_smooth * batchwise_smoothness_loss) + `loss.backward()`); with
lambda_dssim > 0 the L1 term is the 3DGS mix (1 - lambda_dssim) * L1 + lambda_dssim * (1 - SSIM).
"""
import torch

from . import _lib
from . import rasterizer as rz
from .loss import mcmc_regularization, photometric_loss


class BlurryViewGraph:
    """Usage:
        step = BlurryViewGraph(cmm, cam_idx, background, gt_shape=(3, H, W))
        step.gt.copy_(ground_truth)            # any stream-ordered copy into the static input
        loss = step.replay()                   # 0-dim device tensor (static storage); .grad of every parameter is set
        ...optimizer.step()                    # .grad tensors are static storage owned by the graph (re-attached on replay)
        step.check()                           # after a synchronisation: re-captures + replays if the capacity was exceeded
    `parameters` (default: the Gaussians' and the trajectory's) get their .grad from the captured backward.
    The store's `antialiasing` flag is read when the step is captured and is part of the graph: a replay after the flag
    was changed raises DgsError (build a new BlurryViewGraph for the other setting) instead of rendering the old one.
    So is the 3-D filter (`filter_3D`): whether it is on and which tensor holds it are fixed at capture, and a replay
    after either changed raises.  Recomputing it in place (`CameraMotionModule.compute_3D_filter` on an unchanged
    store) is what a replay sees: the graph reads the tensor's current values.  The same holds for the in-place
    3DGS-MCMC moves (`relocate_gs`, `mcmc.add_sgld_noise`); `add_new_gs` changes P and needs a new graph.
    opacity_reg / scale_reg > 0 add loss.mcmc_regularization to the captured loss."""

    def __init__(self, cmm, cam_idx, background, gt_shape, lambda_t_smooth=0.0, parameters=None, pre_backward=None,
                 caller_owned_grads=(), capacity_margin=1.25, post_backward=None, render_fn=None,
                 lambda_dssim=0.0, opacity_reg=0.0, scale_reg=0.0):
        self.cmm, self.cam_idx, self.bg, self.lam = cmm, cam_idx, background, float(lambda_t_smooth)
        self.lam_dssim = float(lambda_dssim)      # > 0: the D-SSIM term of loss.photometric_loss inside the graph
        # 3DGS-MCMC's regularisers (loss.mcmc_regularization) inside the graph; both 0: not captured at all
        self.opacity_reg, self.scale_reg = float(opacity_reg), float(scale_reg)
        dev = cmm.gaussians.get_xyz.device
        self.device = dev
        self.params = list(parameters) if parameters is not None else cmm.gaussians.parameters() + cmm.parameters()
        # pre_backward: optional callable captured in front of the step (e.g. zeroing a flat gradient buffer whose views
        # are the .grad of `caller_owned_grads`: those accumulate in place; every other .grad is produced by the graph)
        self.pre_backward = pre_backward
        self.post_backward = post_backward        # captured behind the backward (e.g. a gradient sink's wait())
        # render_fn(graph) -> (blurred [3,H,W], subframes [F',3,H,W], batched package): replaces cmm.query, e.g. the
        # sub-frame-sharded render of dist.render_blurry_sharded (its NCCL all-reduce is captured with the rest)
        self.render_fn = render_fn
        self.collective = post_backward is not None or render_fn is not None    # may hold NCCL nodes: see check()
        self.owned = set(id(p) for p in caller_owned_grads)
        self.margin = float(capacity_margin)
        self.gt = torch.zeros(gt_shape, dtype=torch.float32, device=dev)
        self.status_host = torch.zeros(6, dtype=torch.int32).pin_memory()
        self.graph, self.loss, self.out, self.capacity = None, None, None, 0
        self.recaptures = 0
        self.antialiasing = self._store_antialiasing()
        self.filter_3D_ptr = self._store_filter_3D()
        self._capture(None)

    # ------------------------------------------------------------------------------------------
    def _run(self):
        if self.pre_backward is not None:
            self.pre_backward()
        if self.render_fn is not None:
            blurred, subframes, pkg = self.render_fn(self)
            out = {"blurred": blurred, "subframes": subframes, "batched": pkg}
        else:
            out = self.cmm.query(self.cam_idx, "all", background=self.bg)
        loss = photometric_loss(out["blurred"], out["subframes"], self.gt, self.lam, self.lam_dssim)
        if self.opacity_reg != 0.0 or self.scale_reg != 0.0:
            loss = loss + mcmc_regularization(self.cmm.gaussians, self.opacity_reg, self.scale_reg)
        loss.backward()
        if self.post_backward is not None:
            self.post_backward()
        return out, loss.detach()

    def _store_antialiasing(self):
        return bool(getattr(self.cmm.gaussians, "antialiasing", False))

    def _store_filter_3D(self):
        f = getattr(self.cmm.gaussians, "filter_3D", None)
        return None if f is None else f.data_ptr()

    def _reset_grads(self):
        for p in self.params:
            if id(p) not in self.owned:
                p.grad = None

    def _capture(self, capacity):
        lib = _lib.load()
        # (the parameters' AccumulateGrad nodes were created on the caller's stream, warm-up and capture run on side
        # streams: expected here, and everything is ordered by the stream waits / the capture itself)
        warn = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
        if warn is not None:
            warn(False)
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            # eager warm-up on a side stream (required before capture); in exact mode it also measures the scene
            self._reset_grads()
            out, _ = self._run()
            if capacity is None:
                pkg = out["batched"]
                F, P = pkg["radii"].shape
                H, W = pkg["render"].shape[2:]
                hint = rz._CAPACITY_HINT.get((self.device.index, P, F, H, W), 0)
                capacity = max(int(hint * self.margin / 1.25), 65536)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        self._reset_grads()
        self.capacity = int(capacity)
        launches0 = int(lib.dgs_launch_count(0))
        graph = torch.cuda.CUDAGraph()
        rz._ASYNC = {"capacity": self.capacity, "geoms": []}
        try:
            with torch.cuda.graph(graph):
                self.out, self.loss = self._run()
                geom, P, F = rz._ASYNC["geoms"][-1]
                off = int(lib.dgs_blur_forward_status_offset(P, F)) + (-geom.data_ptr()) % 128
                self.status_host.copy_(geom[off:off + 24].view(torch.int32), non_blocking=True)
        finally:
            rz._ASYNC = None
        self.launches_per_replay = int(lib.dgs_launch_count(0)) - launches0   # library kernels inside one replay
        self.grads = [p.grad for p in self.params]     # static storage the replays write into
        self.graph = graph

    # ------------------------------------------------------------------------------------------
    def replay(self):
        if self._store_antialiasing() != self.antialiasing:
            raise _lib.DgsError("the store's antialiasing flag changed since this step was captured (captured with "
                                "antialiasing=%s): build a new BlurryViewGraph for the new setting" % self.antialiasing)
        if self._store_filter_3D() != self.filter_3D_ptr:
            raise _lib.DgsError("the store's 3-D filter was %s since this step was captured: build a new BlurryViewGraph "
                                "(an in-place compute_3D_filter keeps the graph valid)"
                                % ("turned on" if self.filter_3D_ptr is None else
                                   "turned off" if self._store_filter_3D() is None else "replaced"))
        self.graph.replay()
        for p, g in zip(self.params, self.grads):      # re-attach if someone replaced or cleared a .grad meanwhile
            if p.grad is not g:
                p.grad = g
        return self.loss

    def num_rendered(self):
        """Duplicates of the last replay (valid after a synchronisation)."""
        s = self.status_host
        return (int(s[0]) & 0xFFFFFFFF) | ((int(s[1]) & 0xFFFFFFFF) << 32)

    def check(self):
        """Call after synchronising on the replay (e.g. after loss.item()).  False: all good.  True: the scene had
        outgrown the binning capacity; the step was re-captured with a larger one and replayed (synchronously), so
        loss / gradients are now complete."""
        over, need = int(self.status_host[4]) != 0, self.num_rendered()
        if self.collective:
            # the graph contains collectives: capture (and its eager warm-up) must happen on every rank or on none
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                t = torch.tensor([int(over), need if over else 0], dtype=torch.int64, device=self.device)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                over, need = bool(t[0].item()), max(need, int(t[1].item()))
        if not over:
            return False
        self._capture(int(need * self.margin) + 65536)
        self.recaptures += 1
        self.graph.replay()
        torch.cuda.synchronize(self.device)
        if int(self.status_host[4]) != 0:
            raise _lib.DgsError("binning capacity still exceeded after re-capture")
        return True

    def step(self, gt=None):
        """Convenience: copy gt in (if given), replay, synchronise, verify; returns the loss as a Python float."""
        if gt is not None:
            self.gt.copy_(gt, non_blocking=True)
        loss = self.replay()
        value = loss.item()
        if self.check():
            value = self.loss.item()
        return value
