"""Multi-GPU plumbing for the blurry-view path: one process per GPU, torch.distributed (NCCL over
NVLink/NVSwitch on the GPU box; gloo in the CPU tests).

The reference is single-GPU (SURVEY.md 5.8); the path shards along its two independent axes:
  * views of a batch   -> each rank renders whole blurry views; the Gaussian gradients are summed with
                          one all-reduce of a flat buffer (`FlatGradBuffer`) -- weak scaling;
  * sub-frames of a view -> each rank renders a contiguous block of the F sub-frames
                          (`subframe_shard`), the partial blurry images are summed (`all_reduce_sum`,
                          identity backward) and the gradients all-reduced as above -- strong scaling.
No collective sits inside the rasterizer itself.
"""
import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


_DIRECT = {}      # device index -> nccl_direct.DirectComm (or None once creation failed)


def direct_comm(device):
    """The process's direct NCCL communicator for the hot-path collectives (see nccl_direct.py), or None when the
    default group is not NCCL on a CUDA device (gloo CPU tests, single process).  Created on first use -- a collective
    call: every rank must reach it, and not from inside a stream capture."""
    device = torch.device(device)
    if device.type != "cuda" or not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() < 2:
        return None
    if dist.get_backend() != "nccl":
        return None
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _DIRECT:
        from .nccl_direct import DirectComm
        _DIRECT[key] = DirectComm(torch.device("cuda", key))
    return _DIRECT[key]


def subframe_shard(num_subframes, rank, world_size):
    """Contiguous block [start, stop) of sub-frames for `rank`; blocks differ by at most one sub-frame
    and keep temporal neighbours on the same rank (except at block edges)."""
    base, rem = divmod(num_subframes, world_size)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


class _AllReduceSum(torch.autograd.Function):
    """y = sum over ranks of x. Every rank then evaluates the SAME loss on y, so dL/dx_r = dL/dy: the
    backward is the identity (the per-rank parameter gradients are summed later by FlatGradBuffer)."""

    @staticmethod
    def forward(ctx, x):
        y = x.contiguous().clone()
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            comm = direct_comm(y.device) if y.dtype == torch.float32 else None
            if comm is not None:
                comm.all_reduce_(y)                 # on the current stream: capturable
            else:
                dist.all_reduce(y, op=dist.ReduceOp.SUM)
        return y

    @staticmethod
    def backward(ctx, g):
        return g


def all_reduce_sum(x):
    return _AllReduceSum.apply(x)


class FlatGradBuffer:
    """One flat fp32 gradient buffer; each parameter's .grad is a view into it.

    Plain use: `zero()`, backward (autograd accumulates into the views), `all_reduce()` -- one collective.
    As a gradient SINK of the Gaussian store (`for_gaussians`, handed to `render_blurry(..., grad_sink=)` or set as
    `gaussians.grad_sink`): the backward writes finished rows straight into the views and calls `rows_done(g0, g1)`,
    which starts the all-reduce of those rows of the largest tensor (the SH rest coefficients, 3/4 of all bytes) on
    NCCL's own stream while the next range of Gaussians is still being computed; `finish()` reduces the five small
    tensors (contiguous in the buffer) in one call; `wait()` makes the current stream wait for all of it."""

    def __init__(self, params, names=None):
        self.params = [p for p in params]
        n = sum(p.numel() for p in self.params)
        self.flat = torch.zeros(n, dtype=torch.float32, device=self.params[0].device)
        self.views, self.spans = {}, {}
        off = 0
        for i, p in enumerate(self.params):
            p.grad = self.flat[off:off + p.numel()].view_as(p)
            key = names[i] if names is not None else i
            self.views[key] = p.grad
            self.spans[key] = (off, off + p.numel())
            off += p.numel()
        self.works, self.big, self.small_span = [], None, None
        # NCCL on a CUDA device: the collectives are issued directly on a side stream (fork / join with events), which
        # also works inside a stream capture; otherwise through torch.distributed (gloo in the CPU tests)
        self.comm = direct_comm(self.flat.device)
        self.comm_stream = torch.cuda.Stream(self.flat.device) if self.comm is not None else None
        self._forked = False
        self.n_ranges = 4          # row ranges the backward finishes one after the other (each followed by its all-reduce)

    @classmethod
    def for_gaussians(cls, g):
        """Sink layout for a `GaussianParams` store: the five small tensors first (one contiguous block), the SH rest
        coefficients last."""
        names = ["xyz", "f_dc", "scaling", "rotation", "opacity", "f_rest"]
        params = [g._xyz, g._features_dc, g._scaling, g._rotation, g._opacity, g._features_rest]
        self = cls(params, names)
        self.big = "f_rest"
        self.small_span = (0, self.spans["f_rest"][0])
        return self

    def zero(self):
        self.flat.zero_()

    def _active(self):
        return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1

    def all_reduce(self):
        if self._active():
            if self.comm is not None:
                self.comm.all_reduce_(self.flat)
            else:
                dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
        return self.flat

    # ---- sink protocol (called from the backward of rasterizer._RenderStoreBlurry) --------------------
    def begin(self):
        self.works = []

    def _async_all_reduce(self, t):
        if self.comm is not None:
            # fork: the side stream picks up behind everything enqueued so far; the caller's stream goes on
            self.comm_stream.wait_stream(torch.cuda.current_stream(self.flat.device))
            self.comm.all_reduce_(t, stream=self.comm_stream)
            self._forked = True
        else:
            self.works.append(dist.all_reduce(t, op=dist.ReduceOp.SUM, async_op=True))

    def rows_done(self, g0, g1):
        """Rows [g0, g1) of every Gaussian gradient are final: reduce them now (asynchronously: the collective runs on a
        side stream behind everything enqueued so far, the caller's stream goes on).  Direct NCCL: the rows of all six
        tensors as one grouped launch; torch.distributed: the big tensor's rows (the small tensors follow in finish())."""
        if not (self._active() and self.big is not None and g1 > g0):
            return
        if self.comm is not None:
            self.comm_stream.wait_stream(torch.cuda.current_stream(self.flat.device))     # fork
            self.comm.all_reduce_group_([v[g0:g1] for v in self.views.values()], stream=self.comm_stream)
            self._forked = True
        else:
            self._async_all_reduce(self.views[self.big][g0:g1])

    def finish(self):
        if self._active() and self.small_span is not None and self.comm is None:
            a, b = self.small_span
            self._async_all_reduce(self.flat[a:b])

    def wait(self):
        """The current stream waits for every collective started since begin()."""
        if self._forked:
            torch.cuda.current_stream(self.flat.device).wait_stream(self.comm_stream)     # join
            self._forked = False
        for w in self.works:
            w.wait()
        self.works = []


@torch.no_grad()
def all_reduce_densification_stats(stats):
    """Make the densification statistics of a step identical on every rank, so that the replicated Gaussian stores
    densify / prune identically.  Works for both shardings: ranks holding different sub-frames of one view, or
    different views of a batch -- the reference accumulates sums over whatever it rendered (train.py:188-193:
    gradient norms and visible fractions add up, radii take the maximum), so: SUM, SUM, MAX.
    `stats` = rasterizer.DensificationStats (filled by the backward pass); modified in place and returned."""
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return stats
    if not stats.ready:
        raise RuntimeError("densification statistics are produced by the backward pass: call loss.backward() first")
    sums = torch.cat((stats.grad_norm_sum.reshape(-1), stats.visible_count.reshape(-1)))
    dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    P = stats.grad_norm_sum.shape[0]
    stats.grad_norm_sum = sums[:P].reshape(P, 1)
    stats.visible_count = sums[P:].reshape(P, 1)
    radius = stats.max_radius.clone()
    dist.all_reduce(radius, op=dist.ReduceOp.MAX)
    stats.max_radius = radius
    return stats


@torch.no_grad()
def all_reduce_contribution(scores):
    """Make contribution scores identical on every rank, so that replicated Gaussian stores prune identically: with
    `render_blurry_sharded` (or views split across ranks) each rank scores only what it rendered.  Weight sums add up,
    maxima take the maximum (SUM on the int64 fixed-point sums, MAX on the float bits): exact, so the result equals
    the scores of one process that rendered everything.  `scores`: rasterizer.ContributionScores, modified in place
    and returned."""
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return scores
    dist.all_reduce(scores.wsum, op=dist.ReduceOp.SUM)
    dist.all_reduce(scores.wmax, op=dist.ReduceOp.MAX)
    return scores


def render_blurry_sharded(cmm, cam_idx, background, nu=None, grad_sink=None, contrib=None):
    """Sub-frame-sharded blurry view: this rank renders its block of the F sub-frames of image
    `cam_idx`; returns (blurred [3,H,W] identical on every rank, local package, (start, stop)).
    Densification: the local package's statistics cover this rank's sub-frames only (already normalised by the
    view's full sub-frame count); call `all_reduce_densification_stats(pkg["densification"])` after backward and
    before `add_densification_stats_blurry(pkg)` so that every rank accumulates the whole view.  Likewise `contrib`
    (rasterizer.ContributionScores) receives this rank's sub-frames only: `all_reduce_contribution` completes it."""
    from . import renderer
    rank, ws = world()
    view, proj, campos = cmm.get_trajectory_tensors(cam_idx, nu)
    F = view.shape[0]
    a, b = subframe_shard(F, rank, ws)
    pkg = renderer.render_blurry(view[a:b].contiguous(), proj[a:b].contiguous(), campos[a:b].contiguous(),
                                 cmm.original_cam[0], cmm.gaussians, background, blur_denominator=float(F),
                                 grad_sink=grad_sink, contrib=contrib)
    return all_reduce_sum(pkg["blurred"]), pkg, (a, b)
