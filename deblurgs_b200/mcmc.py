"""3DGS-MCMC densification (Kheradmand et al., NeurIPS 2024; gsplat's `MCMCStrategy`): the pieces outside the store.

`DensificationMixin.relocate_gs` / `add_new_gs` (densify.py) move low-opacity Gaussians onto live ones and grow the
store towards a fixed cap; this module holds what they and the training loop share:
  sample_by_opacity     live rows drawn with probability proportional to their opacity, from an exact integer CDF
  relocation_values     the relocation formula as an fp64 torch statement (the CPU path, and the tests' reference)
  add_sgld_noise        the per-step SGLD position noise, one launch of `dgs_mcmc_noise` (csrc/dgs_mcmc.cu)
The loss-side regularisers are `loss.mcmc_regularization`.  When to relocate and what cap to use is the caller's
policy.  Identically seeded generators give identical draws on every rank that holds an identical store, so
replicated stores stay identical without a broadcast of the sampled rows.
"""
import ctypes as C
import math

import torch

from . import _lib

N_MAX = 51                     # copies per source the relocation formula is evaluated for (larger ratios are clamped)
MIN_OPACITY = 0.005            # the relocated opacity's lower bound, and the default dead threshold
MAX_OPACITY = 1.0 - 2.0 ** -23
# the relocated opacity's stored lower bound: the smallest float32 above 0.005 (the nearest one lies below it, and a
# relocated Gaussian must not count as dead by the `get_opacity <= 0.005` rule)
MIN_OPACITY_F32 = 0.005000000353902578
NOISE_K, NOISE_X0 = 100.0, 0.995   # gate(o) = 1 / (1 + exp(-k ((1 - o) - x0))): only near-transparent Gaussians move


def sample_by_opacity(opacity, n, generator=None):
    """`n` row indices drawn with replacement, row i with probability w_i / sum(w), w_i = floor(clamp(o_i, 0, 1) 2^24)
    (int64).  The CDF is an exact integer cumsum and the draws are `torch.randint` + `torch.searchsorted(right=True)`:
    a weight-0 row (pass 0 for dead rows) is never drawn, the result is a pure function of the generator's state, and
    there is no 2^24-category limit as with `torch.multinomial`.  The draws are made on the generator's device (the
    opacities' without one) and returned on the opacities' device."""
    o = opacity.detach().reshape(-1)
    w = torch.floor(o.double().clamp(0.0, 1.0) * 2.0 ** 24).to(torch.int64)
    cdf = torch.cumsum(w, 0)
    total = int(cdf[-1]) if cdf.numel() else 0
    if total <= 0:
        raise ValueError("sample_by_opacity: no row has a positive weight")
    dev = generator.device if generator is not None else o.device
    u = torch.randint(0, total, (int(n),), generator=generator, device=dev, dtype=torch.int64)
    return torch.searchsorted(cdf, u.to(o.device), right=True)


def relocation_ratio(src, P):
    """N[r] = 1 + (number of entries drawing the same source): the source and its copies share its opacity."""
    return (torch.bincount(src, minlength=P)[src] + 1).to(torch.int32)


def relocation_values(opacity, scaling, ratio, scale_lower_bound=0.0, isotropic=False):
    """The relocation formula as an fp64 torch statement (what `dgs_mcmc_relocate` computes per entry):
    raw opacity' and raw scaling' [n,3] (float32) of a source with raw opacity [n] / [n,1], raw scaling [n,3] that is
    split N = ratio ways.  Also returns o' before its clamp and the scale coefficient c (float64)."""
    N = ratio.reshape(-1).to(torch.float64).clamp(1, N_MAX)
    o = opacity.reshape(-1).to(torch.float64).clamp(0.0, 1.0)
    o_new = -torch.expm1(torch.log1p(-o) / N)
    j = torch.arange(1, N_MAX + 1, dtype=torch.float64, device=o.device)
    # C(N, j) (0 for j > N), exact in fp64: C(51, 25) < 2^53
    table = torch.tensor([[float(math.comb(n, k)) for k in range(1, N_MAX + 1)] for n in range(N_MAX + 1)],
                         dtype=torch.float64, device=o.device)
    binom = table[N.long()]
    sign = torch.where(j % 2 == 1, 1.0, -1.0).to(torch.float64)
    D = (sign * binom * o_new[:, None] ** j / torch.sqrt(j)).sum(1)
    c = o / D
    raw = scaling.to(torch.float64)
    if isotropic:
        raw = raw[:, :1].expand(-1, 3)
    lb = float(scale_lower_bound)
    if lb == 0.0:
        sc = raw + torch.log(c)[:, None]
    else:
        sc = torch.log((c[:, None] * (torch.exp(raw) + lb) - lb).clamp_min(0.001))
    op = o_new.clamp_max(MAX_OPACITY).float().clamp_min(MIN_OPACITY_F32)
    return op.reshape(opacity.shape), sc.float(), o_new, c


@torch.no_grad()
def add_sgld_noise(gaussians, lr, step, noise_lr=5e5, seed=0):
    """The SGLD move of 3DGS-MCMC after the optimizer step: xyz += Sigma eps gate(o) noise_lr lr in place, Sigma the
    Gaussian's covariance (unfiltered scale), gate = 1 / (1 + exp(-100 ((1 - o) - 0.995))), eps ~ N(0, I3) a pure
    function of (seed, step, row).  `lr`: the current learning rate of the optimizer's 'xyz' group.  One launch."""
    xyz, sc, rot, op = gaussians._xyz, gaussians._scaling, gaussians._rotation, gaussians._opacity
    if not xyz.is_cuda:
        raise _lib.DgsError("add_sgld_noise: CUDA tensors required (libdgs_b200 has no CPU path)")
    for t in (xyz, sc, rot, op):
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise _lib.DgsError("add_sgld_noise: the store's tensors must be contiguous float32")
    lib = _lib.load()
    dev = xyz.device
    with torch.cuda.device(dev):
        rc = lib.dgs_mcmc_noise(xyz.shape[0], xyz.data_ptr(), sc.data_ptr(), rot.data_ptr(), op.data_ptr(),
                                float(gaussians.scale_lower_bound), int(bool(gaussians.use_isotropic)),
                                float(noise_lr) * float(lr), NOISE_K, NOISE_X0, int(seed) & 0xFFFFFFFFFFFFFFFF,
                                int(step), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _lib.check(rc, "dgs_mcmc_noise")


def debug_normals(P, seed, step, device):
    """The eps [P,3] `add_sgld_noise` draws for (seed, step) (test hook, `dgs_debug_mcmc_normals`)."""
    lib = _lib.load()
    out = torch.empty((P, 3), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        rc = lib.dgs_debug_mcmc_normals(P, int(seed) & 0xFFFFFFFFFFFFFFFF, int(step), _lib.ptr(out),
                                        C.c_void_p(torch.cuda.current_stream(device).cuda_stream))
    _lib.check(rc, "dgs_debug_mcmc_normals")
    return out


def growth_target(P, cap_max, growth):
    """Rows `add_new_gs` appends: min(cap_max, floor((1 + growth) P)) - P, at least 0."""
    return max(0, min(int(cap_max), int(math.floor((1.0 + growth) * P))) - P)
