"""CPU: 3DGS-MCMC densification (deblurgs_b200/mcmc.py, DensificationMixin.relocate_gs / add_new_gs): the relocation
formula's closed form against a 60-digit evaluation of the paper's double sum, the integer-CDF sampler, and the
in-place relocation and growth of a CPU store with both optimizers that share torch's `param_groups` / `state` layout
(the semantics the GPU path is tested against), plus the C-ABI's argument checks."""
import ctypes as C
import math

import pytest
import torch

from deblurgs_b200 import _lib, mcmc
from deblurgs_b200.motion import GaussianParams

mpmath = pytest.importorskip("mpmath")
mpmath.mp.dps = 60

OPACITIES = [1e-4, 0.005, 0.3, 0.9, 0.999, 1.0 - 2.0 ** -23]
NAMES = ["xyz", "f_dc", "f_rest", "opacity", "scaling", "rotation"]
ATTR = {"xyz": "_xyz", "f_dc": "_features_dc", "f_rest": "_features_rest", "opacity": "_opacity",
        "scaling": "_scaling", "rotation": "_rotation"}


def _mp_coeffs(o, N):
    """(o', D as the paper's double sum, D in closed form) at 60 digits."""
    o = mpmath.mpf(o)
    on = 1 - (1 - o) ** (mpmath.mpf(1) / N)
    double = mpmath.fsum(mpmath.binomial(i - 1, k) * (-1) ** k * on ** (k + 1) / mpmath.sqrt(k + 1)
                         for i in range(1, N + 1) for k in range(i))
    closed = mpmath.fsum((-1) ** (j - 1) * mpmath.binomial(N, j) * on ** j / mpmath.sqrt(j) for j in range(1, N + 1))
    return on, double, closed


def test_closed_form_equals_the_double_sum_and_the_fp64_statement_matches_it():
    Ns = list(range(1, mcmc.N_MAX + 1))
    o_grid = torch.tensor([o for o in OPACITIES for _ in Ns], dtype=torch.float64)
    N_grid = torch.tensor([N for _ in OPACITIES for N in Ns], dtype=torch.int32)
    _, _, o_new, c = mcmc.relocation_values(o_grid, torch.zeros(len(o_grid), 3), N_grid)
    worst = 0.0
    for i, (o, N) in enumerate(zip(o_grid.tolist(), N_grid.tolist())):
        on, double, closed = _mp_coeffs(o, N)
        assert abs(double - closed) <= mpmath.mpf(10) ** -40 * abs(double)
        c_ref = mpmath.mpf(o) / closed
        worst = max(worst, float(abs(float(c[i]) - c_ref) / c_ref), float(abs(float(o_new[i]) - on) / on))
        # 1 - (1 - o')^N = o
        assert abs(1 - (1 - on) ** N - o) <= mpmath.mpf(10) ** -50
    assert worst <= 1e-9, worst


def test_single_copy_is_the_identity():
    o = torch.tensor(OPACITIES, dtype=torch.float64)
    raw = torch.randn(len(OPACITIES), 3, generator=torch.Generator().manual_seed(0))
    op, sc, o_new, c = mcmc.relocation_values(o, raw, torch.ones(len(OPACITIES), dtype=torch.int32))
    assert torch.allclose(c, torch.ones_like(c), rtol=1e-14, atol=0)
    assert torch.allclose(o_new, o, rtol=1e-14, atol=0)
    assert torch.equal(sc, raw)                          # raw + log(1)


def test_ratio_clamp_opacity_clamp_and_lower_bound_inverse():
    o = torch.tensor([0.9, 0.9, 0.006, 1.0], dtype=torch.float64)
    raw = torch.tensor([[-2.0, -1.0, -3.0]] * 4)
    op, sc, o_new, c = mcmc.relocation_values(o, raw, torch.tensor([51, 80, 4, 1], dtype=torch.int32))
    assert float(c[0]) == float(c[1])                   # N clamped to 51
    assert float(op[2]) == pytest.approx(0.005, rel=1e-7)   # 1 - 0.994^(1/4) < 0.005: clamped up
    assert float(op[2]) > 0.005                             # ... to a float that is not dead by `<= 0.005`
    assert float(op[3]) == pytest.approx(1.0 - 2.0 ** -23, rel=0, abs=0)
    lb = 1e-3
    op2, sc2, _, c2 = mcmc.relocation_values(o, raw, torch.tensor([3, 3, 3, 3], dtype=torch.int32), lb)
    s = torch.exp(raw.double()) + lb
    assert torch.allclose(sc2.double(), torch.log((c2[:, None] * s - lb).clamp_min(1e-3)), rtol=1e-6)
    # isotropic: every column from column 0
    _, sc3, _, _ = mcmc.relocation_values(o, raw, torch.tensor([3, 3, 3, 3], dtype=torch.int32), 0.0, True)
    assert torch.equal(sc3[:, 1], sc3[:, 0]) and torch.equal(sc3[:, 2], sc3[:, 0])


# ---- sampler ---------------------------------------------------------------------------------------------------------
def test_sampler_never_draws_zero_weight_rows_and_matches_the_distribution():
    from scipy import stats
    g = torch.Generator().manual_seed(5)
    o = torch.rand(50, generator=g)
    o[::3] = 0.0                                        # dead rows
    o[1] = 1e-8                                         # floor(1e-8 * 2^24) = 0: never drawn either
    n = 200_000
    idx = mcmc.sample_by_opacity(o, n, torch.Generator().manual_seed(1))
    w = torch.floor(o.double() * 2.0 ** 24)
    assert bool((w[idx] > 0).all())
    counts = torch.bincount(idx, minlength=50).double()
    live = w > 0
    expected = w[live] / w.sum() * n
    chi2, p = stats.chisquare(counts[live].numpy(), expected.numpy())
    assert p > 1e-3, (chi2, p)
    assert torch.equal(idx, mcmc.sample_by_opacity(o, n, torch.Generator().manual_seed(1)))
    assert not torch.equal(idx, mcmc.sample_by_opacity(o, n, torch.Generator().manual_seed(2)))
    with pytest.raises(ValueError):
        mcmc.sample_by_opacity(torch.zeros(4), 3)


def test_sampler_beyond_2_to_the_24_rows():
    P = (1 << 24) + 1000
    o = torch.zeros(P)
    o[-7:] = torch.tensor([0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7])    # only rows past 2^24 are live
    idx = mcmc.sample_by_opacity(o, 10_000, torch.Generator().manual_seed(3))
    assert int(idx.min()) >= P - 7 and int(idx.max()) == P - 1


# ---- relocation / growth of a CPU store ------------------------------------------------------------------------------
def _store(P=60, M=4, seed=0, optimizer_cls=None, lb=0.0, isotropic=False, filter3d=False):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    gp = GaussianParams(r(P, 3), r(P, 1, 3), r(P, M - 1, 3), r(P, 3) * 0.5 - 2.0, r(P, 4),
                        torch.rand(P, 1, generator=g) * 0.9 + 0.05, 1, scale_lower_bound=lb, use_isotropic=isotropic)
    if filter3d:
        gp.filter_3D = torch.rand(P, 1, generator=g) * 0.01
    opt = gp.training_setup(optimizer_cls=optimizer_cls)
    for grp in opt.param_groups:
        p = grp["params"][0]
        opt.state[p] = {"step": 7 if optimizer_cls is None else torch.tensor(7.0), "exp_avg": r(*p.shape),
                        "exp_avg_sq": r(*p.shape).abs()}
    gp._ensure_stats()
    gp.xyz_gradient_accum += torch.rand(P, 1, generator=g)
    gp.denom += 1.0
    gp.max_radii2D += torch.arange(P).float() + 1.0
    return gp, opt


def _snapshot(gp, opt):
    snap = {}
    for grp in opt.param_groups:
        p = grp["params"][0]
        st = opt.state[p]
        snap[grp["name"]] = (p, p.detach().clone(), st["exp_avg"], st["exp_avg"].clone(), st["exp_avg_sq"].clone(),
                             float(st["step"]))
    stats = [(t, t.clone()) for t in (gp.xyz_gradient_accum, gp.denom, gp.max_radii2D)]
    filt = None if gp.filter_3D is None else (gp.filter_3D, gp.filter_3D.clone())
    return snap, stats, filt


def _check_relocated(gp, opt, before, dst, src, n_rows):
    """dst rows = copies of src rows (apart from opacity / scaling), opacity / scaling = the fp64 statement at dst and
    src, moments / statistics zeroed at dst and src, every other row bit-unchanged, identity and step counts kept."""
    snap, stats, filt = before
    touched = torch.zeros(n_rows, dtype=torch.bool)
    touched[dst] = True
    touched[src] = True
    ratio = mcmc.relocation_ratio(src, n_rows)
    op, sc, _, _ = mcmc.relocation_values(snap["opacity"][1][src], snap["scaling"][1][src], ratio,
                                          gp.scale_lower_bound, gp.use_isotropic)
    for name in NAMES:
        p0, v0, m_obj, m0, v_sq0, step0 = snap[name]
        p = getattr(gp, ATTR[name])
        st = opt.state[p]
        assert p is p0 and st["exp_avg"] is m_obj and float(st["step"]) == step0
        v = p.detach()
        assert torch.equal(v[~touched], v0[~touched])
        if name == "opacity":
            assert torch.equal(v[dst], op) and torch.equal(v[src], op)
        elif name == "scaling":
            assert torch.equal(v[dst], sc) and torch.equal(v[src], sc)
        else:
            assert torch.equal(v[dst], v0[src]) and torch.equal(v[src], v0[src])
        for cur, old in ((st["exp_avg"], m0), (st["exp_avg_sq"], v_sq0)):
            assert torch.equal(cur[~touched], old[~touched]) and float(cur[touched].abs().max()) == 0.0
    for (t, old), cur in zip(stats, (gp.xyz_gradient_accum, gp.denom, gp.max_radii2D)):
        assert cur is t and torch.equal(t[~touched], old[~touched]) and float(t[touched].abs().max()) == 0.0
    if filt is not None:
        assert gp.filter_3D is filt[0]
        assert torch.equal(gp.filter_3D[~touched], filt[1][~touched]) and torch.equal(gp.filter_3D[dst], filt[1][src])


@pytest.mark.parametrize("optimizer_cls", [None, torch.optim.Adam])
@pytest.mark.parametrize("lb,isotropic", [(0.0, False), (1e-3, False), (0.0, True)])
def test_relocate_in_place(optimizer_cls, lb, isotropic):
    gp, opt = _store(optimizer_cls=optimizer_cls, lb=lb, isotropic=isotropic, filter3d=True)
    with torch.no_grad():
        gp._opacity[[3, 10, 11, 40]] = torch.tensor([[0.0], [0.004], [0.005], [-0.2]])
        gp._opacity[[0, 1]] = torch.tensor([[1.0], [0.999]])       # heavy sources: drawn more than once
    before = _snapshot(gp, opt)
    # the plan relocate_gs draws with this generator
    dead = gp.get_opacity.detach().reshape(-1) <= 0.005
    w = torch.where(dead, torch.zeros_like(gp.get_opacity.detach().reshape(-1)), gp.get_opacity.detach().reshape(-1))
    src = mcmc.sample_by_opacity(w, 4, torch.Generator().manual_seed(11))
    n = gp.relocate_gs(generator=torch.Generator().manual_seed(11))
    assert n == 4
    _check_relocated(gp, opt, before, torch.tensor([3, 10, 11, 40]), src, 60)
    assert float(gp.get_opacity.detach().min()) >= 0.005 - 1e-9
    if optimizer_cls is torch.optim.Adam:       # still steppable
        for p in gp.parameters():
            p.grad = torch.ones_like(p)
        opt.step()
        assert all(float(opt.state[p]["step"]) == 8.0 for p in gp.parameters())


def test_relocate_with_many_copies_of_one_source_and_explicit_mask():
    gp, opt = _store(P=200, seed=4)
    dead = torch.zeros(200, dtype=torch.bool)
    dead[100:] = True
    with torch.no_grad():
        gp._opacity[:100] = 0.001
        gp._opacity[7] = 0.99                     # ~100 draws of the same source: ratio beyond 51, clamped
    before = _snapshot(gp, opt)
    w = torch.where(dead, torch.zeros(200), gp.get_opacity.detach().reshape(-1))
    src = mcmc.sample_by_opacity(w, 100, torch.Generator().manual_seed(2))
    assert int((src == 7).sum()) > 51
    assert gp.relocate_gs(dead_mask=dead, generator=torch.Generator().manual_seed(2)) == 100
    _check_relocated(gp, opt, before, torch.arange(100, 200), src, 200)


def test_relocate_does_nothing_without_dead_or_live_rows():
    gp, opt = _store()
    before = [t.detach().clone() for t in gp.parameters()]
    assert gp.relocate_gs() == 0                                       # every opacity >= 0.05
    assert gp.relocate_gs(dead_mask=torch.ones(60, dtype=torch.bool)) == 0   # nothing live to draw from
    assert all(torch.equal(a, b.detach()) for a, b in zip(before, gp.parameters()))


@pytest.mark.parametrize("optimizer_cls", [None, torch.optim.Adam])
def test_add_new_gs_grows_by_the_stated_amount_and_stops_at_the_cap(optimizer_cls):
    gp, opt = _store(P=100, optimizer_cls=optimizer_cls, filter3d=True)
    snap, stats, filt = _snapshot(gp, opt)
    src = mcmc.sample_by_opacity(gp.get_opacity.detach(), 5, torch.Generator().manual_seed(9))
    assert gp.add_new_gs(cap_max=1000, generator=torch.Generator().manual_seed(9)) == 5   # floor(1.05 * 100) - 100
    assert gp._xyz.shape[0] == 105
    # the same result as a relocation onto 5 appended rows: rebuild the expectation on the old tensors
    touched = torch.zeros(105, dtype=torch.bool)
    touched[100:] = True
    touched[src] = True
    ratio = mcmc.relocation_ratio(src, 100)
    op, sc, _, _ = mcmc.relocation_values(snap["opacity"][1][src], snap["scaling"][1][src], ratio)
    for name in NAMES:
        p = getattr(gp, ATTR[name])
        st = opt.state[p]
        assert opt.param_groups[NAMES.index(name)]["params"][0] is p and float(st["step"]) == snap[name][5]
        v, v0 = p.detach(), snap[name][1]
        keep = ~touched[:100]
        assert torch.equal(v[:100][keep], v0[keep])
        if name == "opacity":
            assert torch.equal(v[100:], op) and torch.equal(v[src], op)
        elif name == "scaling":
            assert torch.equal(v[100:], sc) and torch.equal(v[src], sc)
        else:
            assert torch.equal(v[100:], v0[src])
        for cur, old in ((st["exp_avg"], snap[name][3]), (st["exp_avg_sq"], snap[name][4])):
            assert cur.shape == v.shape and torch.equal(cur[:100][keep], old[keep])
            assert float(cur[touched].abs().max()) == 0.0
    for (_, old), cur in zip(stats, (gp.xyz_gradient_accum, gp.denom, gp.max_radii2D)):
        assert cur.shape[0] == 105 and torch.equal(cur[:100][~touched[:100]], old[~touched[:100]])
        assert float(cur[touched].abs().max()) == 0.0
    assert torch.equal(gp.filter_3D[100:], filt[1][src])
    assert gp.add_new_gs(cap_max=107) == 2                 # capped
    assert gp.add_new_gs(cap_max=107) == 0 and gp._xyz.shape[0] == 107
    assert gp.add_new_gs(cap_max=50) == 0                  # above the cap already: no-op
    assert mcmc.growth_target(100, 10**9, 0.05) == 5 and mcmc.growth_target(19, 10**9, 0.05) == 0


def test_mcmc_regularization_is_the_torch_statement():
    from deblurgs_b200.loss import mcmc_regularization
    gp, _ = _store()
    v = mcmc_regularization(gp, 0.01, 0.02)
    expect = 0.01 * gp._opacity.clamp(0, 1).abs().mean() + 0.02 * (torch.exp(gp._scaling)).abs().mean()
    assert torch.allclose(v, expect, rtol=1e-6)
    v.backward()
    assert gp._opacity.grad is not None and gp._scaling.grad is not None


def test_mcmc_entry_points_validate_arguments():
    lib = _lib.load()
    one = C.c_void_p(1)   # never dereferenced: validation fails first
    n = 3
    ptrs = (C.c_void_p * n)(1, 1, 1)
    width_ok, kind_ok = (C.c_int * n)(3, 1, 3), (C.c_int * n)(0, 1, 2)
    args = (one, one, one, 0.0, 0, one, None)
    assert lib.dgs_mcmc_relocate(n, ptrs, width_ok, kind_ok, -1, *args) == -1
    assert lib.dgs_mcmc_relocate(25, ptrs, width_ok, kind_ok, 4, *args) == -1           # > DGS_GATHER_MAX_TENSORS
    assert lib.dgs_mcmc_relocate(n, ptrs, width_ok, (C.c_int * n)(0, 1, 1), 4, *args) == -1   # no scaling tensor
    assert lib.dgs_mcmc_relocate(n, ptrs, (C.c_int * n)(3, 2, 3), kind_ok, 4, *args) == -1   # opacity of width 2
    assert lib.dgs_mcmc_relocate(n, ptrs, width_ok, (C.c_int * n)(0, 1, 7), 4, *args) == -1   # unknown kind
    assert lib.dgs_mcmc_relocate(n, ptrs, width_ok, kind_ok, 4, one, one, None, 0.0, 0, one, None) == -1
    assert lib.dgs_mcmc_relocate(n, ptrs, width_ok, kind_ok, 4, one, one, one, -1.0, 0, one, None) == -1
    assert b"dgs_mcmc_relocate" in lib.dgs_last_error()
    assert lib.dgs_mcmc_relocate(n, ptrs, width_ok, kind_ok, 0, None, None, None, 0.0, 0, None, None) == 0
    assert lib.dgs_mcmc_relocate_scratch_bytes(10) == 160 and lib.dgs_mcmc_relocate_scratch_bytes(0) == 0
    assert lib.dgs_mcmc_noise(-1, one, one, one, one, 0.0, 0, 1.0, 100.0, 0.995, 0, 0, None) == -1
    assert lib.dgs_mcmc_noise(10, one, None, one, one, 0.0, 0, 1.0, 100.0, 0.995, 0, 0, None) == -1
    assert lib.dgs_mcmc_noise(10, one, one, one, one, 0.0, 0, 1.0, 100.0, 0.995, 0, -1, None) == -1
    assert lib.dgs_mcmc_noise(0, None, None, None, None, 0.0, 0, 1.0, 100.0, 0.995, 0, 0, None) == 0
    assert lib.dgs_debug_mcmc_normals(10, 0, 0, None, None) == -1
    assert lib.dgs_debug_mcmc_normals(0, 0, 0, None, None) == 0


def test_noise_needs_cuda_tensors():
    gp, _ = _store()
    with pytest.raises(_lib.DgsError, match="CUDA"):
        mcmc.add_sgld_noise(gp, lr=1e-4, step=0)
    assert math.isclose(mcmc.NOISE_K * ((1 - 0.5) - mcmc.NOISE_X0), -49.5)
