"""GPU: 3DGS-MCMC densification on sm_100a (csrc/dgs_mcmc.cu).  The in-place relocation against the CPU path of
`relocate_gs` on a 300k store whose sources are drawn up to and beyond 51 times; the SGLD noise (its Philox normals,
the move against a float64 statement, determinism and the opacity gate); a captured training step replayed after a
relocation and a noise step; and a short MCMC training run."""
import numpy as np
import pytest
import torch

from deblurgs_b200 import mcmc
from deblurgs_b200.densify import build_rotation
from deblurgs_b200.motion import GaussianParams

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def _store(P, device, seed=0, n_heavy=10):
    """Half the rows dead (opacity 0.001), live rows at 0.01 except `n_heavy` at 0.99 (each drawn ~100 times by a
    relocation of every dead row); optimizer state and statistics on every row."""
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    op = torch.full((P, 1), 0.01)
    op[P // 2:] = 0.001
    op[torch.randperm(P // 2, generator=g)[:n_heavy]] = 0.99
    gp = GaussianParams(r(P, 3), r(P, 1, 3), r(P, 15, 3), r(P, 3) * 0.5 - 2.0, r(P, 4), op, 3)
    gp.filter_3D = torch.rand(P, 1, generator=g) * 0.01
    opt = gp.training_setup()
    for grp in opt.param_groups:
        p = grp["params"][0]
        opt.state[p] = {"step": 7, "exp_avg": r(*p.shape), "exp_avg_sq": r(*p.shape).abs()}
    gp._ensure_stats()
    gp.xyz_gradient_accum += torch.rand(P, 1, generator=g)
    gp.denom += 1.0
    gp.max_radii2D += 1.0
    if device.type == "cuda":
        gp = _to(gp, device)
    return gp


def _to(gp, device):
    out = GaussianParams(*(t.detach().to(device) for t in gp.parameters()), gp.active_sh_degree)
    out.filter_3D = gp.filter_3D.to(device)
    opt = out.training_setup()
    for grp, old in zip(opt.param_groups, gp.optimizer.param_groups):
        st = gp.optimizer.state[old["params"][0]]
        opt.state[grp["params"][0]] = {"step": st["step"], "exp_avg": st["exp_avg"].to(device),
                                       "exp_avg_sq": st["exp_avg_sq"].to(device)}
    out._ensure_stats()
    out.xyz_gradient_accum, out.denom = gp.xyz_gradient_accum.to(device), gp.denom.to(device)
    out.max_radii2D = gp.max_radii2D.to(device)
    return out


def _tensors(gp):
    ts = {}
    for grp in gp.optimizer.param_groups:
        p = grp["params"][0]
        st = gp.optimizer.state[p]
        ts[grp["name"]] = p.detach()
        ts[grp["name"] + ".exp_avg"], ts[grp["name"] + ".exp_avg_sq"] = st["exp_avg"], st["exp_avg_sq"]
    ts.update(accum=gp.xyz_gradient_accum, denom=gp.denom, max_radii2D=gp.max_radii2D, filter_3D=gp.filter_3D)
    return ts


def test_relocation_matches_the_cpu_path_at_300k():
    P = 300_000
    cpu, gpu, gpu2 = _store(P, torch.device("cpu")), _store(P, DEV), _store(P, DEV)
    ptrs = {k: v.data_ptr() for k, v in _tensors(gpu).items()}
    # the plan all three draw: sources shared up to ~100 times (ratio clamped to 51) and once or twice
    w = torch.where(cpu.get_opacity.reshape(-1) <= 0.005, 0.0, cpu.get_opacity.reshape(-1).detach())
    src = mcmc.sample_by_opacity(w, P // 2, torch.Generator().manual_seed(7))
    counts = torch.bincount(src)
    assert int(counts.max()) > 51 and int(((counts > 0) & (counts <= 2)).sum()) > 1000
    n = [s.relocate_gs(generator=torch.Generator().manual_seed(7)) for s in (cpu, gpu, gpu2)]
    assert n == [P // 2] * 3
    torch.cuda.synchronize()
    t_cpu, t_gpu, t_gpu2 = _tensors(cpu), _tensors(gpu), _tensors(gpu2)
    assert {k: v.data_ptr() for k, v in t_gpu.items()} == ptrs          # in place: every tensor keeps its storage
    for k, v in t_cpu.items():
        got = t_gpu[k].cpu()
        assert torch.equal(t_gpu[k], t_gpu2[k]), k                          # run to run: bit for bit
        if k in ("opacity", "scaling"):
            rel = ((got.double() - v.double()).abs() / v.double().abs().clamp_min(1e-30)).max().item()
            assert rel <= 1e-6, (k, rel)
        else:
            assert torch.equal(got, v), k
    assert float(gpu.get_opacity.detach().min()) > 0.005
    assert all(float(gpu.optimizer.state[p]["step"]) == 7 for p in gpu.parameters())


def _noise_store(P, seed=1):
    g = torch.Generator().manual_seed(seed)
    gp = GaussianParams(torch.zeros(P, 3), torch.zeros(P, 1, 3), torch.zeros(P, 0, 3),
                        torch.rand(P, 3, generator=g) * 1.5 - 3.0, torch.randn(P, 4, generator=g),
                        torch.rand(P, 1, generator=g), 0)
    with torch.no_grad():
        gp._opacity[: P // 4] *= 0.02                 # near-transparent: the gate is open
        gp._opacity[P // 4: P // 4 + 1000] = 0.5      # gate ~3e-22: must stay put
        gp._opacity[-10:] = 1.0                       # exp overflows in the gate: exactly 0
    return _to_plain(gp, DEV)


def _to_plain(gp, device):
    return GaussianParams(*(t.detach().to(device) for t in gp.parameters()), gp.active_sh_degree)


def test_philox_normals_are_standard_normal_and_independent():
    from scipy import stats
    P = 400_000
    e = mcmc.debug_normals(P, 3, 7, DEV).double().cpu().numpy()
    for c in range(3):
        assert stats.kstest(e[:, c], "norm").pvalue > 1e-4, c
    bound = 5.0 / np.sqrt(P)
    corr = lambda a, b: abs(np.corrcoef(a, b)[0, 1])
    assert corr(e[:, 0], e[:, 1]) < bound and corr(e[:, 0], e[:, 2]) < bound and corr(e[:, 1], e[:, 2]) < bound
    for c in range(3):
        assert corr(e[:-1, c], e[1:, c]) < bound                            # adjacent g
    e8 = mcmc.debug_normals(P, 3, 8, DEV).double().cpu().numpy()
    e_other_seed = mcmc.debug_normals(P, 4, 7, DEV).double().cpu().numpy()
    for c in range(3):
        assert corr(e[:, c], e8[:, c]) < bound and corr(e[:, c], e_other_seed[:, c]) < bound   # adjacent step, seed
    again = mcmc.debug_normals(P, 3, 7, DEV).double().cpu().numpy()
    assert np.array_equal(e, again)
    # a pure function of (seed, step, g): a shorter launch draws the same prefix
    assert np.array_equal(mcmc.debug_normals(1000, 3, 7, DEV).double().cpu().numpy(), e[:1000])


def test_noise_move_equals_the_float64_statement():
    P = 200_000
    lr, noise_lr, seed, step = 1.6e-4, 5e5, 11, 3
    gp = _noise_store(P)
    eps = mcmc.debug_normals(P, seed, step, DEV).double()
    mcmc.add_sgld_noise(gp, lr, step, noise_lr=noise_lr, seed=seed)
    d = gp._xyz.detach().double()                                       # xyz started at 0: the move itself
    s = torch.exp(gp._scaling.detach().double())
    R = build_rotation(torch.nn.functional.normalize(gp._rotation.detach().double()))
    step_scale = float(np.float32(noise_lr * lr))
    x0 = float(np.float32(mcmc.NOISE_X0))
    o = gp._opacity.detach().double().clamp(0, 1)
    gate = 1.0 / (1.0 + torch.exp(-mcmc.NOISE_K * ((1.0 - o) - x0)))
    sigma = R @ torch.diag_embed(s * s) @ R.transpose(1, 2)
    d64 = (sigma @ eps[:, :, None])[:, :, 0] * gate * step_scale
    scale = (gate[:, 0] * step_scale * (s * s).max(1).values * eps.norm(dim=1))
    err = (d - d64).norm(dim=1)
    assert bool((err <= 1e-5 * scale + 1e-30).all()), float((err / scale.clamp_min(1e-30)).max())
    assert float(d[: P // 4].abs().max()) > 1e-4                        # the open gate really moves them
    assert float(d[P // 4: P // 4 + 1000].abs().max()) <= 1e-20         # o = 0.5
    assert float(d[-10:].abs().max()) == 0.0                            # o = 1
    # the same (seed, step) moves an identical store identically; another step does not
    gp2, gp3 = _noise_store(P), _noise_store(P)
    mcmc.add_sgld_noise(gp2, lr, step, noise_lr=noise_lr, seed=seed)
    mcmc.add_sgld_noise(gp3, lr, step + 1, noise_lr=noise_lr, seed=seed)
    assert torch.equal(gp2._xyz, gp._xyz) and not torch.equal(gp3._xyz, gp._xyz)


def _eager(w, gt, reg):
    from deblurgs_b200.loss import blur_photometric_loss, mcmc_regularization
    params = w["gaussians"].parameters() + w["cmm"].parameters()
    for p in params:
        p.grad = None
    out = w["cmm"].query(0, "all", background=w["bg"])
    loss = blur_photometric_loss(out["blurred"], out["subframes"], gt, 0.0)
    if reg:
        loss = loss + mcmc_regularization(w["gaussians"], reg, reg)
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), [p.grad.clone() for p in params]


@pytest.mark.parametrize("reg", [0.0, 0.01])
def test_graph_replays_after_relocation_and_noise_without_recapture(reg):
    import bench
    from deblurgs_b200.graph import BlurryViewGraph
    w = bench.build_workload("small", 0, DEV)
    store = w["gaussians"]
    store.training_setup()
    params = store.parameters() + w["cmm"].parameters()
    gt = w["gt_host"].to(DEV)
    g = BlurryViewGraph(w["cmm"], 0, w["bg"], (3, w["H"], w["W"]), 0.0, opacity_reg=reg, scale_reg=reg)
    graph = g.graph
    g.step(gt)
    dead = torch.zeros(w["P"], dtype=torch.bool, device=DEV)
    dead[::97] = True
    with torch.no_grad():
        store._opacity[::97] = 0.001
    assert store.relocate_gs(dead_mask=dead, generator=torch.Generator().manual_seed(0)) == int(dead.sum())
    mcmc.add_sgld_noise(store, lr=1e-3, step=1)
    l_ref, g_ref = _eager(w, gt, reg)
    val = g.step(gt)
    assert abs(val - l_ref) <= 1e-6
    for p, r in zip(params, g_ref):
        assert ((p.grad - r).abs().max() / r.abs().max().clamp_min(1e-30)).item() <= 1e-3
    assert g.graph is graph and g.recaptures == 0


def test_short_mcmc_training_run():
    import bench
    from deblurgs_b200.loss import blur_photometric_loss, mcmc_regularization
    w = bench.build_workload("small", 0, DEV)
    store, cmm = w["gaussians"], w["cmm"]
    opt = store.training_setup(position_lr_init=1.6e-5, feature_lr=0.01, opacity_lr=0.02, scaling_lr=0.002)
    gt = w["gt_host"].to(DEV)
    cap = int(w["P"] * 1.12)
    gen = torch.Generator().manual_seed(0)
    losses = []
    for it in range(60):
        for p in store.parameters():
            p.grad = None
        out = cmm.query(0, "all", background=w["bg"])
        loss = blur_photometric_loss(out["blurred"], out["subframes"], gt) + mcmc_regularization(store)
        loss.backward()
        opt.step()
        mcmc.add_sgld_noise(store, opt.param_groups[0]["lr"], it)
        losses.append(loss.item())
        if it % 10 == 9:
            with torch.no_grad():
                store._opacity[it::50] = 0.0          # some dead rows for every round
            assert store.relocate_gs(generator=gen) > 0
            assert int((store.get_opacity <= 0.005).sum()) == 0
            store.add_new_gs(cap, generator=gen)
            assert store._xyz.shape[0] <= cap
    assert store._xyz.shape[0] == cap
    assert losses[-1] < losses[0]
