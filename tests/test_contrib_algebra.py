"""CPU: the fixed-point algebra of the contribution scores (include/dgs_b200.h, dgs_blur_forward_contrib), the
selection of DensificationMixin.prune_by_contribution, the ContributionScores container, the C-ABI argument checks
and the cross-rank reduction of dist.all_reduce_contribution."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from deblurgs_b200 import _lib, synthetic
from deblurgs_b200 import dist as dd
from deblurgs_b200 import rasterizer as rz
from deblurgs_b200.motion import GaussianParams

SCALE = 1 << 26
W_MAX = 0.99          # alpha <= 0.99 and T <= 1: no blending weight is larger


def test_scale_is_the_header_define():
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "dgs_b200.h")).read()
    assert "#define DGS_CONTRIB_SCALE (1 << 26)" in hdr
    assert rz.CONTRIB_SCALE == SCALE


def test_warp_sum_cannot_overflow_32_bits():
    # one lane rounds two pixels, REDUX sums 32 lanes: 64 pixels of at most round(0.99 * 2^26) each
    per_pixel = int(np.rint(np.float32(W_MAX) * np.float32(SCALE)))
    assert 64 * per_pixel < 2 ** 32
    assert 64 * W_MAX * SCALE < 2 ** 32


def test_u64_sum_has_headroom_for_a_c3_sweep_of_1000_views():
    # a Gaussian can blend in at most every pixel of every sub-frame of every view, with weight <= 0.99
    _, W, H, F, _ = synthetic.CONFIGS["c3"]
    worst = 1000 * F * W * H * round(W_MAX * SCALE)
    assert worst < 2 ** 63          # also fits the int64 that holds it on the Python side
    assert worst < 2 ** 64


def _fixed_point_warp(w):
    """The kernel's arithmetic for one (warp, entry) pair: w [64] float32 in lane order (pixel 2k, 2k+1 = lane k's
    two rows); per lane round-to-nearest of w * 2^26, the pair added in u32, the 32 lanes summed (REDUX)."""
    q = np.rint(w.astype(np.float32) * np.float32(SCALE)).astype(np.uint64)   # __float2uint_rn, exact scaling
    lane = (q[0::2] + q[1::2]).astype(np.uint32)
    return int(lane.astype(np.uint64).sum())


def test_fixed_point_sum_equals_the_float64_sum_within_n_times_2_to_minus_27():
    rng = np.random.default_rng(0)
    total_q, total_f, n = 0, 0.0, 0
    for _ in range(2000):
        w = (rng.random(64) * W_MAX).astype(np.float32)
        w[rng.random(64) < 0.4] = 0.0                        # pixels that did not blend contribute exact zeros
        nz = int((w > 0).sum())
        q = _fixed_point_warp(w)
        assert q < 2 ** 32
        f = float(w.astype(np.float64).sum())
        assert abs(q / SCALE - f) <= nz * 2.0 ** -27
        total_q += q
        total_f += f
        n += nz
    assert abs(total_q / SCALE - total_f) <= n * 2.0 ** -27
    # the largest weights of a full warp still fit
    assert _fixed_point_warp(np.full(64, W_MAX, np.float32)) < 2 ** 32


def test_max_as_float_bits_orders_like_the_floats():
    rng = np.random.default_rng(1)
    w = np.concatenate([[0.0, 1e-30, 1e-7, W_MAX], rng.random(1000) * W_MAX]).astype(np.float32)
    bits = w.view(np.uint32)
    assert np.array_equal(np.argsort(bits, kind="stable"), np.argsort(w, kind="stable"))


def test_contribution_scores_decode_and_reset():
    sc = rz.ContributionScores(4, "cpu")
    assert sc.wsum.dtype == torch.int64 and sc.wmax.dtype == torch.int32 and sc.num_points == 4
    sc.wsum.copy_(torch.tensor([0, SCALE, 3 * SCALE // 2, 7]))
    sc.wmax.copy_(torch.tensor([0.0, 0.5, 0.99, 1e-6], dtype=torch.float32).view(torch.int32))
    assert sc.weight_sum.dtype == torch.float64
    assert torch.equal(sc.weight_sum, torch.tensor([0.0, 1.0, 1.5, 7.0 / SCALE], dtype=torch.float64))
    assert torch.equal(sc.weight_max, torch.tensor([0.0, 0.5, 0.99, 1e-6], dtype=torch.float32))
    sc.reset()
    assert int(sc.wsum.abs().sum()) == 0 and int(sc.wmax.abs().sum()) == 0


def test_forward_with_scores_of_another_size_is_rejected():
    sc = rz.ContributionScores(5, "cpu")
    with pytest.raises(_lib.DgsError, match="holds 5 Gaussians"):
        sc._check(6, torch.device("cpu"))


def _store(P=10, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.rand(*s, generator=g)
    gp = GaussianParams(r(P, 3), r(P, 1, 3), r(P, 3, 3), r(P, 3) - 2.0, r(P, 4), r(P, 1), 1)
    opt = gp.training_setup()
    for group in opt.param_groups:            # non-trivial Adam state: the moments are the parameters' row ids
        p = group["params"][0]
        row = torch.arange(P, dtype=torch.float32).view((P,) + (1,) * (p.dim() - 1)).expand_as(p)
        opt.state[p] = {"step": torch.tensor(3.0), "exp_avg": row.clone(), "exp_avg_sq": row.clone() + 100.0}
    return gp, opt


def _scores(wsum, wmax):
    sc = rz.ContributionScores(len(wsum), "cpu")
    sc.wsum.copy_(torch.tensor(wsum, dtype=torch.int64))
    sc.wmax.copy_(torch.tensor(wmax, dtype=torch.float32).view(torch.int32))
    return sc


def _kept_rows(gp, opt):
    """Original row ids of the surviving Gaussians, read back from the carried Adam moments."""
    rows = None
    for group in opt.param_groups:
        st = opt.state[group["params"][0]]
        r = st["exp_avg"].reshape(st["exp_avg"].shape[0], -1)[:, 0]
        assert torch.equal(st["exp_avg_sq"].reshape(r.shape[0], -1)[:, 0], r + 100.0)
        assert group["params"][0].shape[0] == r.shape[0]
        if rows is None:
            rows = r
        assert torch.equal(rows, r)
    return rows.long().tolist()


def test_prune_by_contribution_fraction_and_threshold():
    gp, opt = _store()
    xyz0 = gp._xyz.detach().clone()
    wsum = [50, 10, 90, 30, 70, 20, 80, 60, 40, 100]
    wmax = [0.5, 0.5, 0.5, 0.5, 0.001, 0.5, 0.5, 0.5, 0.5, 0.002]
    mask = gp.prune_by_contribution(_scores(wsum, wmax), fraction=0.3, min_weight_max=0.005)
    removed = {1, 5, 3} | {4, 9}         # three lowest sums, plus the two below the max-weight threshold
    assert set(torch.nonzero(mask).squeeze(1).tolist()) == removed
    kept = [i for i in range(10) if i not in removed]
    assert _kept_rows(gp, opt) == kept
    assert torch.equal(gp._xyz.detach(), xyz0[kept])
    assert gp.xyz_gradient_accum.shape == (len(kept), 1)


def test_prune_by_contribution_breaks_ties_by_index():
    gp, opt = _store()
    wsum = [5, 3, 3, 3, 9, 3, 7, 1, 3, 8]           # 1 (index 7), then 3 at indices 1, 2, 3, 5, 8
    mask = gp.prune_by_contribution(_scores(wsum, [0.5] * 10), fraction=0.4)
    assert torch.nonzero(mask).squeeze(1).tolist() == [1, 2, 3, 7]
    assert _kept_rows(gp, opt) == [0, 4, 5, 6, 8, 9]


def test_prune_by_contribution_defaults_remove_nothing_and_check_the_size():
    gp, opt = _store()
    mask = gp.prune_by_contribution(_scores([0] * 10, [0.0] * 10))
    assert not mask.any() and _kept_rows(gp, opt) == list(range(10))
    with pytest.raises(ValueError):
        gp.prune_by_contribution(_scores([0] * 9, [0.0] * 9), fraction=0.5)
    with pytest.raises(ValueError):
        gp.prune_by_contribution(_scores([0] * 10, [0.0] * 10), fraction=1.5)


def _contrib_call(lib, wsum, wmax, aa, P=10, F=1):
    n = C.c_int64(0)
    cb = _lib.ALLOC_FN(lambda ctx, nbytes: 0)
    one = C.c_void_p(1)    # never dereferenced: validation fails first
    return lib.dgs_blur_forward_contrib(cb, None, cb, None, cb, None, P, F, 3, 16, one, 32, 32, one, one, None, one,
                                        one, 1.0, one, None, one, one, one, 1.0, 1.0, 0.2, 100.0, 0, 0, one, one, one,
                                        None, 1.0, 0, C.byref(n), aa, wsum, wmax, None)


def test_contrib_entry_rejects_null_scores_before_device_work():
    lib = _lib.load()
    one = C.c_void_p(1)
    for wsum, wmax in ((None, one), (one, None), (None, None)):
        assert _contrib_call(lib, wsum, wmax, 0) == -1
        assert b"contribution" in lib.dgs_last_error()


@pytest.mark.parametrize("aa", [2, -1])
def test_contrib_entry_rejects_a_bad_antialiasing_value(aa):
    lib = _lib.load()
    one = C.c_void_p(1)
    assert _contrib_call(lib, one, one, aa) == -1 and b"antialiasing" in lib.dgs_last_error()


def test_contrib_entry_keeps_the_other_argument_checks():
    lib = _lib.load()
    one = C.c_void_p(1)
    assert _contrib_call(lib, one, one, 0, P=-1) == -1 and b"negative" in lib.dgs_last_error()


def test_python_surface_defaults_to_no_scores():
    import inspect
    from deblurgs_b200 import renderer
    from deblurgs_b200.motion import CameraMotionModule
    for fn in (rz.rasterize_gaussians, rz.rasterize_blurry, rz.render_store_blurry, renderer.render,
               renderer.render_blurry, CameraMotionModule.query, dd.render_blurry_sharded):
        assert inspect.signature(fn).parameters["contrib"].default is None
    for fn in (renderer.render, renderer.render_blurry):
        assert inspect.signature(fn).parameters["contrib"].kind is inspect.Parameter.KEYWORD_ONLY


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        P = 9
        g = torch.Generator().manual_seed(7)
        wsum = torch.randint(0, 2 ** 40, (world, P), generator=g)
        wmax = (torch.rand(world, P, generator=g) * 0.99).float()
        sc = rz.ContributionScores(P, "cpu")
        sc.wsum.copy_(wsum[rank])
        sc.wmax.copy_(wmax[rank].view(torch.int32))
        assert dd.all_reduce_contribution(sc) is sc
        assert torch.equal(sc.wsum, wsum.sum(0))                      # exact integer sum
        assert torch.equal(sc.weight_max, wmax.max(0).values)         # max of the float bits = max of the floats
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        q.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_world2_gloo_all_reduce_contribution():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=100) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res


def test_all_reduce_contribution_is_the_identity_without_a_process_group():
    sc = _scores([1, 2], [0.1, 0.2])
    assert dd.all_reduce_contribution(sc) is sc and sc.wsum.tolist() == [1, 2]
