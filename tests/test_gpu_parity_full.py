"""GPU parity at BASELINE.json's headline sizes (pytest -m gpu), against the stored outputs of the reference's own CUDA
rasterizer and of the reference extension driven by the reference's per-sub-frame loop and pose chain (the bench's
reference arm), stored in tests/golden/parity.npz:

  * c2 (300 k Gaussians, 600x400, F=16): every forward intermediate bit-exact / images <= 1e-4, and every
    gradient PER ELEMENT within max(1e-3, 2 x the reference's own run-to-run spread).  The reference accumulates
    with float atomics in scheduling order, so two runs of the reference on identical inputs differ; that spread
    was measured on a B200 (five reference runs, profiles/r2_final_gpu_tests.log) and is kept below.
  * c3 (1 M Gaussians, 1920x1080, F=16): forward only, same bars (63 M duplicates).
  * end to end at c1: gradients of the Bezier control points, the sub-frame alignment parameters and all
    Gaussian parameters from `CameraMotionModule.query` + L1 against the reference's per-sub-frame render loop.

Metric (north_star: "within 1e-3 relative error"): per element |a - b| / max(|b|, 1e-3 * max|b|).
"""
import pytest
import torch

from tests import parity_utils as pu
from tests.test_gpu_parity import _compare_forward

pytestmark = pytest.mark.gpu

GAUSS = ["dL_dmeans3D", "dL_dsh", "dL_dopacity", "dL_dscales", "dL_drotations"]
POSE = ["dL_dviewmatrix", "dL_dprojmatrix", "dL_dmeans2D"]
# the reference's run-to-run spread (per element, floor 1e-3 of the max): c2 gradients, five runs; c1 end to end, three
C2_NOISE = {"dL_dmeans3D": 1.51e-4, "dL_dsh": 2.70e-4, "dL_dopacity": 1.75e-4, "dL_dscales": 1.49e-3,
            "dL_drotations": 8.49e-4, "dL_dviewmatrix": 3.60e-4, "dL_dprojmatrix": 1.37e-3, "dL_dmeans2D": 9.54e-5}
C1_POSE_NOISE = {"ctrl_trans": 1.59e-4, "ctrl_rot": 1.92e-5, "nu": 1.12e-5}


def test_c2_forward_and_gradients_vs_reference_cuda_with_noise_floor(capsys):
    cam, scene, bg, view, proj, campos, fw = _compare_forward("c2")       # forward: bit-exact bars inside
    F, W, H = view.shape[0], cam.width, cam.height
    g = torch.Generator().manual_seed(7)
    dpix = (torch.randn(F, 3, H, W, generator=g) / (3 * H * W)).cuda()
    ddep = (torch.randn(F, 1, H, W, generator=g) / (H * W) * 0.1).cuda()
    mine = pu.ours_backward(cam, scene, bg, view, proj, campos, fw, dpix, ddep)
    gd = pu.Golden("bwd_c2")    # Gaussian gradients summed over the sub-frames, the POSE ones per sub-frame
    lines, bad = [], []
    for k in GAUSS + POSE:
        err = gd.rel_err(k, mine[k])
        bar = max(1e-3, 2.0 * C2_NOISE[k])
        lines.append("%-16s err %.2e   reference run-to-run %.2e   bar %.2e" % (k, err, C2_NOISE[k], bar))
        if not err <= bar:
            bad.append(k)
    gd.done()
    with capsys.disabled():
        print("\nc2 gradients, per element (floor 1e-3 of the tensor's max):\n  " + "\n  ".join(lines))
    assert not bad, (bad, lines)


def test_c3_forward_vs_reference_cuda():
    _compare_forward("c3")


def test_end_to_end_control_point_gradients_vs_reference_chain(capsys):
    """The two arms of bench.py on the same c1 workload: this library (`cmm.query` -> fused L1 -> backward) against
    the reference extension driven by the reference's per-sub-frame loop and torch pose chain (autograd)."""
    import bench
    dev = torch.device("cuda", 0)
    w = bench.build_workload("c1", 0, dev)
    gt = w["gt_host"].to(dev)
    params = w["gaussians"].parameters() + w["cmm"].parameters()
    names = ["xyz", "features_dc", "features_rest", "scaling", "rotation", "opacity", "ctrl_trans", "ctrl_rot", "nu"]
    loss = bench.make_step_ours(w, 1)(gt)
    torch.cuda.synchronize()
    gd = pu.Golden("e2e_c1")
    gd.abs_close("loss", loss.detach().reshape(1), 1e-6)
    lines, bad = [], []
    for n, p in zip(names, params):
        err = gd.rel_err(n, p.grad)
        a, b, m = gd.sample(n, p.grad)
        relmax = float((a - b).abs().max()) / max(m, 1e-30)
        pose = n in C1_POSE_NOISE
        # Pose parameters (what this test is for): per element.  Gaussian tensors: max-abs error over max-abs here;
        # their per-element accuracy is pinned against the float64 evaluation in tests/test_gpu_accuracy.py, where
        # the reference's own rotation / scale gradients are 1e-3 .. 1e-2 off per element (float cancellation in the
        # covariance backward), far above its run-to-run spread -- a per-element bar derived from that spread would
        # test the reference's rounding, not this library.
        ok = err <= max(1e-3, 2.0 * C1_POSE_NOISE[n]) if pose else relmax <= 1e-3
        lines.append("%-14s per-element %.2e   max-abs/max-abs %.2e" % (n, err, relmax))
        if not ok:
            bad.append(n)
    gd.done()
    with capsys.disabled():
        print("\nc1 end-to-end gradients (per element: floor 1e-3 of the tensor's max):\n  " + "\n  ".join(lines))
    assert not bad, (bad, lines)
